#include "lexicon.h"

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <memory>

#include "common.h"
#include "tokenizer.h"
#include "tuatara_c.h"

namespace tt {

namespace {

constexpr int kMaxWordLen = TT_MAX_LABEL_LEN - 1;   // the end class needs the last position

// The classes (1..94, not eos_id) printing each byte, in class order: backslash has two.
const std::vector<int>* byte_classes() {
  static const std::vector<std::vector<int>> table = [] {
    const TokenizerTable& t = tokenizer_table();
    std::vector<std::vector<int>> v(256);
    for (int c = 1; c < TT_NUM_CLASSES; ++c)
      if (c != t.eos_id) v[static_cast<uint8_t>(t.itos[c])].push_back(c);
    return v;
  }();
  return table.data();
}

bool allowed(const ClassMask& m, int c) { return (m[c >> 5] >> (c & 31)) & 1u; }

}  // namespace

std::string lexicon_word_error(const char* word, int index) {
  const std::string at = "word " + std::to_string(index);
  if (!word) return at + " is NULL";
  const size_t len = std::strlen(word);
  if (len < 1 || len > static_cast<size_t>(kMaxWordLen))
    return at + " is " + std::to_string(len) + " bytes long; a word has 1 to " + std::to_string(kMaxWordLen) + " bytes";
  const std::vector<int>* bc = byte_classes();
  for (size_t i = 0; i < len; ++i) {
    const uint8_t b = static_cast<uint8_t>(word[i]);
    if (bc[b].empty()) {
      char buf[64];
      if (b >= 0x20 && b < 0x7f)
        std::snprintf(buf, sizeof(buf), "byte 0x%02x ('%c')", b, b);
      else
        std::snprintf(buf, sizeof(buf), "byte 0x%02x", b);
      return at + " holds " + buf + " at offset " + std::to_string(i) + ", which no class prints";
    }
  }
  return std::string();
}

bool word_allowed(const std::string& word, const ClassMask& mask) {
  const std::vector<int>* bc = byte_classes();
  for (char ch : word) {
    bool ok = false;
    for (int c : bc[static_cast<uint8_t>(ch)]) ok = ok || allowed(mask, c);
    if (!ok) return false;
  }
  return true;
}

Automaton build_trie(const std::vector<std::string>& words) {
  // nodes with their children as (byte, child) pairs and whether a word ends there
  struct Node {
    std::vector<std::pair<uint8_t, int32_t>> kids;
    bool end = false;
  };
  std::vector<Node> nodes(1);
  for (const std::string& w : words) {
    int32_t s = 0;
    for (char ch : w) {
      const uint8_t b = static_cast<uint8_t>(ch);
      int32_t nxt = -1;
      for (const auto& k : nodes[s].kids)
        if (k.first == b) { nxt = k.second; break; }
      if (nxt < 0) {
        nxt = static_cast<int32_t>(nodes.size());
        nodes[s].kids.emplace_back(b, nxt);
        nodes.emplace_back();
      }
      s = nxt;
    }
    nodes[s].end = true;
  }
  const std::vector<int>* bc = byte_classes();
  Automaton a;
  a.allow.resize(nodes.size());
  a.first.resize(nodes.size());
  std::vector<std::pair<int, int32_t>> edges;   // (class, successor) of one state, sorted by class
  for (size_t s = 0; s < nodes.size(); ++s) {
    edges.clear();
    if (nodes[s].end) edges.emplace_back(0, Automaton::kDone);
    for (const auto& k : nodes[s].kids)
      for (int c : bc[k.first]) edges.emplace_back(c, k.second);
    std::sort(edges.begin(), edges.end());
    ClassMask m{0, 0, 0, 0};
    a.first[s] = static_cast<int32_t>(a.next.size());
    for (const auto& e : edges) {
      m[e.first >> 5] |= 1u << (e.first & 31);
      a.next.push_back(e.second);
    }
    a.allow[s] = m;
  }
  return a;
}

Automaton one_state(const ClassMask& mask) {
  Automaton a;
  a.allow.push_back(mask);
  a.first.push_back(0);
  for (int c = 0; c < TT_NUM_CLASSES; ++c)
    if (allowed(mask, c)) a.next.push_back(c == 0 ? Automaton::kDone : 0);
  return a;
}

LexTableBuilder::LexTableBuilder() {
  ClassMask all{0, 0, 0, 0};
  for (int c = 0; c < TT_NUM_CLASSES; ++c) all[c >> 5] |= 1u << (c & 31);
  allow_.push_back(all);
  first_.push_back(0);
  next_.assign(TT_NUM_CLASSES, 0);
}

int LexTableBuilder::append(const Automaton& a) {
  const int32_t s0 = static_cast<int32_t>(allow_.size()), e0 = static_cast<int32_t>(next_.size());
  allow_.insert(allow_.end(), a.allow.begin(), a.allow.end());
  for (int32_t f : a.first) first_.push_back(f + e0);
  for (int32_t v : a.next) next_.push_back(v == Automaton::kDone ? 0 : v + s0);
  return s0;
}

std::vector<uint32_t> LexTableBuilder::words() const {
  std::vector<uint32_t> out;
  out.reserve(allow_.size() * 5 + next_.size());
  for (const ClassMask& m : allow_) out.insert(out.end(), m.begin(), m.end());
  out.insert(out.end(), first_.begin(), first_.end());
  out.insert(out.end(), next_.begin(), next_.end());
  return out;
}

}  // namespace tt

using namespace tt;

extern "C" {

int tt_lexicon_create(const char* const* words, int n_words, tt_lexicon** out) {
  try {
    if (!out) { set_error("tt_lexicon_create: out is NULL"); return 1; }
    *out = nullptr;
    if (!words || n_words < 1) {
      set_error("tt_lexicon_create: need at least one word (words is " + std::string(words ? "not NULL" : "NULL") +
                ", n_words is " + std::to_string(n_words) + ")");
      return 1;
    }
    std::unique_ptr<tt_lexicon> lex(new tt_lexicon);
    lex->words.reserve(n_words);
    for (int i = 0; i < n_words; ++i) {
      const std::string err = lexicon_word_error(words[i], i);
      if (!err.empty()) { set_error("tt_lexicon_create: " + err); return 1; }
      lex->words.emplace_back(words[i]);
    }
    std::sort(lex->words.begin(), lex->words.end());
    lex->words.erase(std::unique(lex->words.begin(), lex->words.end()), lex->words.end());
    lex->trie = build_trie(lex->words);
    *out = lex.release();
    return 0;
  } catch (const std::exception& ex) {
    set_error(std::string("tt_lexicon_create: ") + ex.what());
    return 1;
  }
}

void tt_lexicon_destroy(tt_lexicon* lex) { delete lex; }

int tt_lexicon_info(const tt_lexicon* lex, int* n_words, int* n_states) {
  if (!lex) { set_error("tt_lexicon_info: null lexicon"); return 1; }
  if (n_words) *n_words = static_cast<int>(lex->words.size());
  if (n_states) *n_states = static_cast<int>(lex->trie.allow.size());
  return 0;
}

}  // extern "C"
