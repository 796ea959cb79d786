#include "tokenizer.h"

#include <map>

namespace tt {

namespace {
constexpr int kNumClasses = 95;   // PARSeq head outputs (TT_NUM_CLASSES)
}

const TokenizerTable& tokenizer_table() {
  static const TokenizerTable table = [] {
    TokenizerTable t;
    // tuatara.cpp:32-34.  The second literal starts with an escaped backslash followed by an
    // apostrophe, so the charset holds a backslash before the apostrophe: 95 symbols, not 94.
    const std::string charset =
        "0123456789abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ!\"#$%&"
        "\\'()*+,-./:;<=>?@[\\]^_`{|}~";
    t.itos = std::string(1, ']') + charset + "[" + "P";  // :36-39
    std::map<char, int> stoi;
    for (size_t i = 0; i < t.itos.size(); ++i) stoi[t.itos[i]] = static_cast<int>(i);  // :41-43, later wins
    t.eos_id = stoi[']'];  // 88: the ']' inside the charset, not slot 0
    t.bos_id = stoi['['];  // 96
    t.pad_id = stoi['P'];  // 97
    return t;
  }();
  return table;
}

std::string decode_ids(const int32_t* ids, int len) {
  const TokenizerTable& t = tokenizer_table();
  std::string s;
  for (int i = 0; i < len; ++i) {
    const int id = ids[i];
    if (id == t.eos_id) continue;
    if (id < 0 || id >= static_cast<int>(t.itos.size())) continue;
    const char ch = t.itos[id];
    if (ch == ']') break;
    s.push_back(ch);
  }
  return s;
}

void decode_ids_scored(const int32_t* ids, const float* p, int len, std::string* text, std::vector<float>* char_conf,
                       float* conf) {
  const TokenizerTable& t = tokenizer_table();
  text->clear();
  char_conf->clear();
  int end = len - 1;   // no end class: every position is a factor
  for (int i = 0; i < len; ++i) {   // decode_ids' loop, keeping the probability of each character it emits
    const int id = ids[i];
    if (id == t.eos_id) continue;
    if (id < 0 || id >= static_cast<int>(t.itos.size())) continue;
    const char ch = t.itos[id];
    if (ch == ']') { end = i; break; }
    text->push_back(ch);
    char_conf->push_back(p[i]);
  }
  double prod = 1.0;
  for (int i = 0; i <= end; ++i) prod *= static_cast<double>(p[i]);
  *conf = static_cast<float>(prod);
}

void char_filter_mask(const char* allow, const char* block, uint32_t mask[4]) {
  const TokenizerTable& t = tokenizer_table();
  auto holds = [](const char* s, char ch) {
    for (; *s; ++s)
      if (*s == ch) return true;
    return false;
  };
  for (int w = 0; w < 4; ++w) mask[w] = 0;
  for (int c = 0; c < kNumClasses; ++c) {
    const char ch = t.itos[c];
    const bool ok = c == 0 || c == t.eos_id || ((!allow || holds(allow, ch)) && (!block || !holds(block, ch)));
    if (ok) mask[c >> 5] |= 1u << (c & 31);
  }
}

}  // namespace tt
