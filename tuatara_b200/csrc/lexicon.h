// Lexicons (INTEGRATION.md section 9): a trie over a caller's words, in the compact automaton format the greedy decode
// walks on the device (nn_kernels.cuh LexDev).
#pragma once
#include <stdint.h>

#include <array>
#include <string>
#include <vector>

namespace tt {

using ClassMask = std::array<uint32_t, 4>;   // bit c & 31 of word c >> 5: class c allowed (tt_char_filter_mask)

// An automaton without its done state.  State s allows the classes set in allow[s]; next[first[s] + k] is the successor
// of its k-th allowed class in class order, kDone for the done state.  State 0 is the root.
struct Automaton {
  static constexpr int32_t kDone = -1;
  std::vector<ClassMask> allow;
  std::vector<int32_t> first;
  std::vector<int32_t> next;
};

// The error of word `index` (empty when valid): 1..25 bytes, each printed by a class in 1..94 other than 88.
std::string lexicon_word_error(const char* word, int index);
// The trie over distinct valid words (at least one): a state allows class 0 iff a word ends there, class c (1..94,
// c != 88) iff a word continues with itos[c]; both backslash classes lead to the same child.  Class 0 goes to kDone.
Automaton build_trie(const std::vector<std::string>& words);
// One state allowing the classes of `mask`: class 0 goes to kDone, every other allowed class back to the state.
Automaton one_state(const ClassMask& mask);
// Whether every byte of `word` is printed by a class of 1..94 (not 88) that `mask` allows.
bool word_allowed(const std::string& word, const ClassMask& mask);

// The automata of one request in the device layout: state 0 is the shared done state (every class, loops to itself),
// then the appended automata.  `words` holds allow [S][4] | first [S] | next [E], all 32-bit.
class LexTableBuilder {
 public:
  LexTableBuilder();
  int append(const Automaton& a);   // -> the global index of a's root
  int n_states() const { return static_cast<int>(allow_.size()); }
  // the table in one block: allow, then first, then next
  std::vector<uint32_t> words() const;

 private:
  std::vector<ClassMask> allow_;
  std::vector<int32_t> first_, next_;
};

}  // namespace tt

// A caller's lexicon (tt_lexicon_create): the distinct words, sorted, and their trie.  Immutable after creation.
struct tt_lexicon {
  std::vector<std::string> words;
  tt::Automaton trie;
};
