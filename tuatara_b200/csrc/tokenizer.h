// The reference's Tokenizer (tuatara.cpp:25-117) and the truncation of :492-505, quirks included.
#pragma once
#include <stdint.h>

#include <string>
#include <vector>

namespace tt {

struct TokenizerTable {
  std::string itos;  // 98 symbols: ']' + 95-char charset + '[' + 'P'
  int eos_id, bos_id, pad_id;
};
const TokenizerTable& tokenizer_table();

// ids: the per-position argmax over the 95 classes (first max wins, like at::max on CPU).
// Drops every id == eos_id (tuatara.cpp:108-116), maps through itos (:93-99), cuts at the first
// ']' character (:497-502).
std::string decode_ids(const int32_t* ids, int len);

// decode_ids with scores.  p[i]: the largest softmax probability at position i.  The end position e is the first
// position whose id is 0 (itos[0] = ']', where decode_ids stops; upstream PARSeq's EOS class), else len - 1.
//   text      == decode_ids(ids, len)
//   char_conf  = p[i] of each position that emits a character of text, in order: positions before the first id 0
//                (every position when there is none) whose id is not eos_id, so char_conf.size() == text.size()
//   conf       = prod_{i=0..e} p[i], multiplied in double in position order and rounded once to float
void decode_ids_scored(const int32_t* ids, const float* p, int len, std::string* text, std::vector<float>* char_conf,
                       float* conf);

// Class mask of a character filter (tt_char_filter_mask): bit c & 31 of mask[c >> 5] is set when class c (0..94) is
// allowed.  Classes 0 and eos_id print nothing and are always allowed; any other class c is allowed iff (allow is null
// or holds itos[c]) and (block is null or does not hold itos[c]).  Characters no class prints are ignored; mask[3] = 0.
void char_filter_mask(const char* allow, const char* block, uint32_t mask[4]);

}  // namespace tt
