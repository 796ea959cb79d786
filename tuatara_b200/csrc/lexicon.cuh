// Device side of the constrained greedy choice: how a choice site gets its class mask, and the two bit operations the
// lexicon walk needs (lexicon.h has the table layout).
#pragma once
#include <stdint.h>

namespace tt {

// Where a choice site's class mask comes from: none (every class), one mask per crop (character filters), or the
// allow row of the crop's current automaton state (lexicons; the state advances with the chosen class).
enum { MASK_NONE = 0, MASK_CROP = 1, MASK_STATE = 2 };

// The lowest class whose bit is set (a state always allows at least one class).
__device__ __forceinline__ int lowest_class(const uint32_t (&w)[4]) {
  return w[0] ? __ffs(w[0]) - 1 : w[1] ? 31 + __ffs(w[1]) : w[2] ? 63 + __ffs(w[2]) : 95 + __ffs(w[3]);
}

// The number of set bits below class c: the rank of allowed class c among its state's successors.
__device__ __forceinline__ int classes_below(const uint32_t (&w)[4], int c) {
  int k = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int lo = c - 32 * i;
    k += lo >= 32 ? __popc(w[i]) : lo > 0 ? __popc(w[i] & ((1u << lo) - 1u)) : 0;
  }
  return k;
}

}  // namespace tt
