// Choice among a word's rotation candidates (INTEGRATION.md section 8), made on the device so that only the winner's
// ids, probabilities and angle are copied back.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace tt {

// The candidate angles of a request: angle[0] = 0, then the requested ones in increasing order; n = 1 + |rotation_info|.
struct OrientSet {
  int n;
  int angle[4];
};

// ids / pmax: [n_words * set.n][L], crop w * set.n + r holding candidate r of word w (the refinement head's argmax and
// probability).  Per candidate, conf = p[0] * ... * p[e] multiplied in double in position order and rounded once to
// float, e being the first position of id 0, else L - 1 (decode_ids_scored's conf).  The winner is candidate 0 unless a
// later candidate's conf is strictly greater than the best so far (ties and NaN stay with the earlier one).  Writes the
// winner's ids to ids_out [n_words][L], its probabilities to pmax_out [n_words][L] (nullable) and its angle to
// angle_out [n_words].  One thread per word.
cudaError_t orient_select(const int* ids, const float* pmax, int n_words, int L, const OrientSet& set, int* ids_out,
                          float* pmax_out, int* angle_out, cudaStream_t s);

}  // namespace tt
