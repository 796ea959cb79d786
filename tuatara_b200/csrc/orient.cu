#include "orient.cuh"

#include "common.h"
#include "word_conf.cuh"

namespace tt {

namespace {

__global__ void __launch_bounds__(128) k_orient_select(const int* __restrict__ ids, const float* __restrict__ pmax,
                                                       int n_words, int L, OrientSet set, int* __restrict__ ids_out,
                                                       float* __restrict__ pmax_out, int* __restrict__ angle_out) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_words) return;
  int best = 0;
  float best_conf = 0.f;
  for (int r = 0; r < set.n; ++r) {
    const size_t row = (static_cast<size_t>(w) * set.n + r) * L;
    const float conf = word_conf(ids + row, pmax + row, L);
    if (r == 0 || conf > best_conf) { best = r; best_conf = conf; }
  }
  const size_t src = (static_cast<size_t>(w) * set.n + best) * L, dst = static_cast<size_t>(w) * L;
  for (int t = 0; t < L; ++t) ids_out[dst + t] = ids[src + t];
  if (pmax_out != nullptr)
    for (int t = 0; t < L; ++t) pmax_out[dst + t] = pmax[src + t];
  angle_out[w] = set.angle[best];
}

}  // namespace

cudaError_t orient_select(const int* ids, const float* pmax, int n_words, int L, const OrientSet& set, int* ids_out,
                          float* pmax_out, int* angle_out, cudaStream_t s) {
  if (n_words <= 0) return cudaSuccess;
  k_orient_select<<<(n_words + 127) / 128, 128, 0, s>>>(ids, pmax, n_words, L, set, ids_out, pmax_out, angle_out);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

}  // namespace tt
