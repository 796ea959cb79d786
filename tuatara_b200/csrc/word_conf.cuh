// The word confidence of one crop, computed on the device by the rotation choice (orient.cu) and the contrast re-read
// (contrast.cu) with the same code, so that both compare exactly the conf the host reports (decode_ids_scored).
#pragma once
#include <cuda_runtime.h>

namespace tt {

// ids / p: one crop's refinement row [L].  conf = p[0] * ... * p[e] multiplied in double in position order and rounded
// once to float, e being the first position of id 0, else L - 1.
__device__ __forceinline__ float word_conf(const int* __restrict__ ids, const float* __restrict__ p, int L) {
  int end = L - 1;
  for (int t = 0; t < L; ++t)
    if (ids[t] == 0) { end = t; break; }
  double prod = 1.0;
  for (int t = 0; t <= end; ++t) prod = __dmul_rn(prod, static_cast<double>(p[t]));
  return __double2float_rn(prod);
}

}  // namespace tt
