#include "contrast.cuh"

#include "common.h"
#include "word_conf.cuh"

namespace tt {

namespace {

constexpr int kCropElems = 128 * 96;   // bf16 values of one crop's patch rows

// The candidate of `angle` in the request's set (0 without rotation candidates).
__device__ __forceinline__ int candidate_of(const int* __restrict__ angle, int w, const OrientSet& set) {
  if (angle == nullptr) return 0;
  const int a = angle[w];
  int r = 0;
  for (int k = 1; k < set.n; ++k)
    if (set.angle[k] == a) r = k;
  return r;
}

// One block per word.  Pixel i of the crop is patch row i / 32, its three channels at columns i % 32 + 0 / 32 / 64
// (crop_resize's layout), so the grey histogram needs no reordering.
__global__ void __launch_bounds__(256) k_contrast_stats(const int* __restrict__ ids, const float* __restrict__ p, int L,
                                                        float contrast_ths, float adjust_contrast,
                                                        const __nv_bfloat16* __restrict__ patches, int R,
                                                        const int* __restrict__ angle, OrientSet set, int* __restrict__ flag,
                                                        double2* __restrict__ lr) {
  __shared__ int hist[256];
  __shared__ int sorted_at[4];   // the sorted grey values of ranks 409, 410, 3685 and 3686
  const int w = blockIdx.x;
  if (ids != nullptr && !(word_conf(ids + static_cast<size_t>(w) * L, p + static_cast<size_t>(w) * L, L) < contrast_ths)) {
    if (threadIdx.x == 0) flag[w] = 0;
    return;
  }
  const __nv_bfloat16* crop = patches + (static_cast<size_t>(w) * R + candidate_of(angle, w, set)) * kCropElems;
  hist[threadIdx.x] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < 4096; i += 256) {
    const __nv_bfloat16* px = crop + (i >> 5) * 96 + (i & 31);
    const int b = static_cast<int>(__bfloat162float(px[0]));
    const int g = static_cast<int>(__bfloat162float(px[32]));
    const int r = static_cast<int>(__bfloat162float(px[64]));
    atomicAdd(&hist[(b * 3735 + g * 19235 + r * 9798 + (1 << 14)) >> 15], 1);   // cv2 BGR2GRAY, 8-bit
  }
  __syncthreads();
  if (threadIdx.x < 32) {   // warp 0: prefix sums over 8 bins per lane
    const int lane = threadIdx.x;
    int c[8], sum = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { c[k] = hist[lane * 8 + k]; sum += c[k]; }
    int incl = sum;
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    int before = incl - sum;
    const int rank[4] = {409, 410, 3685, 3686};
#pragma unroll
    for (int k = 0; k < 8; ++k) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (before <= rank[j] && rank[j] < before + c[k]) sorted_at[j] = lane * 8 + k;
      before += c[k];
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    // np.percentile's linear rule at index 409.5 / 3685.5: b - (b - a) * 0.5, exact for these integers
    const double a0 = sorted_at[0], b0 = sorted_at[1], a1 = sorted_at[2], b1 = sorted_at[3];
    const double low = __dadd_rn(b0, -__dmul_rn(__dadd_rn(b0, -a0), 0.5));
    const double high = __dadd_rn(b1, -__dmul_rn(__dadd_rn(b1, -a1), 0.5));
    const double contrast = __ddiv_rn(__dadd_rn(high, -low), fmax(10.0, __dadd_rn(high, low)));
    const bool stretch = contrast < static_cast<double>(adjust_contrast);
    flag[w] = stretch ? 1 : 0;
    if (stretch) lr[w] = make_double2(low, __ddiv_rn(200.0, fmax(10.0, __dadd_rn(high, -low))));
  }
}

// Order-preserving compaction of the flagged words (one block, as k_dec_compact).
__global__ void __launch_bounds__(1024) k_contrast_compact(const int* __restrict__ flag, int n, int* __restrict__ list,
                                                           int* __restrict__ count) {
  __shared__ int s_off[32];
  __shared__ int s_total;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int base = 0;
  for (int s0 = 0; s0 < n; s0 += 1024) {
    const int w = s0 + threadIdx.x;
    const bool keep = w < n && flag[w] != 0;
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s_off[warp] = __popc(m);
    __syncthreads();
    if (warp == 0) {
      const int v = s_off[lane];
      int incl = v;
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      s_off[lane] = incl - v;
      if (lane == 31) s_total = incl;
    }
    __syncthreads();
    if (keep) list[base + s_off[warp] + __popc(m & ((1u << lane) - 1u))] = w;
    base += s_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *count = base;
}

// One block per listed word: the 256-entry table, then the crop through it.
__global__ void __launch_bounds__(256) k_contrast_apply(const int* __restrict__ list, const __nv_bfloat16* __restrict__ patches,
                                                        int R, const int* __restrict__ angle, OrientSet set,
                                                        const double2* __restrict__ lr, __nv_bfloat16* __restrict__ out_patches,
                                                        uint8_t* __restrict__ out_u8, const uint32_t* __restrict__ mask,
                                                        uint32_t* __restrict__ mask_out, const int* __restrict__ root,
                                                        int* __restrict__ root_out) {
  __shared__ __nv_bfloat16 table[256];
  const int i = blockIdx.x, w = list[i];
  const size_t c = static_cast<size_t>(w) * R + candidate_of(angle, w, set);
  const __nv_bfloat16* crop = patches + c * kCropElems;
  {
    const double2 q = lr[w];
    const double x = __dmul_rn(__dadd_rn(__dadd_rn(static_cast<double>(threadIdx.x), -q.x), 25.0), q.y);
    table[threadIdx.x] = __float2bfloat16(static_cast<float>(__double2int_rz(fmin(255.0, fmax(0.0, x)))));
  }
  if (mask != nullptr && threadIdx.x < 4) mask_out[4 * static_cast<size_t>(i) + threadIdx.x] = mask[4 * c + threadIdx.x];
  if (root != nullptr && threadIdx.x == 0) root_out[i] = root[c];
  __syncthreads();
  if (out_patches != nullptr) {
    const uint4* src = reinterpret_cast<const uint4*>(crop);
    uint4* dst = reinterpret_cast<uint4*>(out_patches + static_cast<size_t>(i) * kCropElems);
    for (int k = threadIdx.x; k < kCropElems / 8; k += 256) {
      uint4 v = src[k];
      __nv_bfloat16* e = reinterpret_cast<__nv_bfloat16*>(&v);
#pragma unroll
      for (int j = 0; j < 8; ++j) e[j] = table[static_cast<int>(__bfloat162float(e[j]))];
      dst[k] = v;
    }
  }
  if (out_u8 != nullptr) {
    for (int k = threadIdx.x; k < kCropElems; k += 256) {
      const int row = k / 96, col = k % 96, ch = col >> 5, rem = col & 31;
      const int y = (row >> 4) * 4 + (rem >> 3), x = (row & 15) * 8 + (rem & 7);
      out_u8[((static_cast<size_t>(w) * 32 + y) * 128 + x) * 3 + ch] =
          static_cast<uint8_t>(__bfloat162float(table[static_cast<int>(__bfloat162float(crop[k]))]));
    }
  }
}

__global__ void __launch_bounds__(128) k_contrast_select(int* __restrict__ ids, float* __restrict__ p, int L,
                                                         const int* __restrict__ list, int n_listed,
                                                         const int* __restrict__ ids2, const float* __restrict__ p2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_listed) return;
  const size_t dst = static_cast<size_t>(list[i]) * L, src = static_cast<size_t>(i) * L;
  if (!(word_conf(ids2 + src, p2 + src, L) > word_conf(ids + dst, p + dst, L))) return;
  for (int t = 0; t < L; ++t) {
    ids[dst + t] = ids2[src + t];
    p[dst + t] = p2[src + t];
  }
}

}  // namespace

cudaError_t contrast_stats(const int* ids, const float* p, int n_words, int L, float contrast_ths, float adjust_contrast,
                           const __nv_bfloat16* patches, int R, const int* angle, const OrientSet& set, int* flag,
                           double2* lr, cudaStream_t s) {
  if (n_words <= 0) return cudaSuccess;
  k_contrast_stats<<<n_words, 256, 0, s>>>(ids, p, L, contrast_ths, adjust_contrast, patches, R, angle, set, flag, lr);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t contrast_compact(const int* flag, int n_words, int* list, int* count, cudaStream_t s) {
  if (n_words <= 0) return cudaSuccess;
  k_contrast_compact<<<1, 1024, 0, s>>>(flag, n_words, list, count);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t contrast_apply(const int* list, int n_listed, const __nv_bfloat16* patches, int R, const int* angle,
                           const OrientSet& set, const double2* lr, __nv_bfloat16* out_patches, uint8_t* out_u8,
                           const uint32_t* mask, uint32_t* mask_out, const int* root, int* root_out, cudaStream_t s) {
  if (n_listed <= 0) return cudaSuccess;
  k_contrast_apply<<<n_listed, 256, 0, s>>>(list, patches, R, angle, set, lr, out_patches, out_u8, mask, mask_out, root,
                                            root_out);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t contrast_select(int* ids, float* p, int L, const int* list, int n_listed, const int* ids2, const float* p2,
                            cudaStream_t s) {
  if (n_listed <= 0) return cudaSuccess;
  k_contrast_select<<<(n_listed + 127) / 128, 128, 0, s>>>(ids, p, L, list, n_listed, ids2, p2);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

}  // namespace tt
