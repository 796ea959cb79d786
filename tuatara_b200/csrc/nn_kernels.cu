// Non-GEMM kernels of CRAFT and PARSeq (see nn_kernels.cuh).  They stand in for the ATen ops the
// reference reaches through TorchScript (tuatara.cpp:376, :307): max_pool2d, upsample_bilinear2d,
// layer_norm, scaled-dot-product attention, embedding, argmax.
#include "nn_kernels.cuh"

#include <cuda.h>
#include <math.h>

#include <algorithm>

#include <cstdlib>

#include "attn_softmax.cuh"
#include "common.h"
#include "epi_math.cuh"
#include "gemm_tc.cuh"
#include "lexicon.cuh"
#include "ptx.cuh"
#include "trace.h"

namespace tt {

namespace {

__device__ __forceinline__ uint4 ld8(const __nv_bfloat16* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void st8(__nv_bfloat16* p, uint4 v) { *reinterpret_cast<uint4*>(p) = v; }
__device__ __forceinline__ uint4 max8(uint4 a, uint4 b) {
  uint4 r;
  const __nv_bfloat162* x = reinterpret_cast<const __nv_bfloat162*>(&a);
  const __nv_bfloat162* y = reinterpret_cast<const __nv_bfloat162*>(&b);
  __nv_bfloat162* z = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) z[i] = __hmax2(x[i], y[i]);
  return r;
}
__device__ __forceinline__ void unpack8(uint4 v, float f[8]) {
  const __nv_bfloat162* x = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) { f[2 * i] = __low2float(x[i]); f[2 * i + 1] = __high2float(x[i]); }
}
__device__ __forceinline__ uint4 pack8(const float f[8]) {
  uint4 r;
  __nv_bfloat162* z = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) z[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return r;
}

// ------------------------------------------------------------------------------- CRAFT aux
__global__ void k_maxpool2(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int B, int H, int W,
                           int C) {
  const int Ho = H / 2, Wo = W / 2, C8 = C / 8;
  const long long total = static_cast<long long>(B) * Ho * Wo * C8;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C8);
    long long t = i / C8;
    const int x = static_cast<int>(t % Wo); t /= Wo;
    const int y = static_cast<int>(t % Ho);
    const int b = static_cast<int>(t / Ho);
    const __nv_bfloat16* p = in + ((static_cast<long long>(b) * H + 2 * y) * W + 2 * x) * C + c * 8;
    const uint4 v = max8(max8(ld8(p), ld8(p + C)), max8(ld8(p + static_cast<long long>(W) * C), ld8(p + static_cast<long long>(W) * C + C)));
    st8(out + ((static_cast<long long>(b) * Ho + y) * Wo + x) * C + c * 8, v);
  }
}

__global__ void k_maxpool3(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int B, int H, int W,
                           int C) {
  const int C8 = C / 8;
  const long long total = static_cast<long long>(B) * H * W * C8;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C8);
    long long t = i / C8;
    const int x = static_cast<int>(t % W); t /= W;
    const int y = static_cast<int>(t % H);
    const int b = static_cast<int>(t / H);
    const __nv_bfloat16* base = in + static_cast<long long>(b) * H * W * C + c * 8;
    uint4 v = ld8(base + (static_cast<long long>(y) * W + x) * C);
    for (int dy = -1; dy <= 1; ++dy)
      for (int dx = -1; dx <= 1; ++dx) {
        const int yy = y + dy, xx = x + dx;
        if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;  // padding is -inf for max pooling
        v = max8(v, ld8(base + (static_cast<long long>(yy) * W + xx) * C));
      }
    st8(out + i * 8, v);
  }
}

__global__ void k_upsample2(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int B, int H, int W,
                            int C) {
  const int Ho = 2 * H, Wo = 2 * W, C8 = C / 8;
  const long long total = static_cast<long long>(B) * Ho * Wo * C8;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C8);
    long long t = i / C8;
    const int x = static_cast<int>(t % Wo); t /= Wo;
    const int y = static_cast<int>(t % Ho);
    const int b = static_cast<int>(t / Ho);
    // area_pixel_compute_source_index(scale 0.5, align_corners=False): max(0, (dst + 0.5) * 0.5 - 0.5)
    const float sy = fmaxf(0.f, (y + 0.5f) * 0.5f - 0.5f), sx = fmaxf(0.f, (x + 0.5f) * 0.5f - 0.5f);
    const int y0 = static_cast<int>(sy), x0 = static_cast<int>(sx);
    const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
    const float ly = sy - y0, lx = sx - x0;
    const __nv_bfloat16* base = in + static_cast<long long>(b) * H * W * C + c * 8;
    float a[8], bb[8], cc[8], d[8], o[8];
    unpack8(ld8(base + (static_cast<long long>(y0) * W + x0) * C), a);
    unpack8(ld8(base + (static_cast<long long>(y0) * W + x1) * C), bb);
    unpack8(ld8(base + (static_cast<long long>(y1) * W + x0) * C), cc);
    unpack8(ld8(base + (static_cast<long long>(y1) * W + x1) * C), d);
#pragma unroll
    for (int k = 0; k < 8; ++k)
      o[k] = (1.f - ly) * ((1.f - lx) * a[k] + lx * bb[k]) + ly * ((1.f - lx) * cc[k] + lx * d[k]);
    st8(out + i * 8, pack8(o));
  }
}

// conv1_1 (3 -> 64, 3x3, + folded BN + ReLU) straight from the u8 page.  Round 1 ran it as a K = 32 tcgen05 GEMM over a
// 64 B/pixel im2col tensor that a separate kernel wrote (70 TFLOP/s; 0.51 ms per 8 pages for a layer whose floor is
// its 128 B/pixel output write, 0.17 ms).  Here a CTA builds the im2col rows of its 16 x 32-pixel tile in smem from a
// u8 halo (each thread one pixel: 27 bytes -> one 64-byte K-major SWIZZLE_64B operand row), one warp issues
// 4 x 2 tcgen05.mma (M = 128 pixels, N = 64, K = 16) into TMEM, and the epilogue (bias, ReLU, bf16) leaves through
// SWIZZLE_128B tiles and TMA stores (image edges clipped by the TMA unit).
//   wt: bf16 [64][32], k = (dy * 3 + dx) * 3 + c (k 27..31 zero), already scaled by 1/255.
constexpr int kC11TileH = 16, kC11TileW = 32, kC11HaloW = kC11TileW + 2;
constexpr int kC11Halo = (kC11TileH + 2) * kC11HaloW * 3;                 // 1836 bytes
constexpr int kC11Smem = 4 * 16384 /* out */ + 4 * 8192 /* A */ + 4096 /* W */ + 2048 /* halo */ + 256 /* bias */ + 64 + 1024;
__global__ void __launch_bounds__(256) k_conv1_1(const uint8_t* __restrict__ img, int H, int W, int n_tiles,
                                                 const __nv_bfloat16* __restrict__ wt, const float* __restrict__ bias,
                                                 const __grid_constant__ CUtensorMap tm_out) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sO = smem;                       // 4 m-tiles x [128 pixels][128 B], SWIZZLE_128B (TMA store source)
  uint8_t* sA = sO + 4 * 16384;             // 4 m-tiles x [128 pixels][32 k] bf16, K-major SWIZZLE_64B
  uint8_t* sW = sA + 4 * 8192;              // [64 couts][32 k] bf16, K-major SWIZZLE_64B
  uint8_t* sHalo = sW + 4096;
  float* sBias = reinterpret_cast<float*>(sHalo + 2048);
  uint64_t* bar = reinterpret_cast<uint64_t*>(sBias + 64);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int tiles_x = (W + kC11TileW - 1) / kC11TileW, tiles_y = (H + kC11TileH - 1) / kC11TileH;
  if (tid == 0) {
    ptx::prefetch_tmap(&tm_out);
    ptx::mbar_init(bar, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 1) ptx::tmem_alloc(tmem_slot, 256);
  {  // weights (swizzled as the MMA reads them): 64 rows x 4 chunks of 16 B; bias
    const int row = tid >> 2, ch = tid & 3;
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(wt + row * 32) + ch);
    *reinterpret_cast<uint4*>(sW + row * 64 + ((ch ^ ((row >> 1) & 3)) << 4)) = v;
  }
  if (tid < 64) sBias[tid] = __ldg(bias + tid);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  // A thread's bytes of a tile's (16 + 2) x (32 + 2) x 3 halo, all requested before any is used.  Persistent CTAs: the
  // NEXT tile's halo is in flight while this one is computed (rolled into a per-CTA loop of dependent loads the kernel
  // was latency bound: 490 us per 8 pages; one tile per CTA with the loads unrolled: 365 us).
  constexpr int kIters = (kC11Halo + 255) / 256;
  auto load_halo = [&](int tile, uint8_t (&hv)[kIters]) {
    const int b = tile / (tiles_x * tiles_y), t = tile - b * tiles_x * tiles_y;
    const int y0 = (t / tiles_x) * kC11TileH, x0 = (t % tiles_x) * kC11TileW;
    const uint8_t* base = img + static_cast<size_t>(b) * H * W * 3;
#pragma unroll
    for (int it = 0; it < kIters; ++it) {
      const int i = it * 256 + tid;
      const int c = i % 3, px = i / 3;
      const int hx = px % kC11HaloW, hy = px / kC11HaloW;
      const int y = y0 + hy - 1, x = x0 + hx - 1;
      hv[it] = (i < kC11Halo && y >= 0 && y < H && x >= 0 && x < W) ? __ldg(base + (static_cast<size_t>(y) * W + x) * 3 + c) : 0;   // zero padding
    }
  };
  uint8_t hv[kIters];
  if (static_cast<int>(blockIdx.x) < n_tiles) load_halo(blockIdx.x, hv);
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int b = tile / (tiles_x * tiles_y), t = tile - b * tiles_x * tiles_y;
    const int y0 = (t / tiles_x) * kC11TileH, x0 = (t % tiles_x) * kC11TileW;
#pragma unroll
    for (int it = 0; it < kIters; ++it) {
      const int i = it * 256 + tid;
      if (i < kC11Halo) sHalo[i] = hv[it];
    }
    __syncthreads();
    if (tile + static_cast<int>(gridDim.x) < n_tiles) load_halo(tile + gridDim.x, hv);
    // im2col rows: pixel p of the tile (2 per thread) -> row (p % 128) of m-tile p / 128; m-tile = 4 image rows x 32 columns
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int p = pass * 256 + tid;
      const int ty = p >> 5, tx = p & 31, mt = p >> 7, r = p & 127;
      const uint8_t* h0 = sHalo + (ty * kC11HaloW + tx) * 3;     // tap (0, 0) of this pixel; a tap row is 9 consecutive bytes
      float v[32];
#pragma unroll
      for (int dy = 0; dy < 3; ++dy)
#pragma unroll
        for (int j = 0; j < 9; ++j) v[dy * 9 + j] = static_cast<float>(h0[dy * kC11HaloW * 3 + j]);
#pragma unroll
      for (int k = 27; k < 32; ++k) v[k] = 0.f;
      uint8_t* arow = sA + mt * 8192 + r * 64;
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        uint4 o;
        __nv_bfloat162 t0 = __floats2bfloat162_rn(v[8 * ch + 0], v[8 * ch + 1]), t1 = __floats2bfloat162_rn(v[8 * ch + 2], v[8 * ch + 3]);
        __nv_bfloat162 t2 = __floats2bfloat162_rn(v[8 * ch + 4], v[8 * ch + 5]), t3 = __floats2bfloat162_rn(v[8 * ch + 6], v[8 * ch + 7]);
        o.x = *reinterpret_cast<uint32_t*>(&t0); o.y = *reinterpret_cast<uint32_t*>(&t1);
        o.z = *reinterpret_cast<uint32_t*>(&t2); o.w = *reinterpret_cast<uint32_t*>(&t3);
        *reinterpret_cast<uint4*>(arow + ((ch ^ ((r >> 1) & 3)) << 4)) = o;
      }
    }
    ptx::fence_proxy_async();
    ptx::tc_fence_before();
    __syncthreads();   // also: every warp finished reading the previous tile's accumulators
    if (warp == 0) {   // all lanes converged, one elected lane issues
      ptx::tc_fence_after();
      const uint32_t idesc = ptx::make_idesc_bf16(128, 64);
      const uint32_t wa = ptx::smem_u32(sW);
#pragma unroll
      for (int mt = 0; mt < 4; ++mt) {
        const uint32_t aa = ptx::smem_u32(sA + mt * 8192);
#pragma unroll
        for (int k = 0; k < 2; ++k)
          ptx::mma_bf16_e(tmem + mt * 64, ptx::make_smem_desc(aa + k * 32, 64), ptx::make_smem_desc(wa + k * 32, 64), idesc, k != 0);
      }
      ptx::mma_commit_e(bar);
    }
    if (tid == 0) ptx::bulk_wait_read<0>();   // the previous tile's TMA stores have read sO
    ptx::mbar_wait(bar, phase);
    phase ^= 1;
    ptx::tc_fence_after();
    __syncthreads();
    // epilogue: warp w reads TMEM lanes (w & 3) * 32 .. of m-tiles (w >> 2) * 2 and + 1
    const int q = warp & 3, r = q * 32 + lane;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int mt = (warp >> 2) * 2 + i;
      uint8_t* orow = sO + mt * 16384 + r * 128;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t raw[32];
        ptx::tmem_ld<32>(tmem + (static_cast<uint32_t>(q * 32) << 16) + mt * 64 + half * 32, raw);
        ptx::tmem_ld_wait(raw);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          float o[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = fmaxf(__uint_as_float(raw[8 * ch + e]) + sBias[half * 32 + 8 * ch + e], 0.f);
          *reinterpret_cast<uint4*>(orow + (((half * 4 + ch) ^ (r & 7)) << 4)) = pack8(o);
        }
      }
    }
    ptx::fence_proxy_async();
    ptx::tc_fence_before();
    __syncthreads();
    if (tid == 0) {
#pragma unroll
      for (int mt = 0; mt < 4; ++mt) ptx::tma_store_4d(&tm_out, sO + mt * 16384, 0, x0, y0 + mt * 4, b);   // rows / columns past the image are clipped
      ptx::bulk_commit();
    }
  }
  if (tid == 0) ptx::bulk_wait_read<0>();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem, 256);
  }
}

int grid_for(long long total, int block) {
  const long long g = (total + block - 1) / block;
  return static_cast<int>(g < 148LL * 16 ? (g > 0 ? g : 1) : 148LL * 16);
}

// ------------------------------------------------------------------------------- LayerNorm
// warp per row; a lane holds PER_LANE elements as PER_LANE / V vectors of V floats (V = 4 when PER_LANE % 4 == 0: D = 384,
// else 2: D = 192), vector j of a lane covers columns (j * 32 + lane) * V ..
template <int PER_LANE>
__global__ void k_layernorm(const float* __restrict__ x, int rows, const float* __restrict__ gamma,
                            const float* __restrict__ beta, float eps, __nv_bfloat16* __restrict__ ob,
                            float* __restrict__ of, int rows_mod) {
  constexpr int D = PER_LANE * 32;
  constexpr int V = (PER_LANE % 4 == 0) ? 4 : 2;
  static_assert(PER_LANE % V == 0, "LayerNorm width");
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + static_cast<long long>(rows_mod > 0 ? row % rows_mod : row) * D;
  float v[PER_LANE];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < PER_LANE / V; ++i) {
    const int col = (i * 32 + lane) * V;
    if constexpr (V == 4) {
      const float4 t = *reinterpret_cast<const float4*>(xr + col);
      v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
      sum += t.x + t.y + t.z + t.w;
    } else {
      const float2 t = *reinterpret_cast<const float2*>(xr + col);
      v[2 * i] = t.x; v[2 * i + 1] = t.y;
      sum += t.x + t.y;
    }
  }
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum / D;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < PER_LANE; ++i) { const float d = v[i] - mean; var += d * d; }
  for (int o = 16; o > 0; o >>= 1) var += __shfl_xor_sync(0xffffffffu, var, o);
  const float rstd = rsqrtf(var / D + eps);
#pragma unroll
  for (int i = 0; i < PER_LANE / V; ++i) {
    const int col = (i * 32 + lane) * V;
    float o[V];
#pragma unroll
    for (int e = 0; e < V; ++e) o[e] = (v[V * i + e] - mean) * rstd * gamma[col + e] + beta[col + e];
    if (ob != nullptr) {
#pragma unroll
      for (int e = 0; e < V; e += 2) {
        __nv_bfloat162 p = __floats2bfloat162_rn(o[e], o[e + 1]);
        *reinterpret_cast<__nv_bfloat162*>(ob + static_cast<long long>(row) * D + col + e) = p;
      }
    }
    if (of != nullptr) {
#pragma unroll
      for (int e = 0; e < V; e += 2)
        *reinterpret_cast<float2*>(of + static_cast<long long>(row) * D + col + e) = make_float2(o[e], o[e + 1]);
    }
  }
}

// ------------------------------------------------------------------------ encoder attention
// grid (heads, crops), 128 threads.  smem (1024-aligned): [Q 16K][K 16K][V 16K]; P (bf16 128x128,
// two 64-key swizzle atoms = 32K) overwrites Q|K once S = QK^T has been consumed.
struct AttnCtl {
  uint64_t bar_load, bar_s, bar_o;
  uint32_t tmem_base;
};
constexpr int kAttnSmem = 3 * 16384 + 1024 + 64;

// ONEPASS: the thread's whole S row (128 fp32) is pulled out of TMEM once and kept in registers for the maximum
// and the exponentials (3 CTAs per SM at <= 168 registers); the two-pass form (4 CTAs per SM) reads S twice and was
// paced by the TMEM read port: 160 KB per CTA at ~64 B/cycle/SM is 2500 of the 3550 cycles an SM spent per CTA
// (profiles/r2_attn_enc.md), ahead of HBM (64 KB per CTA).
template <bool ONEPASS>
__global__ void __launch_bounds__(128, ONEPASS ? 3 : 4) k_attn_enc(const __grid_constant__ CUtensorMap tm_qkv,
                                                                   __nv_bfloat16* __restrict__ out, int D, float scale_log2e,
                                                                   uint32_t* trace, uint32_t serial) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = smem + 16384;
  uint8_t* sV = smem + 32768;
  uint8_t* sP = smem;  // aliases Q|K
  AttnCtl* ctl = reinterpret_cast<AttnCtl*>(smem + 49152);
  const int head = blockIdx.x, crop = blockIdx.y;
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // warp-uniform: warp 0 issues through the uniform datapath

  if (tid == 0) {
    trace_small(trace, serial, TR_ENTER);
    ptx::prefetch_tmap(&tm_qkv);
    ptx::mbar_init(&ctl->bar_load, 1);
    ptx::mbar_init(&ctl->bar_s, 1);
    ptx::mbar_init(&ctl->bar_o, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 0) ptx::tmem_alloc(&ctl->tmem_base, 128);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, ctl->tmem_base, 0);
  if (tid == 0) { trace_small(trace, serial, TR_ALLOC); trace_tmem_event(trace, serial, blockIdx.y * gridDim.x + blockIdx.x, 1); }

  if (warp == 0) {  // all 32 lanes converged, one elected lane issues (ptx.cuh "_e" wrappers)
    ptx::mbar_arrive_expect_tx_e(&ctl->bar_load, 3 * 16384);
    ptx::tma_load_2d_e(sQ, &tm_qkv, &ctl->bar_load, head * 64, crop * 128);
    ptx::tma_load_2d_e(sK, &tm_qkv, &ctl->bar_load, D + head * 64, crop * 128);
    ptx::tma_load_2d_e(sV, &tm_qkv, &ctl->bar_load, 2 * D + head * 64, crop * 128);
    ptx::mbar_wait(&ctl->bar_load, 0);
    __syncwarp();
    ptx::tc_fence_after();
    // S[128 q][128 k] = Q K^T : both operands K-major over the 64 head dims
    const uint32_t idesc = ptx::make_idesc_bf16(128, 128);
    const uint32_t qa = ptx::smem_u32(sQ), ka = ptx::smem_u32(sK);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      ptx::mma_bf16_e(tmem, ptx::make_smem_desc(qa + k * 32, 128), ptx::make_smem_desc(ka + k * 32, 128), idesc, k != 0);
    ptx::mma_commit_e(&ctl->bar_s);
  }
  ptx::mbar_wait(&ctl->bar_s, 0);
  ptx::tc_fence_after();

  // softmax over this thread's row (row == TMEM lane == tid)
  const uint32_t t_row = tmem + (static_cast<uint32_t>(warp * 32) << 16);
  float sum = 0.f;
  const int r = tid;
  if constexpr (ONEPASS) {
    sum = attn_softmax_onepass(t_row, sP, r, scale_log2e);
  } else {
    float mx = -INFINITY;
#pragma unroll
    for (int ch = 0; ch < 8; ++ch) {
      uint32_t raw[16];
      ptx::tmem_ld16(t_row + ch * 16, raw);
      ptx::tmem_ld_wait(raw);
#pragma unroll
      for (int i = 0; i < 16; ++i) mx = fmaxf(mx, __uint_as_float(raw[i]));
    }
#pragma unroll
    for (int ch = 0; ch < 8; ++ch) {
      uint32_t raw[16];
      ptx::tmem_ld16(t_row + ch * 16, raw);
      ptx::tmem_ld_wait(raw);
      float p[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        p[i] = exp2f((__uint_as_float(raw[i]) - mx) * scale_log2e);
        sum += p[i];
      }
      attn_store_p16(sP, r, ch, p);
    }
  }
  // generic-proxy smem writes -> visible to the tensor core (async proxy); all S reads retired
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    ptx::tc_fence_after();
    // O[128 q][64 d] = P V : A = P (K-major over keys), B = V as loaded: rows = keys, 64 dims contiguous
    // == MN-major SWIZZLE_128B, one 1024-byte atom per 8 keys (SBO = 1024), 16 keys per MMA.
    const uint32_t idesc = ptx::make_idesc_bf16(128, 64) | (1u << 16);  // b_major = MN
    const uint32_t pa = ptx::smem_u32(sP), va = ptx::smem_u32(sV);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const uint64_t da = ptx::make_smem_desc(pa + (k >> 2) * 16384 + (k & 3) * 32, 128);
      const uint64_t db = ptx::make_smem_desc(va + k * 2048, 128);
      ptx::mma_bf16_e(tmem, da, db, idesc, k != 0);
    }
    ptx::mma_commit_e(&ctl->bar_o);
  }
  ptx::mbar_wait(&ctl->bar_o, 0);
  ptx::tc_fence_after();
  const float inv = 1.f / sum;
  __nv_bfloat16* orow = out + (static_cast<long long>(crop) * 128 + r) * D + head * 64;
  {
    uint32_t raw[2][32];
    ptx::tmem_ld<32>(t_row, raw[0]);
    ptx::tmem_ld<32>(t_row + 32, raw[1]);
    ptx::tmem_ld_wait(raw[0]);
    ptx::tmem_ld_wait(raw[1]);
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
      float o[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) o[i] = __uint_as_float(raw[ch >> 1][(ch & 1) * 16 + i]) * inv;
      st8(orow + ch * 16, pack8(o));
      st8(orow + ch * 16 + 8, pack8(o + 8));
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem, 128);
    if (tid == 0) { trace_small(trace, serial, TR_DONE); trace_tmem_event(trace, serial, blockIdx.y * gridDim.x + blockIdx.x, 2); }
  }
}

// ------------------------------------------------------------------------- decoder kernels
// one warp per crop: content embedding -> LayerNorm -> bf16
template <int PER_LANE>
__global__ void k_dec_context(const int* __restrict__ tokens, const float* __restrict__ embed,
                              const float* __restrict__ posq, const float* __restrict__ g, const float* __restrict__ b,
                              float eps, int pos, int n, int L, __nv_bfloat16* __restrict__ out) {
  constexpr int D = PER_LANE * 32;
  const int crop = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (crop >= n) return;
  const int tok = tokens[crop * L + pos];
  const float* e = embed + static_cast<long long>(tok) * D;
  float v[PER_LANE];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < PER_LANE; ++i) {
    const int col = i * 32 + lane;
    v[i] = e[col] + (pos > 0 ? posq[(pos - 1) * D + col] : 0.f);
    sum += v[i];
  }
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum / D;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < PER_LANE; ++i) { const float d = v[i] - mean; var += d * d; }
  for (int o = 16; o > 0; o >>= 1) var += __shfl_xor_sync(0xffffffffu, var, o);
  const float rstd = rsqrtf(var / D + eps);
#pragma unroll
  for (int i = 0; i < PER_LANE; ++i) {
    const int col = i * 32 + lane;
    out[static_cast<long long>(crop) * D + col] = __float2bfloat16((v[i] - mean) * rstd * g[col] + b[col]);
  }
}

// Decoder self-attention.  grid (np, crops), block = heads*32 threads: warp = head.
// Scores: lane j owns key j (L <= 32 keys): it reads the head's 64 contiguous bytes of K row j and dots
// them with the query.  Values: lane = head dim, loop over the keys with the probabilities broadcast.
__global__ void k_dec_self_attn(DecoderStep st, const float* __restrict__ q_table,
                                const __nv_bfloat16* __restrict__ kv, const int* __restrict__ tokens, int eos_id,
                                int n_tok, __nv_bfloat16* __restrict__ out) {
  const int pi = blockIdx.x, crop = blockIdx.y;
  const int p = st.p0 + pi;
  const int head = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int D = st.D, L = st.L;
  // key j of this crop = row (j, tokens[crop][j]) of the content K|V table; lane l keeps row l's offset
  const int my_tok = lane < L ? tokens[crop * L + lane] : 0;
  const long long my_row = (static_cast<long long>(lane) * n_tok + my_tok) * 2 * D;
  const __nv_bfloat16* kbase = kv + head * 32;
  // key j allowed?  AR: j <= p.  refine: j != p+1 and no EOS among tokens[1..j]
  int first_eos = L;  // first j >= 1 with tokens[j] == eos
  if (st.refine) {
    const int t = (lane + 1 < L) ? tokens[crop * L + lane + 1] : -1;  // lane l holds token l+1
    const unsigned m = __ballot_sync(0xffffffffu, t == eos_id);
    if (m) first_eos = __ffs(m);
  }
  const int nkeys = st.refine ? L : p + 1;
  const bool mine = lane < nkeys && (st.refine ? (lane != p + 1 && lane < first_eos) : true);
  // every V element this lane will need (dim = lane of keys 0..nkeys-1) is requested before the scores are computed:
  // one memory round trip for the whole kernel instead of one per 8 keys
  const __nv_bfloat16* vbase = kbase + D + lane;
  __nv_bfloat16 vraw[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    const long long row_j = __shfl_sync(0xffffffffu, my_row, j);
    vraw[j] = (j < nkeys) ? vbase[row_j] : __float2bfloat16(0.f);
  }
  float score = -INFINITY;
  if (mine) {
    const float4* q4 = reinterpret_cast<const float4*>(q_table + p * D + head * 32);
    const uint4* k4 = reinterpret_cast<const uint4*>(kbase + my_row);
    float acc = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float f[8];
      unpack8(__ldg(k4 + c), f);
      const float4 qa = __ldg(q4 + 2 * c), qb = __ldg(q4 + 2 * c + 1);
      acc += qa.x * f[0] + qa.y * f[1] + qa.z * f[2] + qa.w * f[3] + qb.x * f[4] + qb.y * f[5] + qb.z * f[6] + qb.w * f[7];
    }
    score = acc * 0.17677669529663687f;  // 1/sqrt(32)
  }
  float mx = score;
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  const float e = mine ? __expf(score - mx) : 0.f;
  float sum = e;
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float pr = e / sum;
  float acc = 0.f;
#pragma unroll
  for (int j = 0; j < 32; ++j) acc += __shfl_sync(0xffffffffu, pr, j) * __bfloat162float(vraw[j]);  // pr == 0 beyond nkeys
  out[(static_cast<long long>(crop) * st.np + pi) * D + head * 32 + lane] = __float2bfloat16(acc);
}

// Self-attention scores of the AR pass as a lookup: with the content K|V a function of (position, token) and the
// queries a function of the position alone, score(i, j, token_j, head) = scale * q_table[i][head] . K[j][token_j][head]
// is a [L][L][n_tok][heads] fp32 table (3.1 MB for PARSeq-base) computed once per engine.  Same summation order as
// k_dec_self_attn, so both produce the same bits.
__global__ void k_dec_score_table(const float* __restrict__ q_table, const __nv_bfloat16* __restrict__ kv_table, int L,
                                  int n_tok, int D, int heads, float* __restrict__ out) {
  const long long total = static_cast<long long>(L) * L * n_tok * heads;
  const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (idx >= total) return;
  const int h = static_cast<int>(idx % heads);
  long long t = idx / heads;
  const int tok = static_cast<int>(t % n_tok); t /= n_tok;
  const int j = static_cast<int>(t % L);
  const int i = static_cast<int>(t / L);
  const float4* q4 = reinterpret_cast<const float4*>(q_table + i * D + h * 32);
  const uint4* k4 = reinterpret_cast<const uint4*>(kv_table + (static_cast<long long>(j) * n_tok + tok) * 2 * D + h * 32);
  float acc = 0.f;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    float f[8];
    unpack8(__ldg(k4 + c), f);
    const float4 qa = __ldg(q4 + 2 * c), qb = __ldg(q4 + 2 * c + 1);
    acc += qa.x * f[0] + qa.y * f[1] + qa.z * f[2] + qa.w * f[3] + qb.x * f[4] + qb.y * f[5] + qb.z * f[6] + qb.w * f[7];
  }
  out[idx] = acc * 0.17677669529663687f;  // 1/sqrt(32)
}

// AR-step self attention, one warp per crop (8 crops per block).  Lane j owns key j: it gathers the heads' scores of
// (step, j, token_j) from the score table (heads * 4 contiguous bytes), the softmax per head runs across the lanes,
// the probabilities go through a per-warp smem tile, and the V rows (row (j, token_j) of the K|V table, L2 resident)
// are accumulated with lane = 16-byte chunk of the row: every load is a full coalesced row.
template <int HEADS>
__global__ void __launch_bounds__(256) k_dec_self_attn_ar(int n, int D, int L, int step, int n_tok,
                                                          const float* __restrict__ sc_table,
                                                          const __nv_bfloat16* __restrict__ kv_table,
                                                          const int* __restrict__ tokens, __nv_bfloat16* __restrict__ out,
                                                          const int* __restrict__ active, const int* __restrict__ n_act) {
  __shared__ float s_p[8][HEADS][32];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int slot = blockIdx.x * 8 + wib;
  if (slot >= (n_act ? *n_act : n)) return;
  const int crop = active ? active[slot] : slot;   // tokens by crop, the output row by slot
  const int nkeys = step + 1;
  const int tok = lane < nkeys ? tokens[crop * L + lane] : 0;
  float sc[HEADS];
  if (lane < nkeys) {
    // HEADS * 4 contiguous bytes (48 / 24): 8-byte loads keep both widths aligned
    const float2* src = reinterpret_cast<const float2*>(sc_table + ((static_cast<long long>(step) * L + lane) * n_tok + tok) * HEADS);
#pragma unroll
    for (int h2 = 0; h2 < HEADS / 2; ++h2) {
      const float2 v = __ldg(src + h2);
      sc[2 * h2] = v.x; sc[2 * h2 + 1] = v.y;
    }
  } else {
#pragma unroll
    for (int h = 0; h < HEADS; ++h) sc[h] = -INFINITY;
  }
#pragma unroll
  for (int h = 0; h < HEADS; ++h) {
    float mx = sc[h];
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    const float e = lane < nkeys ? __expf(sc[h] - mx) : 0.f;
    float sum = e;
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    s_p[wib][h][lane] = e / sum;
  }
  __syncwarp();
  // V accumulation: chunk c (8 dims) belongs to head c / 4
  const int chunks = D / 8;                       // 48 (base) / 24 (tiny): lanes take chunk `lane` and `lane + 32`
  const bool two = lane + 32 < chunks;
  const bool one = lane < chunks;
  const int h0 = lane >> 2, h1 = (lane + 32) >> 2;
  float a0[8], a1[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { a0[e] = 0.f; a1[e] = 0.f; }
  const __nv_bfloat16* vbase = kv_table + D;
  for (int j0 = 0; j0 < nkeys; j0 += 4) {
    uint4 u0[4], u1[4];
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int j = j0 + jj;
      const int tj = __shfl_sync(0xffffffffu, tok, j & 31);
      const uint4* row = reinterpret_cast<const uint4*>(vbase + (static_cast<long long>(j) * n_tok + tj) * 2 * D);
      u0[jj] = (j < nkeys && one) ? __ldg(row + lane) : make_uint4(0u, 0u, 0u, 0u);
      u1[jj] = (j < nkeys && two) ? __ldg(row + lane + 32) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int j = j0 + jj;
      if (j >= nkeys) break;
      float f[8];
      if (one) {
        const float pa = s_p[wib][h0][j];
        unpack8(u0[jj], f);
#pragma unroll
        for (int e = 0; e < 8; ++e) a0[e] += pa * f[e];
      }
      if (two) {
        const float pb = s_p[wib][h1][j];
        unpack8(u1[jj], f);
#pragma unroll
        for (int e = 0; e < 8; ++e) a1[e] += pb * f[e];
      }
    }
  }
  __nv_bfloat16* orow = out + static_cast<long long>(slot) * D;
  if (one) st8(orow + lane * 8, pack8(a0));
  if (two) st8(orow + (lane + 32) * 8, pack8(a1));
}

// Decoder cross-attention over the 128 memory tokens of a crop.  grid (np, crops), 12 warps (= heads).
// Every load is a full coalesced row: a memory row holds K (D bf16) then V (D bf16); a warp takes keys
// w, w+12, ... and reads each K row as 16-byte units (unit u = head u/4, dims (u%4)*8..+8), dots it with
// the matching slice of q, reduces over the 4 lanes of a head -> all heads' scores for that key.  After a
// per-head softmax in smem the V rows are streamed the same way and the 12 warps' partial sums combined.
template <int kD>
__global__ void __launch_bounds__(kD) k_dec_cross_attn(DecoderStep st, const __nv_bfloat16* __restrict__ q,
                                                       const __nv_bfloat16* __restrict__ mem_kv,
                                                       __nv_bfloat16* __restrict__ out) {
  constexpr int kHeads = kD / 32, kKeys = 128, kWarps = kHeads, kUnits = kD / 8;  // 48 (base) / 24 (tiny) 16-byte units per K row
  __shared__ float s_sc[kHeads][kKeys];         // scores, then probabilities
  __shared__ float s_part[kWarps][kD];          // per-warp partial outputs
  const int pi = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // early-exit AR pass: the grid covers at most all crops, the blocks walk the active slots (q / out rows by slot, the
  // memory K|V by crop); without a list every block has exactly its own crop
  const int n_slots = st.n_act ? *st.n_act : st.n_crops;
  for (int slot = blockIdx.y; slot < n_slots; slot += gridDim.y) {
  const int crop = st.active ? st.active[slot] : slot;
  const long long row = static_cast<long long>(slot) * st.np + pi;
  const __nv_bfloat16* kvb = mem_kv + static_cast<long long>(crop) * kKeys * 2 * kD;
  // q slices for the (up to) two units this lane covers: unit lane, unit 32 + lane (lane < 16)
  float qa[8], qb[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { qa[i] = 0.f; qb[i] = 0.f; }
  if (lane < kUnits) unpack8(*reinterpret_cast<const uint4*>(q + row * kD + lane * 8), qa);
  if (lane < kUnits - 32) unpack8(*reinterpret_cast<const uint4*>(q + row * kD + (32 + lane) * 8), qb);
  for (int key = warp; key < kKeys; key += kWarps) {
    const uint4* kr = reinterpret_cast<const uint4*>(kvb + static_cast<long long>(key) * 2 * kD);
    float f[8];
    float a = 0.f, b = 0.f;
    if (lane < kUnits) {
      unpack8(__ldg(kr + lane), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) a += qa[i] * f[i];
    }
    if (lane < kUnits - 32) {
      unpack8(__ldg(kr + 32 + lane), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) b += qb[i] * f[i];
    }
    a += __shfl_xor_sync(0xffffffffu, a, 1); a += __shfl_xor_sync(0xffffffffu, a, 2);
    b += __shfl_xor_sync(0xffffffffu, b, 1); b += __shfl_xor_sync(0xffffffffu, b, 2);
    if ((lane & 3) == 0) {
      if (lane < kUnits) s_sc[lane >> 2][key] = a * 0.17677669529663687f;
      if (lane < kUnits - 32) s_sc[8 + (lane >> 2)][key] = b * 0.17677669529663687f;
    }
  }
  __syncthreads();
  {  // softmax of head `warp` over the 128 keys
    float v[4], mx = -INFINITY;
#pragma unroll
    for (int t = 0; t < 4; ++t) { v[t] = s_sc[warp][t * 32 + lane]; mx = fmaxf(mx, v[t]); }
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) { v[t] = __expf(v[t] - mx); sum += v[t]; }
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = 1.f / sum;
#pragma unroll
    for (int t = 0; t < 4; ++t) s_sc[warp][t * 32 + lane] = v[t] * inv;
  }
  __syncthreads();
  float oa[8], ob[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { oa[i] = 0.f; ob[i] = 0.f; }
  for (int key = warp; key < kKeys; key += kWarps) {
    const uint4* vr = reinterpret_cast<const uint4*>(kvb + static_cast<long long>(key) * 2 * kD + kD);
    float f[8];
    if (lane < kUnits) {
      unpack8(__ldg(vr + lane), f);
      const float pa = s_sc[lane >> 2][key];
#pragma unroll
      for (int i = 0; i < 8; ++i) oa[i] += pa * f[i];
    }
    if (lane < kUnits - 32) {
      unpack8(__ldg(vr + 32 + lane), f);
      const float pb = s_sc[8 + (lane >> 2)][key];
#pragma unroll
      for (int i = 0; i < 8; ++i) ob[i] += pb * f[i];
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    if (lane < kUnits) s_part[warp][lane * 8 + i] = oa[i];
    if (lane < kUnits - 32) s_part[warp][(32 + lane) * 8 + i] = ob[i];
  }
  __syncthreads();
  {
    const int d = threadIdx.x;  // kD threads = kD output dims
    float acc = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) acc += s_part[w][d];
    out[row * kD + d] = __float2bfloat16(acc);
  }
  __syncthreads();   // s_sc / s_part are reused by the next slot
  }
}

// Refinement pass: all L (<= 32) query positions of a crop at once, on mma.sync tensor cores (the per-position
// kernels above re-read a crop's K/V once per position: 26 x 196 KB from L2 for the cross attention).
// grid (3, crops), 4 warps: block = one 128-dim slice of the 384 (4 heads), warp = head (32 dims).  The slice's K
// and V rows (KEYS x 256 B each) are staged with cp.async into padded smem (272-byte pitch: ldmatrix rows fall in
// distinct banks); S = Q K^T and O = P V are m16n8k16 bf16 MMAs, softmax in registers on the accumulator layout.
//   SELF = false: cross attention, q bf16 [crop*np + p][D], kv = memory K|V [crop][128][2D], no mask.
//   SELF = true : self attention over the content cache, q fp32 table [p][D] shared by all crops,
//                 kv = [crop][L][2D], cloze mask (key != p + 1) and key padding from the first EOS on.
constexpr int kRefPitch = 136;  // bf16 elements per staged row (128 + 8 pad)
template <int KEYS, bool SELF>
__global__ void __launch_bounds__(128) k_dec_attn_refine(const void* __restrict__ q_in, const __nv_bfloat16* __restrict__ kv,
                                                         int nkeys, int np, const int* __restrict__ tokens, int eos_id,
                                                         int L, int n_tok, __nv_bfloat16* __restrict__ out) {
  constexpr int kD = 384, kNT = KEYS / 8, kKS = KEYS / 16;
  extern __shared__ __align__(16) uint8_t ref_smem[];
  __nv_bfloat16* sK = reinterpret_cast<__nv_bfloat16*>(ref_smem);
  __nv_bfloat16* sV = sK + KEYS * kRefPitch;
  const int hg = blockIdx.x, crop = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // SELF: key row j = row (j, tokens[crop][j]) of the content K|V table; cross attention: the crop's memory rows
  const __nv_bfloat16* kvb = kv + (SELF ? 0 : static_cast<long long>(crop) * nkeys * 2 * kD) + hg * 128;
  // stage K then V: 16 chunks of 16 B per row
  for (int pass = 0; pass < 2; ++pass) {
    __nv_bfloat16* dst = pass ? sV : sK;
    for (int c = threadIdx.x; c < KEYS * 16; c += 128) {
      const int row = c >> 4, ch = c & 15;
      const uint32_t d = ptx::smem_u32(dst + row * kRefPitch + ch * 8);
      if (row < nkeys) {
        const long long grow = SELF ? static_cast<long long>(row) * n_tok + tokens[crop * L + row] : row;
        const __nv_bfloat16* src = kvb + grow * 2 * kD + pass * kD + ch * 8;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src) : "memory");
      } else {
        ptx::sts128(d, make_uint4(0u, 0u, 0u, 0u));
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  // Q fragments of this warp's head: A (row-major 16x16) x 2 m-tiles x 2 k-steps
  const int dbase = hg * 128 + warp * 32;
  uint32_t qa[2][2][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int p = mt * 16 + (lane >> 2) + (i & 1) * 8;
        const int col = dbase + ks * 16 + (lane & 3) * 2 + (i >> 1) * 8;
        uint32_t v = 0u;
        if (p < np) {
          if constexpr (SELF) {
            const float2 f = *reinterpret_cast<const float2*>(static_cast<const float*>(q_in) + p * kD + col);
            __nv_bfloat162 h = __floats2bfloat162_rn(f.x, f.y);
            v = *reinterpret_cast<uint32_t*>(&h);
          } else {
            v = *reinterpret_cast<const uint32_t*>(static_cast<const __nv_bfloat16*>(q_in) +
                                                   (static_cast<long long>(crop) * np + p) * kD + col);
          }
        }
        qa[mt][ks][i] = v;
      }
  int first_eos = L;
  if constexpr (SELF) {
    const int t = (lane + 1 < L) ? tokens[crop * L + lane + 1] : -1;  // lane l holds token l+1
    const unsigned m = __ballot_sync(0xffffffffu, t == eos_id);
    if (m) first_eos = __ffs(m);
  }
  asm volatile("cp.async.wait_group 1;" ::: "memory");
  __syncthreads();
  float sc[2][kNT][4];
#pragma unroll
  for (int nt = 0; nt < kNT; ++nt) {
    uint32_t b[4];
    const uint32_t addr = ptx::smem_u32(sK + (nt * 8 + (lane & 7)) * kRefPitch + warp * 32 + (lane >> 3) * 8);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(b[0]), "=r"(b[1]), "=r"(b[2]), "=r"(b[3]) : "r"(addr));
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      float* c = sc[mt][nt];
      c[0] = c[1] = c[2] = c[3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                     : "r"(qa[mt][ks][0]), "r"(qa[mt][ks][1]), "r"(qa[mt][ks][2]), "r"(qa[mt][ks][3]), "r"(b[2 * ks]), "r"(b[2 * ks + 1]));
    }
  }
  // masked softmax per query row; a row's 2*kNT values per thread, 4 threads per row
  const float scale = 0.17677669529663687f;  // 1/sqrt(32)
  float inv[2][2];
  uint32_t pp[2][kNT][2];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const int p = mt * 16 + (lane >> 2) + hf * 8;
      float mx = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < kNT; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int key = nt * 8 + (lane & 3) * 2 + e;
          bool ok = key < nkeys;
          if constexpr (SELF) ok = ok && key != p + 1 && key < first_eos;
          float& v = sc[mt][nt][hf * 2 + e];
          v = ok ? v * scale : -INFINITY;
          mx = fmaxf(mx, v);
        }
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      float sum = 0.f;
#pragma unroll
      for (int nt = 0; nt < kNT; ++nt) {
        const float e0 = __expf(sc[mt][nt][hf * 2] - mx), e1 = __expf(sc[mt][nt][hf * 2 + 1] - mx);
        sum += e0 + e1;
        __nv_bfloat162 h = __floats2bfloat162_rn(e0, e1);
        pp[mt][nt][hf] = *reinterpret_cast<uint32_t*>(&h);
      }
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      inv[mt][hf] = 1.f / sum;
    }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  float o[2][4][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int n4 = 0; n4 < 4; ++n4) o[mt][n4][0] = o[mt][n4][1] = o[mt][n4][2] = o[mt][n4][3] = 0.f;
#pragma unroll
  for (int ks = 0; ks < kKS; ++ks) {
#pragma unroll
    for (int dp = 0; dp < 2; ++dp) {  // two 16-dim halves of the head
      uint32_t b[4];
      const int mi = lane >> 3;
      const uint32_t addr = ptx::smem_u32(sV + (ks * 16 + (mi & 1) * 8 + (lane & 7)) * kRefPitch + warp * 32 + dp * 16 + (mi >> 1) * 8);
      asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                   : "=r"(b[0]), "=r"(b[1]), "=r"(b[2]), "=r"(b[3]) : "r"(addr));
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          float* c = o[mt][dp * 2 + j];
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                       : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                       : "r"(pp[mt][2 * ks][0]), "r"(pp[mt][2 * ks][1]), "r"(pp[mt][2 * ks + 1][0]), "r"(pp[mt][2 * ks + 1][1]),
                         "r"(b[2 * j]), "r"(b[2 * j + 1]));
        }
    }
  }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const int p = mt * 16 + (lane >> 2) + hf * 8;
      if (p >= np) continue;
      __nv_bfloat16* orow = out + (static_cast<long long>(crop) * np + p) * kD + dbase + (lane & 3) * 2;
#pragma unroll
      for (int n4 = 0; n4 < 4; ++n4) {
        __nv_bfloat162 h = __floats2bfloat162_rn(o[mt][n4][hf * 2] * inv[mt][hf], o[mt][n4][hf * 2 + 1] * inv[mt][hf]);
        *reinterpret_cast<__nv_bfloat162*>(orow + n4 * 8) = h;
      }
    }
}

// MM (MASK_NONE / MASK_CROP / MASK_STATE, lexicon.cuh): only the classes whose bit is set in the row's class mask
// compete.  MASK_CROP: mask [rows / rows_per_mask][4], bit c & 31 of word c >> 5.  MASK_STATE (row = crop, the unfused AR
// step): the allow row of the crop's state st_in[row]; an all-NaN row takes the lowest allowed class, and lx.state[row]
// becomes the chosen class's successor.  Lane `lane` visits classes lane + 32 k, so its bit of word k is bit `lane`.
template <int MM>
__global__ void k_argmax(const float* __restrict__ logits, int rows, int n_cls, int ld, int* __restrict__ ids,
                         int ids_stride, int* __restrict__ next, int next_stride, const int* __restrict__ forced,
                         int forced_stride, const uint32_t* __restrict__ mask, int rows_per_mask, LexDev lx,
                         const int* __restrict__ st_in) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* l = logits + static_cast<long long>(row) * ld;
  uint4 mw = make_uint4(~0u, ~0u, ~0u, ~0u);
  int st = 0;
  if constexpr (MM == MASK_CROP) mw = *reinterpret_cast<const uint4*>(mask + static_cast<long long>(row / rows_per_mask) * 4);
  if constexpr (MM == MASK_STATE) {
    st = st_in[row];
    mw = lx.allow[st];
  }
  const uint32_t mws[4] = {mw.x, mw.y, mw.z, mw.w};
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int c = lane, k = 0; c < n_cls; c += 32, ++k) {
    const float v = l[c];
    if ((MM == MASK_NONE || ((mws[k & 3] >> lane) & 1u)) && v > best) { best = v; bi = c; }  // strictly greater: first max per lane
  }
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }  // ties -> lowest index (at::max on CPU)
  }
  if (bi >= n_cls) bi = MM == MASK_STATE ? lowest_class(mws) : 0;  // all-NaN row: no comparison succeeded (the id is used as a table index downstream)
  if (lane == 0) {
    if (ids != nullptr) ids[static_cast<long long>(row) * ids_stride] = bi;
    if (next != nullptr) next[static_cast<long long>(row) * next_stride] = forced ? forced[static_cast<long long>(row) * forced_stride] : bi;
    if constexpr (MM == MASK_STATE) lx.state[row] = lx.next[lx.first[st] + classes_below(mws, bi)];
  }
}

// One row of the refinement head with scores: the argmax of k_argmax (same per-lane and cross-lane rules, so the ids are
// bit-identical) and the sum whose inverse is the row's largest softmax probability, p = 1 / sum_c exp(l[c] - max),
// summed per lane in class order and then over a fixed xor butterfly (every lane ends with the same bits), accurate
// expf: p is deterministic.  A row with a NaN gets p = NaN.  The second pass re-reads the row from L1.  MASK: the argmax
// and the sum both skip the classes whose bit is clear (p renormalised over the allowed classes); a mask that allows
// every class gives the bits of MASK = false.  `none`: the id of a row where no allowed class compares (all NaN).
// k_argmax_conf and k_lexicon_walk share it, so a one-state automaton gives k_argmax_conf's bits.
struct RowChoice {
  int id;
  float sum;
};
template <bool MASK>
__device__ __forceinline__ RowChoice argmax_conf_row(const float* l, int n_cls, int lane,
                                                     const uint32_t (&mws)[4], int none) {
  int bi = 0x7fffffff;
  float best = -INFINITY;
  for (int c = lane, k = 0; c < n_cls; c += 32, ++k) {
    const float v = l[c];
    if ((!MASK || ((mws[k & 3] >> lane) & 1u)) && v > best) { best = v; bi = c; }  // strictly greater: first max per lane
  }
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }  // ties -> lowest index (at::max on CPU)
  }
  if (bi >= n_cls) bi = none;  // all-NaN row
  float sum = 0.f;
  for (int c = lane, k = 0; c < n_cls; c += 32, ++k)
    if (!MASK || ((mws[k & 3] >> lane) & 1u)) sum += expf(l[c] - best);
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  return RowChoice{bi, sum};
}

// Refinement head with scores (argmax_conf_row per row); an all-NaN row gets id 0.
template <bool MASK>
__global__ void k_argmax_conf(const float* __restrict__ logits, int rows, int n_cls, int ld, int* __restrict__ ids,
                              float* __restrict__ pmax, const uint32_t* __restrict__ mask, int rows_per_mask) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* l = logits + static_cast<long long>(row) * ld;
  uint4 mw = make_uint4(~0u, ~0u, ~0u, ~0u);
  if constexpr (MASK) mw = *reinterpret_cast<const uint4*>(mask + static_cast<long long>(row / rows_per_mask) * 4);
  const uint32_t mws[4] = {mw.x, mw.y, mw.z, mw.w};
  const RowChoice r = argmax_conf_row<MASK>(l, n_cls, lane, mws, 0);
  if (lane == 0) {
    ids[row] = r.id;
    pmax[row] = 1.f / r.sum;
  }
}

// Refinement head of a lexicon request: one warp per crop walks its L rows in order from the crop's root, each row's
// choice being argmax_conf_row under the current state's allow row (an all-NaN row takes the lowest allowed class); the
// state then advances by the chosen class.  ids [n][L]; pmax (nullable) [n][L].
__global__ void k_lexicon_walk(const float* __restrict__ logits, int n, int L, int n_cls, int ld, LexDev lx,
                               int* __restrict__ ids, float* __restrict__ pmax) {
  const int crop = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (crop >= n) return;
  int st = lx.root[crop];
  for (int t = 0; t < L; ++t) {
    const long long row = static_cast<long long>(crop) * L + t;
    const uint4 mw = lx.allow[st];
    const uint32_t mws[4] = {mw.x, mw.y, mw.z, mw.w};
    const RowChoice r = argmax_conf_row<true>(logits + row * ld, n_cls, lane, mws, lowest_class(mws));
    if (lane == 0) {
      ids[row] = r.id;
      if (pmax != nullptr) pmax[row] = 1.f / r.sum;
    }
    st = lx.next[lx.first[st] + classes_below(mws, r.id)];
  }
}

// fp32 -> (hi, lo) bf16 pair with x ~= hi + lo (the split residual stream of gemm_tc.cuh, RES_SPLIT)
__global__ void k_split_f32(const float* __restrict__ x, long long n, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  const float v = x[i];
  const __nv_bfloat16 h = __float2bfloat16(v);
  hi[i] = h;
  lo[i] = __float2bfloat16(v - __bfloat162float(h));
}

__global__ void k_patchify(const uint8_t* __restrict__ crops, int n, __nv_bfloat16* __restrict__ out) {
  const int dy = blockIdx.x, b = blockIdx.y, dx = threadIdx.x;
  const uint8_t* p = crops + ((static_cast<size_t>(b) * 32 + dy) * 128 + dx) * 3;
  const size_t row = static_cast<size_t>(b) * 128 + (dy >> 2) * 16 + (dx >> 3);
  __nv_bfloat16* o = out + row * 96 + (dy & 3) * 8 + (dx & 7);
#pragma unroll
  for (int c = 0; c < 3; ++c) o[c * 32] = __float2bfloat16(static_cast<float>(p[c]));
}

}  // namespace

cudaError_t conv1_1_u8(const uint8_t* img, int B, int H, int W, const __nv_bfloat16* wt, const float* bias, __nv_bfloat16* out,
                       cudaStream_t s) {
  CUtensorMap tm;
  const cuuint64_t dims[4] = {64, static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(B)};
  const cuuint64_t strides[3] = {128, 128ull * W, 128ull * W * H};
  const cuuint32_t box[4] = {64, kC11TileW, 4, 1};
  if (!make_tmap_bf16(&tm, out, 4, dims, strides, box, 128)) return cudaErrorInvalidValue;
  TT_CUDA_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(k_conv1_1), kC11Smem));
  const int n_tiles = B * ((W + kC11TileW - 1) / kC11TileW) * ((H + kC11TileH - 1) / kC11TileH);
  int sms = 148;
  {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  k_conv1_1<<<std::min(n_tiles, 2 * sms), 256, kC11Smem, s>>>(img, H, W, n_tiles, wt, bias, tm);   // 2 persistent CTAs per SM (105 KB smem, 256 TMEM columns each)
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t maxpool2x2(const __nv_bfloat16* in, __nv_bfloat16* out, int B, int H, int W, int C, cudaStream_t s) {
  const long long total = static_cast<long long>(B) * (H / 2) * (W / 2) * (C / 8);
  k_maxpool2<<<grid_for(total, 256), 256, 0, s>>>(in, out, B, H, W, C);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}
cudaError_t maxpool3x3s1(const __nv_bfloat16* in, __nv_bfloat16* out, int B, int H, int W, int C, cudaStream_t s) {
  const long long total = static_cast<long long>(B) * H * W * (C / 8);
  k_maxpool3<<<grid_for(total, 256), 256, 0, s>>>(in, out, B, H, W, C);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}
cudaError_t upsample2x(const __nv_bfloat16* in, __nv_bfloat16* out, int B, int H, int W, int C, cudaStream_t s) {
  const long long total = static_cast<long long>(B) * 4 * H * W * (C / 8);
  // one element group per thread (no grid-stride tail): with 2368 blocks looping 23 times each the kernel sat at 24 % of
  // the HBM peak waiting on its four dependent loads (profiles/r1c_other_kernels.md)
  k_upsample2<<<static_cast<unsigned>((total + 255) / 256), 256, 0, s>>>(in, out, B, H, W, C);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t layernorm(const float* x, int rows, int D, const float* gamma, const float* beta, float eps,
                      __nv_bfloat16* ob, float* of, int rows_mod, cudaStream_t s) {
  if (rows <= 0) return cudaSuccess;
  const int grid = (rows + 7) / 8;
  if (D == 384) k_layernorm<12><<<grid, 256, 0, s>>>(x, rows, gamma, beta, eps, ob, of, rows_mod);
  else if (D == 192) k_layernorm<6><<<grid, 256, 0, s>>>(x, rows, gamma, beta, eps, ob, of, rows_mod);
  else { set_error("layernorm: unsupported width (PARSeq-base D = 384 or PARSeq-tiny D = 192)"); return cudaErrorInvalidValue; }
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t attention_enc(const __nv_bfloat16* qkv, __nv_bfloat16* out, int crops, int D, int heads, bool onepass,
                          cudaStream_t s) {
  if (crops <= 0) return cudaSuccess;
  if (D != heads * 64) { set_error("attention_enc: head dim must be 64"); return cudaErrorInvalidValue; }
  CUtensorMap tm;
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(3 * D), static_cast<cuuint64_t>(crops) * 128};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(3 * D) * 2};
  const cuuint32_t box[2] = {64, 128};
  if (!make_tmap_bf16(&tm, qkv, 2, dims, strides, box, 128)) return cudaErrorInvalidValue;
  const void* fn = onepass ? reinterpret_cast<const void*>(k_attn_enc<true>) : reinterpret_cast<const void*>(k_attn_enc<false>);
  TT_CUDA_TRY(ensure_dynamic_smem(fn, kAttnSmem));
  const float scale_log2e = 0.125f * 1.4426950408889634f;  // head_dim^-0.5 * log2(e)
  uint32_t* const trace = trace_dev();
  const uint32_t serial = trace ? trace_launch("k_attn_enc", 0 /* tracked per SM slot, not per CTA */, 128, kAttnSmem, s) : 0;
  if (onepass) k_attn_enc<true><<<dim3(heads, crops), 128, kAttnSmem, s>>>(tm, out, D, scale_log2e, trace, serial);
  else k_attn_enc<false><<<dim3(heads, crops), 128, kAttnSmem, s>>>(tm, out, D, scale_log2e, trace, serial);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t dec_context(const int* tokens, const float* embed, const float* posq, const float* g, const float* b,
                        float eps, int pos, int n, int D, int L, __nv_bfloat16* out, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  if (D == 384) k_dec_context<12><<<(n + 7) / 8, 256, 0, s>>>(tokens, embed, posq, g, b, eps, pos, n, L, out);
  else if (D == 192) k_dec_context<6><<<(n + 7) / 8, 256, 0, s>>>(tokens, embed, posq, g, b, eps, pos, n, L, out);
  else { set_error("dec_context: unsupported width"); return cudaErrorInvalidValue; }
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t dec_score_table(const float* q_table, const __nv_bfloat16* kv_table, int L, int n_tok, int D, int heads,
                            float* out, cudaStream_t s) {
  if (D != heads * 32) { set_error("dec_score_table: head dim must be 32"); return cudaErrorInvalidValue; }
  const long long total = static_cast<long long>(L) * L * n_tok * heads;
  k_dec_score_table<<<static_cast<unsigned>((total + 255) / 256), 256, 0, s>>>(q_table, kv_table, L, n_tok, D, heads, out);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t dec_self_attn(const DecoderStep& st, const float* q_table, const float* sc_table, const __nv_bfloat16* kv,
                          const int* tokens, int eos_id, int n_tok, __nv_bfloat16* out, cudaStream_t s) {
  if (st.n_crops <= 0) return cudaSuccess;
  if (st.D != st.heads * 32 || st.L > 32) { set_error("dec_self_attn: head dim must be 32, L <= 32"); return cudaErrorInvalidValue; }
  if (!st.refine && st.np == 1 && sc_table != nullptr && (st.heads == 12 || st.heads == 6) && st.D <= 512) {
    const int grid = (st.n_crops + 7) / 8;
    if (st.heads == 12) k_dec_self_attn_ar<12><<<grid, 256, 0, s>>>(st.n_crops, st.D, st.L, st.p0, n_tok, sc_table, kv, tokens, out, st.active, st.n_act);
    else k_dec_self_attn_ar<6><<<grid, 256, 0, s>>>(st.n_crops, st.D, st.L, st.p0, n_tok, sc_table, kv, tokens, out, st.active, st.n_act);
    TT_LAUNCH_CHECK();
    return cudaSuccess;
  }
  if (st.refine && st.p0 == 0 && st.np == st.L && st.D == 384) {
    constexpr int smem = 2 * 32 * kRefPitch * 2;
    k_dec_attn_refine<32, true><<<dim3(3, st.n_crops), 128, smem, s>>>(q_table, kv, st.L, st.np, tokens, eos_id, st.L, n_tok, out);
    TT_LAUNCH_CHECK();
    return cudaSuccess;
  }
  k_dec_self_attn<<<dim3(st.np, st.n_crops), st.heads * 32, 0, s>>>(st, q_table, kv, tokens, eos_id, n_tok, out);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t dec_cross_attn(const DecoderStep& st, const __nv_bfloat16* q, const __nv_bfloat16* mem_kv,
                           __nv_bfloat16* out, cudaStream_t s) {
  if (st.n_crops <= 0) return cudaSuccess;
  if (!((st.D == 384 && st.heads == 12) || (st.D == 192 && st.heads == 6))) {
    set_error("dec_cross_attn: built for PARSeq-base (D = 384, 12 heads) and PARSeq-tiny (D = 192, 6 heads)");
    return cudaErrorInvalidValue;
  }
  if (st.D == 384 && st.np > 1 && st.np <= 32) {
    constexpr int smem = 2 * 128 * kRefPitch * 2;
    TT_CUDA_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(k_dec_attn_refine<128, false>), smem));
    k_dec_attn_refine<128, false><<<dim3(3, st.n_crops), 128, smem, s>>>(q, mem_kv, 128, st.np, nullptr, 0, st.L, 0, out);
    TT_LAUNCH_CHECK();
    return cudaSuccess;
  }
  // with an active list the live count is only known on the device: a bounded grid whose blocks stride over the slots
  const int gy = st.n_act ? std::min(st.n_crops, 8 * 148) : st.n_crops;   // 8 blocks per B200 SM
  if (st.D == 384) k_dec_cross_attn<384><<<dim3(st.np, gy), 384, 0, s>>>(st, q, mem_kv, out);
  else k_dec_cross_attn<192><<<dim3(st.np, gy), 192, 0, s>>>(st, q, mem_kv, out);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

// Order-preserving compaction of the AR pass's active list (one block: a half-batch is a few thousand crops).
__global__ void __launch_bounds__(1024) k_dec_compact(const int* __restrict__ active_in, const int* __restrict__ n_in, int n,
                                                      const int* __restrict__ tokens, int L, int pos, int eos_id,
                                                      int* __restrict__ active_out, int* __restrict__ n_out) {
  __shared__ int s_off[32];    // exclusive offsets of the 32 warps inside a 1024-slot chunk
  __shared__ int s_total;      // kept slots of the chunk
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_slots = n_in ? *n_in : n;
  int base = 0;                // kept slots of the chunks before this one (the same in every thread)
  for (int s0 = 0; s0 < n_slots; s0 += 1024) {
    const int slot = s0 + threadIdx.x;
    int crop = 0;
    bool keep = false;
    if (slot < n_slots) {
      crop = active_in ? active_in[slot] : slot;
      keep = tokens[static_cast<long long>(crop) * L + pos] != eos_id;
    }
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
    if (keep) active_out[base + s_off[warp] + __popc(m & ((1u << lane) - 1u))] = crop;
    base += s_total;
    __syncthreads();           // s_off / s_total are rewritten by the next chunk
  }
  if (threadIdx.x == 0) *n_out = base;
}

cudaError_t dec_compact(const int* active_in, const int* n_in, int n, const int* tokens, int L, int pos, int eos_id,
                        int* active_out, int* n_out, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  k_dec_compact<<<1, 1024, 0, s>>>(active_in, n_in, n, tokens, L, pos, eos_id, active_out, n_out);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

// tokens[crop][0] = bos, the rest pad: the AR context before the first step (upstream PARSeq forward(): tgt_in)
__global__ void k_tokens_init(int* __restrict__ tokens, int n, int L, int bos, int pad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n * L) tokens[i] = (i % L == 0) ? bos : pad;
}
cudaError_t tokens_init(int* tokens, int n, int L, int bos, int pad, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  k_tokens_init<<<(n * L + 255) / 256, 256, 0, s>>>(tokens, n, L, bos, pad);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t argmax_rows(const float* logits, int rows, int n_cls, int ld, int* ids, int ids_stride, int* next,
                        int next_stride, const int* forced, int forced_stride, cudaStream_t s, const uint32_t* mask,
                        int rows_per_mask, const LexDev* lex, bool first_step) {
  if (rows <= 0) return cudaSuccess;
  if (lex)
    k_argmax<MASK_STATE><<<(rows + 7) / 8, 256, 0, s>>>(logits, rows, n_cls, ld, ids, ids_stride, next, next_stride, forced,
                                                        forced_stride, nullptr, 1, *lex, first_step ? lex->root : lex->state);
  else if (mask)
    k_argmax<MASK_CROP><<<(rows + 7) / 8, 256, 0, s>>>(logits, rows, n_cls, ld, ids, ids_stride, next, next_stride, forced,
                                                       forced_stride, mask, rows_per_mask, LexDev{}, nullptr);
  else
    k_argmax<MASK_NONE><<<(rows + 7) / 8, 256, 0, s>>>(logits, rows, n_cls, ld, ids, ids_stride, next, next_stride, forced,
                                                       forced_stride, nullptr, 1, LexDev{}, nullptr);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t argmax_conf_rows(const float* logits, int rows, int n_cls, int ld, int* ids, float* pmax, cudaStream_t s,
                             const uint32_t* mask, int rows_per_mask) {
  if (rows <= 0) return cudaSuccess;
  if (mask)
    k_argmax_conf<true><<<(rows + 7) / 8, 256, 0, s>>>(logits, rows, n_cls, ld, ids, pmax, mask, rows_per_mask);
  else
    k_argmax_conf<false><<<(rows + 7) / 8, 256, 0, s>>>(logits, rows, n_cls, ld, ids, pmax, nullptr, 1);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t lexicon_walk(const float* logits, int n, int L, int n_cls, int ld, const LexDev& lex, int* ids, float* pmax,
                         cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  k_lexicon_walk<<<(n + 7) / 8, 256, 0, s>>>(logits, n, L, n_cls, ld, lex, ids, pmax);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t split_f32(const float* x, long long n, __nv_bfloat16* hi, __nv_bfloat16* lo, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  k_split_f32<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(x, n, hi, lo);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t patchify_u8(const uint8_t* crops, int n, __nv_bfloat16* out, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  k_patchify<<<dim3(32, n), 128, 0, s>>>(crops, n, out);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

}  // namespace tt
