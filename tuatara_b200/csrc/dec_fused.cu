// Fused dense kernels of the PARSeq decoder's AR loop: see dec_fused.cuh for what they replace and why.
//
// Layout of one CTA (320 threads, 128 crops = 128 TMEM lanes):
//   warp 0      TMA producer : the CTA's 128 input rows -> sA once, then every weight tile of the step, in a static
//                              order, through a ring of [128 weight rows][64 k] SWIZZLE_128B units
//   warp 1      MMA issuer   : tcgen05.mma M=128, N<=128 per unit, fp32 accumulators in TMEM
//   warps 2..9  row owners   : thread = crop = TMEM lane, two warps per lane quadrant splitting a phase's columns.
//                              LayerNorm / GELU / bias in registers; results go back to smem as the next GEMM's A operand
//                              (K-major SWIZZLE_128B, written with the same XOR the TMA uses)
// TMEM columns [0, D) hold the residual row t for the whole kernel: `t += x W^T` is an accumulating MMA onto those
// columns, the fp32 input row is written there with tcgen05.st.  Columns [D, D+128) take the GEMMs whose result feeds an
// activation (l1 chunk, head).  MMA and row-owner phases alternate; they meet on a 288-thread named barrier (A operand /
// TMEM ready for the tensor core) and on two mbarriers the MMA warp commits to in turn (accumulator ready for the rows).
#include "dec_fused.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <math.h>

#include "common.h"
#include "epi_math.cuh"
#include "gemm_tc.cuh"
#include "lexicon.cuh"
#include "ptx.cuh"

namespace tt {

namespace {

constexpr int kUnit = 16384;   // [128 rows][64 bf16]
constexpr int kRowThreads = 256;            // 8 row-owner warps: two per TMEM lane quadrant
constexpr int kThreads = 64 + kRowThreads;  // + TMA producer warp + MMA issuer warp
constexpr int kTmemCols = 512;
constexpr int kMaxStages = 8;

enum { MODE_B = 0, MODE_A2 = 1 };

struct DenseParams {
  CUtensorMap tm_in;                     // [n][D] bf16 activation rows of this step, box {64, 128}
  CUtensorMap tm_w0, tm_w1, tm_w2, tm_wh;
  const float* vec_src;                  // the kernel's per-column vectors, packed in smem order (dec_dense_init): one bulk copy
  float* t_scratch;                      // [tiles][D][128]
  __nv_bfloat16* q_out;                  // A2
  float* logits;                         // B: [n][L][ncp]
  int* tokens;                           // B: [n][L]
  const int* forced;                     // B: [n][L-1] or null
  int n, L, step, n_cls, ncp;
  // early-exit AR pass: rows are the first *n_act slots of `active` (slot -> crop; logits / tokens are indexed by crop).
  // Both null: n rows, slot == crop.
  const int* active;
  const int* n_act;
  unsigned long long* dbg;               // TT_DEC_DEBUG=1 (development): role cycle counters of CTA 0
  const uint32_t* mask;                  // B, MASK_CROP only: [n][4] class masks, indexed by crop like tokens
  // B, MASK_STATE only (lexicon.h): the automaton table and the crops' states, indexed by crop like tokens
  const int* st_in;                      // state of each crop before this step (the roots at step 0)
  int* st_out;                           // its state after this step's token
  const uint4* lx_allow;
  const int* lx_first;
  const int* lx_next;
};

struct alignas(16) Ctl {
  uint64_t full[kMaxStages], empty[kMaxStages];
  uint64_t a_full, vec_full;
  uint64_t md[2];
  uint32_t tmem_base;
};

// 32 consecutive floats of a per-column vector in smem (explicit LDS.128: the dynamic-smem pointers decay to generic)
__device__ __forceinline__ void lds_f32x32(uint32_t addr, float (&o)[32]) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint4 u = ptx::lds128(addr + i * 16);
    o[4 * i] = __uint_as_float(u.x); o[4 * i + 1] = __uint_as_float(u.y);
    o[4 * i + 2] = __uint_as_float(u.z); o[4 * i + 3] = __uint_as_float(u.w);
  }
}

template <int D, int MLP, int MODE>
struct Cfg {
  static constexpr int KB = D / 64;
  static constexpr int kStages = MODE == MODE_B ? 5 : 6;
  static constexpr int kVec = MODE == MODE_B ? 6 * D + MLP + 128 : 4 * D;
  static constexpr int kXch = MODE == MODE_B ? 0 : 2 * 128 * 2 * 4;   // statistics exchange of the row-owner halves (MODE_B: inside sH)
  static constexpr int kSmem = KB * kUnit + (MODE == MODE_B ? 2 * kUnit : 0) + kStages * kUnit + kVec * 4 + static_cast<int>(sizeof(Ctl)) + kXch + 1024;
  static_assert(D % 64 == 0 && D + 128 <= kTmemCols && MLP % 128 == 0, "decoder width");
  static_assert(kSmem <= 227 * 1024, "shared memory budget");
};

// MM (MODE_B only, lexicon.cuh): the greedy token is the argmax over the classes allowed by the crop's class mask
// (MASK_CROP) or by its automaton state (MASK_STATE: an all-NaN row takes the lowest allowed class, and the state
// advances by the chosen class).
template <int D, int MLP, int MODE, int MM>
__global__ void __launch_bounds__(kThreads, 1) k_dec_dense(const __grid_constant__ DenseParams p) {
  using C = Cfg<D, MLP, MODE>;
  constexpr int KB = C::KB, kStages = C::kStages;
  constexpr int NC = MLP / 128;          // hidden chunks of the MLP
  constexpr float kEps = 1e-5f;          // nn.LayerNorm default (PARSeq decoder)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sH = sA + KB * kUnit;
  uint8_t* ring = sH + (MODE == MODE_B ? 2 * kUnit : 0);
  float* vec = reinterpret_cast<float*>(ring + kStages * kUnit);
  Ctl* ctl = reinterpret_cast<Ctl*>(vec + C::kVec);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int tile = blockIdx.x;
  const int n_rows = p.n_act ? *p.n_act : p.n;   // live rows of this step (the grid covers all n)
  if (tile * 128 >= n_rows) return;              // the whole CTA, before any barrier or TMEM allocation
  const long long t_entry = (p.dbg != nullptr && blockIdx.x == 0) ? clock64() : 0;

  if (threadIdx.x == 0) {
    ptx::prefetch_tmap(&p.tm_in);
    ptx::prefetch_tmap(&p.tm_w0);
    ptx::prefetch_tmap(&p.tm_w1);
    for (int s = 0; s < kStages; ++s) { ptx::mbar_init(&ctl->full[s], 1); ptx::mbar_init(&ctl->empty[s], 1); }
    ptx::mbar_init(&ctl->a_full, 1);
    ptx::mbar_init(&ctl->vec_full, 1);
    ptx::mbar_init(&ctl->md[0], 1);
    ptx::mbar_init(&ctl->md[1], 1);
    ptx::fence_barrier_init();
    // per-column vectors (biases, LayerNorm weights: packed in smem order at init) -> smem with ONE bulk copy that
    // runs under the rest of the prologue; the row owners wait for it before their first phase.  (Per-thread staging
    // loops took 12 000 cycles of a 100 000-cycle kernel.)
    ptx::mbar_arrive_expect_tx(&ctl->vec_full, C::kVec * 4);
    ptx::bulk_load(vec, p.vec_src, C::kVec * 4, &ctl->vec_full);
  }
  if (warp == 1) ptx::tmem_alloc(&ctl->tmem_base, kTmemCols);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, ctl->tmem_base, 0);
  if (p.dbg != nullptr && blockIdx.x == 0 && threadIdx.x == 0) p.dbg[5] = clock64() - t_entry;   // prologue

  if (warp == 0) {
    // ------------------------------------------------------------------------------ TMA producer
    int stage = 0;
    uint32_t phase = 0;
    const bool pdbg = p.dbg != nullptr && blockIdx.x == 0;
    long long p_wait = 0;
    const long long p_start = pdbg ? clock64() : 0;
    auto load = [&](const CUtensorMap* tm, int n_base, int k_base, int N, int K, int box_rows) {
      for (int kb = 0; kb < K / 64; ++kb)
        for (int n0 = 0; n0 < N; n0 += 128) {
          { const long long t0 = pdbg ? clock64() : 0; ptx::mbar_wait(&ctl->empty[stage], phase ^ 1); __syncwarp(); p_wait += pdbg ? clock64() - t0 : 0; }
          ptx::mbar_arrive_expect_tx_e(&ctl->full[stage], static_cast<uint32_t>(box_rows) * 128u);
          ptx::tma_load_2d_e(ring + stage * kUnit, tm, &ctl->full[stage], k_base + kb * 64, n_base + n0);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
    };
    ptx::mbar_arrive_expect_tx_e(&ctl->a_full, KB * kUnit);   // rows past n arrive as zeros
    for (int kb = 0; kb < KB; ++kb) ptx::tma_load_2d_e(sA + kb * kUnit, &p.tm_in, &ctl->a_full, kb * 64, tile * 128);
    if constexpr (MODE == MODE_A2) {
      load(&p.tm_w0, 0, 0, D, D, 128);
      load(&p.tm_w1, 0, 0, D, D, 128);
    } else {
      load(&p.tm_w0, 0, 0, D, D, 128);
      for (int c = 0; c < NC; ++c) {
        load(&p.tm_w1, c * 128, 0, 128, D, 128);
        load(&p.tm_w2, 0, c * 128, D, 128, 128);
      }
      load(&p.tm_wh, 0, 0, p.ncp, D, p.ncp < 128 ? p.ncp : 128);
    }
    if (pdbg && lane == 0) { p.dbg[3] = p_wait; p.dbg[4] = clock64() - p_start; }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------- MMA issuer
    int stage = 0;
    uint32_t phase = 0, cnt = 0;
    const bool dbg = p.dbg != nullptr && blockIdx.x == 0;
    long long w_full = 0, w_bar = 0;
    const long long t_start = dbg ? clock64() : 0;
    // acc[:, dcol + [0, N)) (+)= A[128 x K] * W[N x K]^T, units in the producer's order (k-block outer, 128-row chunk inner)
    auto gemm = [&](uint32_t a_addr0, int N, int K, uint32_t dcol, bool acc) {
      for (int kb = 0; kb < K / 64; ++kb)
        for (int n0 = 0; n0 < N; n0 += 128) {
          const int nn = N - n0 < 128 ? N - n0 : 128;
          { const long long t0 = dbg ? clock64() : 0; ptx::mbar_wait(&ctl->full[stage], phase); __syncwarp(); w_full += dbg ? clock64() - t0 : 0; }
          ptx::tc_fence_after();
          const uint32_t b_addr = ptx::smem_u32(ring + stage * kUnit);
          const uint32_t idesc = ptx::make_idesc_bf16(128, nn);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            ptx::mma_bf16_e(tmem_base + dcol + n0, ptx::make_smem_desc(a_addr0 + kb * kUnit + k * 32, 128),
                            ptx::make_smem_desc(b_addr + k * 32, 128), idesc, (acc || kb > 0 || k > 0) ? 1u : 0u);
          ptx::mma_commit_e(&ctl->empty[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
    };
    auto commit_md = [&]() { ptx::mma_commit_e(&ctl->md[cnt & 1]); ++cnt; };
    auto rows_done = [&]() {
      const long long t0 = dbg ? clock64() : 0;
      ptx::tc_fence_before(); ptx::named_bar_sync<1, 32 + kRowThreads>(); ptx::tc_fence_after();
      w_bar += dbg ? clock64() - t0 : 0;
    };
    const uint32_t a_addr = ptx::smem_u32(sA), h_addr = ptx::smem_u32(sH);
    ptx::mbar_wait(&ctl->a_full, 0); __syncwarp();
    ptx::tc_fence_after();
    if constexpr (MODE == MODE_A2) {
      gemm(a_addr, D, D, 0, false);     // t = ab Wo^T
      commit_md();
      rows_done();                      // t saved, LN1(t) in sA
      gemm(a_addr, D, D, 0, false);     // q = LN1(t) Wq^T
      commit_md();
    } else {
      gemm(a_addr, D, D, 0, false);     // ab2 Wco^T
      commit_md();
      rows_done();                      // t (fp32) back in TMEM columns [0, D), LN2(t) in sA
      gemm(a_addr, 128, D, D, false);   // hidden chunk 0
      commit_md();
      for (int c = 0; c < NC; ++c) {
        rows_done();                    // GELU(hidden chunk c) in sH
        gemm(h_addr, D, 128, 0, true);  // t += GELU(h_c) W2[:, c]^T
        if (c + 1 < NC) gemm(a_addr, 128, D, D, false);
        commit_md();
      }
      rows_done();                      // LN(t) in sA
      gemm(a_addr, p.ncp, D, D, false); // head
      commit_md();
    }
    if (dbg && lane == 0) { p.dbg[0] = w_full; p.dbg[1] = w_bar; p.dbg[2] = clock64() - t_start; }
  } else {
    // ------------------------------------------------- row owners (thread = crop; two warps per TMEM lane quadrant)
    // Warps 2..5 take the lower half of a phase's columns, warps 6..9 the upper half of the same rows: LayerNorm's
    // (sum, sum of squares) and the head's argmax are combined through a small smem exchange.
    const int q = warp & 3;                       // TMEM lane quadrant this warp may access
    const int half = (warp - 2) >> 2;
    const int r = q * 32 + lane;
    const long long m = static_cast<long long>(tile) * 128 + r;
    const bool valid = m < n_rows;   // rows past the live count hold stale activations: computed, never stored
    const uint32_t tl = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    uint32_t ecnt = 0;
    auto wait_md = [&]() { ptx::mbar_wait(&ctl->md[ecnt & 1], (ecnt >> 1) & 1); ++ecnt; ptx::tc_fence_after(); };
    auto rows_done = [&]() { ptx::fence_proxy_async(); ptx::tc_fence_before(); ptx::named_bar_sync<1, 32 + kRowThreads>(); };
    float* const xch = reinterpret_cast<float*>(MODE == MODE_B ? sH : reinterpret_cast<uint8_t*>(ctl + 1));   // [2][128][2] floats
    // this thread's 32-column blocks [b0, b1) of TMEM columns tbase + blk * 32, the next block's load in flight while
    // the current one is processed
    auto for_blocks = [&](uint32_t tbase, int b0, int b1, auto&& f) {
      uint32_t ra[32], rb[32];
      if (b0 < b1) ptx::tmem_ld<32>(tbase + b0 * 32, ra);
#pragma unroll 1
      for (int blk = b0; blk < b1; blk += 2) {
        ptx::tmem_ld_wait(ra);
        if (blk + 1 < b1) ptx::tmem_ld<32>(tbase + (blk + 1) * 32, rb);
        f(blk, ra);
        if (blk + 1 < b1) {
          ptx::tmem_ld_wait(rb);
          if (blk + 2 < b1) ptx::tmem_ld<32>(tbase + (blk + 2) * 32, ra);
          f(blk + 1, rb);
        }
      }
    };
    // 32 bf16 columns [col0, col0 + 32) of this thread's row into a K-major SWIZZLE_128B operand buffer
    auto store_row32 = [&](uint8_t* base, int col0, const float (&y)[32]) {
      const uint32_t rowaddr = ptx::smem_u32(base) + (col0 >> 6) * kUnit + r * 128;
      const int j0 = (col0 & 32) >> 3;
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        uint4 o;
        o.x = pack_bf16(y[8 * jj + 0], y[8 * jj + 1]); o.y = pack_bf16(y[8 * jj + 2], y[8 * jj + 3]);
        o.z = pack_bf16(y[8 * jj + 4], y[8 * jj + 5]); o.w = pack_bf16(y[8 * jj + 6], y[8 * jj + 7]);
        ptx::sts128(rowaddr + (((j0 + jj) ^ (r & 7)) << 4), o);
      }
    };
    const uint32_t vec_s = ptx::smem_u32(vec);
    ptx::mbar_wait(&ctl->vec_full, 0);
    constexpr int kDB = D / 32;                    // 32-column blocks of a row
    const int db0 = half * (kDB / 2), db1 = db0 + kDB / 2;
    // row statistics from the two halves' partial sums -> (mean, rstd)
    auto combine_stats = [&](float s1, float s2, float& mean, float& rstd) {
      xch[(half * 128 + r) * 2] = s1;
      xch[(half * 128 + r) * 2 + 1] = s2;
      ptx::named_bar_sync<2, kRowThreads>();
      s1 += xch[((half ^ 1) * 128 + r) * 2];
      s2 += xch[((half ^ 1) * 128 + r) * 2 + 1];
      mean = s1 * (1.f / D);
      rstd = rsqrtf(fmaxf(s2 * (1.f / D) - mean * mean, 0.f) + kEps);
    };
    // LayerNorm of the row held in TMEM columns [0, D) (+ bias vector `add`) -> bf16 -> sA  (add / g / b: float offsets
    // into `vec`; add < 0: none)
    auto layernorm_to_sA = [&](int add, int g, int b, float mean, float rstd) {
      for_blocks(tl, db0, db1, [&](int blk, uint32_t (&raw)[32]) {
        float y[32], gv[32], bv[32];
        if (add >= 0) lds_f32x32(vec_s + (add + blk * 32) * 4, y);
        lds_f32x32(vec_s + (g + blk * 32) * 4, gv);
        lds_f32x32(vec_s + (b + blk * 32) * 4, bv);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float x = __uint_as_float(raw[j]) + (add >= 0 ? y[j] : 0.f);
          y[j] = (x - mean) * rstd * gv[j] + bv[j];
        }
        store_row32(sA, blk * 32, y);
      });
    };
    float* const tcol = p.t_scratch + static_cast<size_t>(tile) * D * 128 + r;

    if constexpr (MODE == MODE_A2) {
      wait_md();
      float sum = 0.f, sq = 0.f;
      for_blocks(tl, db0, db1, [&](int blk, uint32_t (&raw)[32]) {
        float av[32];
        lds_f32x32(vec_s + blk * 32 * 4, av);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float x = __uint_as_float(raw[j]) + av[j];   // + sa.out bias + pos_queries[step]
          sum += x; sq += x * x;
          tcol[static_cast<size_t>(blk * 32 + j) * 128] = x;            // lanes = consecutive crops: coalesced
        }
      });
      float mean, rstd;
      combine_stats(sum, sq, mean, rstd);
      layernorm_to_sA(0, D, 2 * D, mean, rstd);
      rows_done();
      wait_md();
      __nv_bfloat16* qrow = p.q_out + m * D;
      for_blocks(tl, db0, db1, [&](int blk, uint32_t (&raw)[32]) {
        float bq[32];
        lds_f32x32(vec_s + (3 * D + blk * 32) * 4, bq);
        if (valid) {
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            float v[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = __uint_as_float(raw[8 * jj + e]) + bq[8 * jj + e];
            uint4 o;
            o.x = pack_bf16(v[0], v[1]); o.y = pack_bf16(v[2], v[3]); o.z = pack_bf16(v[4], v[5]); o.w = pack_bf16(v[6], v[7]);
            *reinterpret_cast<uint4*>(qrow + blk * 32 + 8 * jj) = o;
          }
        }
      });
    } else {
      // ---- t = t_in + ca.out(ab2) + bias: into TMEM as fp32, LN2 -> sA
      float tin[2][32];
#pragma unroll
      for (int j = 0; j < 32; ++j) tin[0][j] = tcol[static_cast<size_t>(db0 * 32 + j) * 128];
      wait_md();
      float sum = 0.f, sq = 0.f;
      {
        uint32_t raw[32];
#pragma unroll
        for (int i = 0; i < kDB / 2; ++i) {
          const int blk = db0 + i;
          ptx::tmem_ld<32>(tl + blk * 32, raw);
          if (i + 1 < kDB / 2) {
#pragma unroll
            for (int j = 0; j < 32; ++j) tin[(i + 1) & 1][j] = tcol[static_cast<size_t>((blk + 1) * 32 + j) * 128];
          }
          float av[32];
          lds_f32x32(vec_s + blk * 32 * 4, av);
          ptx::tmem_ld_wait(raw);
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float x = __uint_as_float(raw[j]) + av[j] + tin[i & 1][j];
            sum += x; sq += x * x;
            raw[j] = __float_as_uint(x);
          }
          ptx::tmem_st32(tl + blk * 32, raw);
          ptx::tmem_st_wait();
        }
      }
      {
        float mean, rstd;
        combine_stats(sum, sq, mean, rstd);
        layernorm_to_sA(-1, D, 2 * D, mean, rstd);
      }
      rows_done();
      // ---- MLP: GELU(l1 chunk) -> sH, chunk by chunk (the l2 MMAs accumulate onto t)
#pragma unroll 1
      for (int c = 0; c < NC; ++c) {
        wait_md();
        for_blocks(tl + D, half * 2, half * 2 + 2, [&](int b4, uint32_t (&raw)[32]) {
          float y[32], b1[32];
          lds_f32x32(vec_s + (3 * D + c * 128 + b4 * 32) * 4, b1);
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            const uint64_t v = gelu_fast2(add2(pk2u(raw[j], raw[j + 1]), pk2(b1[j], b1[j + 1])));
            upk2(v, y[j], y[j + 1]);
          }
          store_row32(sH, b4 * 32, y);
        });
        rows_done();
      }
      // ---- final norm of t (+ l2 bias) -> sA
      wait_md();
      {
        float s1 = 0.f, s2 = 0.f;
        for_blocks(tl, db0, db1, [&](int blk, uint32_t (&raw)[32]) {
          float b2[32];
          lds_f32x32(vec_s + (3 * D + MLP + blk * 32) * 4, b2);
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float x = __uint_as_float(raw[j]) + b2[j];
            s1 += x; s2 += x * x;
          }
        });
        float mean, rstd;
        combine_stats(s1, s2, mean, rstd);
        layernorm_to_sA(3 * D + MLP, 4 * D + MLP, 5 * D + MLP, mean, rstd);
      }
      rows_done();
      // ---- head: logits row + greedy token (the halves' maxima meet in smem; the lower half holds the lower classes)
      // MASK_STATE: the crop's state and its allow row are loaded before the accumulator wait, so that the two dependent
      // loads overlap it; half 0 also fetches where the state's successors start.
      int st = 0, st_first = 0;
      uint4 st_mw = make_uint4(~0u, ~0u, ~0u, ~0u);
      if constexpr (MM == MASK_STATE) {
        if (valid) {
          const long long crop = p.active ? p.active[m] : m;
          st = p.st_in[crop];
          st_mw = p.lx_allow[st];
          if (half == 0) st_first = p.lx_first[st];
        }
      }
      wait_md();
      {
        const long long crop = (valid && p.active) ? p.active[m] : m;
        float* lrow = p.logits + (crop * p.L + p.step) * p.ncp;
        // MASK_CROP: the crop's class mask, one 16-byte load (rows past the live count compete unmasked: never stored)
        uint4 mw = make_uint4(~0u, ~0u, ~0u, ~0u);
        if constexpr (MM == MASK_CROP) {
          if (valid) mw = *reinterpret_cast<const uint4*>(p.mask + crop * 4);
        }
        if constexpr (MM == MASK_STATE) mw = st_mw;
        const uint32_t mws[4] = {mw.x, mw.y, mw.z, mw.w};
        float best = -INFINITY;
        int bi = MM == MASK_STATE ? lowest_class(mws) : 0;
        const int nb = p.ncp / 32, hb0 = half ? (nb + 1) / 2 : 0, hb1 = half ? nb : (nb + 1) / 2;
        for_blocks(tl + D, hb0, hb1, [&](int blk, uint32_t (&raw)[32]) {
          float l[32];
          lds_f32x32(vec_s + (6 * D + MLP + blk * 32) * 4, l);
          const uint32_t bits = MM != MASK_NONE ? (blk == 0 ? mw.x : blk == 1 ? mw.y : blk == 2 ? mw.z : mw.w) : ~0u;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            l[j] += __uint_as_float(raw[j]);
            if (blk * 32 + j < p.n_cls && (MM == MASK_NONE || ((bits >> j) & 1u)) && l[j] > best) { best = l[j]; bi = blk * 32 + j; }   // first max wins (at::max on CPU)
          }
          if (valid) {
#pragma unroll
            for (int jj = 0; jj < 8; ++jj)
              *reinterpret_cast<float4*>(lrow + blk * 32 + 4 * jj) = make_float4(l[4 * jj], l[4 * jj + 1], l[4 * jj + 2], l[4 * jj + 3]);
          }
        });
        if (half == 1) { xch[r * 2] = best; xch[r * 2 + 1] = __int_as_float(bi); }
        ptx::named_bar_sync<2, kRowThreads>();
        if (half == 0) {
          const float ob = xch[r * 2];
          if (ob > best) { best = ob; bi = __float_as_int(xch[r * 2 + 1]); }
          if (valid && p.step + 1 < p.L)
            p.tokens[crop * p.L + p.step + 1] = p.forced ? p.forced[crop * (p.L - 1) + p.step] : bi;
          if constexpr (MM == MASK_STATE) {
            if (valid) p.st_out[crop] = p.lx_next[st_first + classes_below(mws, bi)];
          }
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (p.dbg != nullptr && blockIdx.x == 0 && threadIdx.x == 0) p.dbg[6] = clock64() - t_entry;   // entry -> all roles done
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

bool make_w_map(CUtensorMap* m, const __nv_bfloat16* w, int N, int K) {
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(N)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(K) * 2};
  const cuuint32_t box[2] = {64, static_cast<cuuint32_t>(N < 128 ? N : 128)};
  return make_tmap_bf16(m, w, 2, dims, strides, box, 128);
}

bool make_in_map(CUtensorMap* m, const __nv_bfloat16* a, int n, int D) {
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(D), static_cast<cuuint64_t>(n)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(D) * 2};
  const cuuint32_t box[2] = {64, 128};
  return make_tmap_bf16(m, a, 2, dims, strides, box, 128);
}

int dense_priority() {
  static const int prio = [] {
    int lo = 0, hi = 0;   // "greatest" priority is the numerically lowest value
    if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess) { cudaGetLastError(); return 0; }
    const char* e = std::getenv("TT_DEC_PRIO");
    return (e && std::atoi(e) == 0) ? 0 : hi;
  }();
  return prio;
}

template <int D, int MLP, int MODE, int MM = MASK_NONE>
cudaError_t launch_dense(const DenseParams& p, cudaStream_t s) {
  using C = Cfg<D, MLP, MODE>;
  TT_CUDA_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(k_dec_dense<D, MLP, MODE, MM>), C::kSmem));
  // Highest launch priority: a CTA needs a whole SM (216 KB smem, 512 TMEM columns).  Next to the other half-batch's
  // cross-attention grid (thousands of small blocks, launched earlier) it would otherwise wait for that grid to drain.
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((p.n + 127) / 128);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = C::kSmem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributePriority;
  at[0].val.priority = dense_priority();
  cfg.attrs = at;
  cfg.numAttrs = 1;
  static const bool dbg_env = std::getenv("TT_DEC_DEBUG") && std::atoi(std::getenv("TT_DEC_DEBUG")) != 0;
  static unsigned long long* dbg_buf = nullptr;
  DenseParams pp = p;
  if (dbg_env) {
    if (!dbg_buf) cudaMalloc(&dbg_buf, 8 * sizeof(unsigned long long));
    cudaMemsetAsync(dbg_buf, 0, 8 * sizeof(unsigned long long), s);
    pp.dbg = dbg_buf;
  }
  TT_CUDA_TRY(cudaLaunchKernelEx(&cfg, k_dec_dense<D, MLP, MODE, MM>, pp));
  TT_LAUNCH_CHECK();
  if (dbg_env && p.step == 13) {
    unsigned long long h[8];
    cudaStreamSynchronize(s);
    cudaMemcpy(h, dbg_buf, sizeof(h), cudaMemcpyDeviceToHost);
    std::fprintf(stderr, "[dec dbg] mode %d n %d: mma wait-full %llu wait-rows %llu total %llu | producer wait-empty %llu total %llu | prologue %llu entry-to-done %llu\n",
                 MODE, p.n, h[0], h[1], h[2], h[3], h[4], h[5], h[6]);
  }
  return cudaSuccess;
}

}  // namespace

bool dec_dense_supported(int D, int mlp, int ncp) {
  return ((D == 384 && mlp == 1536) || (D == 192 && mlp == 768)) && ncp % 32 == 0 && ncp <= 128;
}

size_t dec_dense_scratch_floats(int n, int D) { return static_cast<size_t>((n + 127) / 128) * D * 128; }

bool dec_dense_init(DecDenseWeights* w, int D, int mlp, int n_cls, int ncp, int L, const __nv_bfloat16* wo,
                    const __nv_bfloat16* wq, const __nv_bfloat16* wco, const __nv_bfloat16* w1, const __nv_bfloat16* w2,
                    const __nv_bfloat16* wh) {
  w->D = D; w->mlp = mlp; w->n_cls = n_cls; w->ncp = ncp; w->L = L;
  w->ready = false;
  if (!dec_dense_supported(D, mlp, ncp)) return true;   // not an error: the caller keeps the unfused path
  if (!make_w_map(&w->tm_wo, wo, D, D) || !make_w_map(&w->tm_wq, wq, D, D) || !make_w_map(&w->tm_wco, wco, D, D) ||
      !make_w_map(&w->tm_w1, w1, mlp, D) || !make_w_map(&w->tm_w2, w2, D, mlp) || !make_w_map(&w->tm_wh, wh, ncp, D))
    return false;
  w->ready = true;
  return true;
}

namespace {
__global__ void k_dec_pack(DecDenseWeights w, float* vec_b, float* vec_a2) {
  const int D = w.D, MLP = w.mlp;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < D) {
    vec_b[i] = w.bco[i]; vec_b[D + i] = w.n2_g[i]; vec_b[2 * D + i] = w.n2_b[i];
    vec_b[3 * D + MLP + i] = w.b2[i]; vec_b[4 * D + MLP + i] = w.nf_g[i]; vec_b[5 * D + MLP + i] = w.nf_b[i];
    for (int st = 0; st < w.L; ++st) {
      float* a = vec_a2 + static_cast<size_t>(st) * 4 * D;
      a[i] = w.bo[i] + w.posq[static_cast<size_t>(st) * D + i];
      a[D + i] = w.n1_g[i]; a[2 * D + i] = w.n1_b[i]; a[3 * D + i] = w.bq[i];
    }
  }
  if (i < MLP) vec_b[3 * D + i] = w.b1[i];
  if (i < 128) vec_b[6 * D + MLP + i] = i < w.ncp ? w.bh[i] : 0.f;
}
}  // namespace

cudaError_t dec_dense_pack(DecDenseWeights* w, cudaStream_t s) {
  if (!w->ready) return cudaSuccess;
  dec_dense_free(w);
  TT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&w->vec_b), sizeof(float) * (6 * w->D + w->mlp + 128)));
  TT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&w->vec_a2), sizeof(float) * w->L * 4 * w->D));
  const int n = std::max(w->mlp, std::max(w->D, 128));
  k_dec_pack<<<(n + 255) / 256, 256, 0, s>>>(*w, w->vec_b, w->vec_a2);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

void dec_dense_free(DecDenseWeights* w) {
  if (w->vec_b) cudaFree(w->vec_b);
  if (w->vec_a2) cudaFree(w->vec_a2);
  w->vec_b = w->vec_a2 = nullptr;
}

cudaError_t dec_dense_a2(const DecDenseWeights& w, const __nv_bfloat16* ab, int n, int step, float* t_scratch,
                         __nv_bfloat16* q_out, cudaStream_t s, const int* active, const int* n_act) {
  if (n <= 0) return cudaSuccess;
  if (!w.ready) { set_error("dec_dense_a2: weights not initialised for this width"); return cudaErrorInvalidValue; }
  DenseParams p{};
  if (!make_in_map(&p.tm_in, ab, n, w.D)) return cudaErrorInvalidValue;
  p.tm_w0 = w.tm_wo; p.tm_w1 = w.tm_wq; p.tm_w2 = w.tm_wq; p.tm_wh = w.tm_wq;
  p.vec_src = w.vec_a2 + static_cast<size_t>(step) * 4 * w.D;
  p.t_scratch = t_scratch; p.q_out = q_out;
  p.n = n; p.L = w.L; p.step = step; p.n_cls = w.n_cls; p.ncp = w.ncp;
  p.active = active; p.n_act = n_act;
  if (w.D == 384) return launch_dense<384, 1536, MODE_A2>(p, s);
  return launch_dense<192, 768, MODE_A2>(p, s);
}

cudaError_t dec_dense_b(const DecDenseWeights& w, const __nv_bfloat16* ab2, int n, int step, const float* t_scratch,
                        float* logits, int* tokens, const int* forced, cudaStream_t s, const int* active, const int* n_act,
                        const uint32_t* mask, const LexDev* lex, bool first_step) {
  if (n <= 0) return cudaSuccess;
  if (!w.ready) { set_error("dec_dense_b: weights not initialised for this width"); return cudaErrorInvalidValue; }
  DenseParams p{};
  if (!make_in_map(&p.tm_in, ab2, n, w.D)) return cudaErrorInvalidValue;
  p.tm_w0 = w.tm_wco; p.tm_w1 = w.tm_w1; p.tm_w2 = w.tm_w2; p.tm_wh = w.tm_wh;
  p.vec_src = w.vec_b;
  p.t_scratch = const_cast<float*>(t_scratch);
  p.logits = logits; p.tokens = tokens; p.forced = forced; p.mask = mask;
  p.n = n; p.L = w.L; p.step = step; p.n_cls = w.n_cls; p.ncp = w.ncp;
  p.active = active; p.n_act = n_act;
  if (lex) {
    p.st_in = first_step ? lex->root : lex->state;
    p.st_out = lex->state;
    p.lx_allow = lex->allow; p.lx_first = lex->first; p.lx_next = lex->next;
    if (w.D == 384) return launch_dense<384, 1536, MODE_B, MASK_STATE>(p, s);
    return launch_dense<192, 768, MODE_B, MASK_STATE>(p, s);
  }
  if (mask) {
    if (w.D == 384) return launch_dense<384, 1536, MODE_B, MASK_CROP>(p, s);
    return launch_dense<192, 768, MODE_B, MASK_CROP>(p, s);
  }
  if (w.D == 384) return launch_dense<384, 1536, MODE_B>(p, s);
  return launch_dense<192, 768, MODE_B>(p, s);
}

}  // namespace tt
