// First half of a PARSeq encoder block in ONE tcgen05 kernel (see enc_qkv_attn.cuh):
//     qkv = LN1(x) Wqkv^T + b      (LayerNorm applied to the accumulators, as gemm_tc.cu's consumer epilogue does)
//     att = softmax(q k^T / 8) v   per head
//
// Why: as two launches (the qkv GEMM, then k_attn_enc) the [rows][3D] bf16 qkv tensor is written to HBM and read back once
// per block: 0.71 GB each way per layer at 2400 crops, and k_attn_enc does too little arithmetic per byte to be anything
// but an HBM kernel.  Here a CTA owns a crop at a time (M = 128 tokens = the 128 TMEM lanes) and produces qkv head by head
// straight into the shared-memory tiles the attention MMAs read.
//
// Persistent, one CTA per SM walking crops blockIdx.x, + gridDim.x, ...; 192 threads:
//   warp 0      TMA producer : the crop's hi rows -> sX (D/64 k-blocks of [128 rows][64], resident for all heads; the next
//                              crop's are loaded as soon as the last projection has read them, under the last heads'
//                              attention); per head and k-block the head's 192 weight rows (its q, k and v rows of the
//                              folded Wqkv) through a ring of three 24 KB slots
//   warp 1      MMA issuer   : acc[h & 1] = hi W_h^T (N = 192, K = D, the GEMM's k order), S = Q K^T, O = P V.  It polls
//                              its barriers and issues whatever is ready, attention first: the projection of head h + 1
//                              (k-block by k-block) runs on the tensor pipe while the row owners work on head h, across
//                              crop boundaries too
//   warps 2..5  row owners   : thread = row.  Per head: acc -> rstd * acc - rstd * mean * c1 + c0 -> bf16 Q | K | V
//                              (K-major SWIZZLE_128B, the layout k_attn_enc's TMA loads give it); the one-pass softmax of
//                              k_attn_enc (attn_softmax.cuh) -> P over Q | K; O / l -> bf16 over Q -> a TMA store of the
//                              warp's 32 rows at column 64 h of att
// TMEM (512 columns): [0, 192) and [192, 384) = the two projection accumulators, [384, 512) = S, then O in its first 64.
// The k-steps, the epilogue arithmetic and the softmax are the ones of the two-launch path, so att is bit for bit the same.
// Every wait is bounded (ptx::mbar_wait traps after 4 s).
#include "enc_qkv_attn.cuh"

#include <algorithm>
#include <cstdio>

#include "attn_softmax.cuh"
#include "common.h"
#include "epi_math.cuh"
#include "gemm_tc.cuh"
#include "ptx.cuh"

namespace tt {

namespace {

constexpr int kUnit = 16384;            // [128 rows][64 bf16], SWIZZLE_128B
constexpr int kWBox = 8192;             // [64 weight rows][64 k]
constexpr int kSlot = 3 * kWBox;        // one k-block of a head's q | k | v weight rows
constexpr int kStages = 3;
constexpr int kRowThreads = 128;
constexpr int kThreads = 64 + kRowThreads;
constexpr int kAccCols = 192;
constexpr int kSCol = 2 * kAccCols;     // S, then O
constexpr int kTmemCols = 512;

struct Ctl {
  uint64_t x_full[6], x_empty;          // x_empty: the crop's last projection has read sX
  uint64_t full[kStages], empty[kStages];
  uint64_t acc_full[2];
  uint64_t qkv_ready, p_ready;          // row owners -> MMA issuer (128 arrivals each)
  uint64_t s_full, o_full;
  uint32_t tmem_base;
};

template <int D>
constexpr int smem_bytes() { return 1024 + (D / 64) * kUnit + kStages * kSlot + 3 * kUnit + static_cast<int>(sizeof(Ctl)); }

// wait-free probe of a barrier, warp-uniform (lane 0's view)
__device__ __forceinline__ bool poll(uint64_t* bar, uint32_t parity) {
  return __shfl_sync(0xffffffffu, ptx::mbar_test_wait(bar, parity) ? 1 : 0, 0) != 0;
}

template <int D>
__global__ void __launch_bounds__(kThreads, 1) k_enc_qkv_attn(const __grid_constant__ CUtensorMap tm_hi,
                                                              const __grid_constant__ CUtensorMap tm_w,
                                                              const __grid_constant__ CUtensorMap tm_att,
                                                              const float2* __restrict__ stats, int parts,
                                                              const float* __restrict__ c0, const float* __restrict__ c1,
                                                              int crops, float eps, float scale_log2e) {
  constexpr int KB = D / 64, H = D / 64;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sX = smem;
  uint8_t* ring = sX + KB * kUnit;
  uint8_t* sQ = ring + kStages * kSlot;   // P spans Q | K once S has been read
  uint8_t* sK = sQ + kUnit;
  uint8_t* sV = sK + kUnit;
  Ctl* ctl = reinterpret_cast<Ctl*>(sV + kUnit);
  const int n_crops = (crops - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int n_heads = n_crops * H;   // this CTA's (crop, head) sequence; g = crop iteration * H + head
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    ptx::prefetch_tmap(&tm_hi);
    ptx::prefetch_tmap(&tm_w);
    ptx::prefetch_tmap(&tm_att);
    for (int i = 0; i < KB; ++i) ptx::mbar_init(&ctl->x_full[i], 1);
    ptx::mbar_init(&ctl->x_empty, 1);
    for (int i = 0; i < kStages; ++i) { ptx::mbar_init(&ctl->full[i], 1); ptx::mbar_init(&ctl->empty[i], 1); }
    for (int i = 0; i < 2; ++i) ptx::mbar_init(&ctl->acc_full[i], 1);
    ptx::mbar_init(&ctl->qkv_ready, kRowThreads);
    ptx::mbar_init(&ctl->p_ready, kRowThreads);
    ptx::mbar_init(&ctl->s_full, 1);
    ptx::mbar_init(&ctl->o_full, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 1) ptx::tmem_alloc(&ctl->tmem_base, kTmemCols);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, ctl->tmem_base, 0);

  if (warp == 0) {
    // ------------------------------------------------------------- TMA producer (converged, one elected lane issues)
    int stage = 0;
    uint32_t phase = 0;
    for (int it = 0; it < n_crops; ++it) {
      const int crop = blockIdx.x + it * gridDim.x;
      if (it > 0) { ptx::mbar_wait(&ctl->x_empty, (it - 1) & 1); __syncwarp(); }
      for (int kb = 0; kb < KB; ++kb) {
        ptx::mbar_arrive_expect_tx_e(&ctl->x_full[kb], kUnit);
        ptx::tma_load_2d_e(sX + kb * kUnit, &tm_hi, &ctl->x_full[kb], kb * 64, crop * 128);
      }
      for (int h = 0; h < H; ++h)
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(&ctl->empty[stage], phase ^ 1); __syncwarp();
          uint8_t* slot = ring + stage * kSlot;
          ptx::mbar_arrive_expect_tx_e(&ctl->full[stage], kSlot);
#pragma unroll
          for (int part = 0; part < 3; ++part)   // the head's q, k, v rows of Wqkv: rows part * D + 64 h ..
            ptx::tma_load_2d_e(slot + part * kWBox, &tm_w, &ctl->full[stage], kb * 64, part * D + h * 64);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
    }
  } else if (warp == 1) {
    // --------------------------------------------------------------- MMA issuer (converged, one elected lane issues)
    const uint32_t idesc_p = ptx::make_idesc_bf16(128, kAccCols);
    const uint32_t idesc_s = ptx::make_idesc_bf16(128, 128);
    const uint32_t idesc_o = ptx::make_idesc_bf16(128, 64) | (1u << 16);   // B = V, MN-major
    const uint32_t xa = ptx::smem_u32(sX), qa = ptx::smem_u32(sQ), ka = ptx::smem_u32(sK), va = ptx::smem_u32(sV);
    int ph = 0, pk = 0;   // next projection: g, k-block
    int ns = 0, np = 0;   // next S, next P V (g)
    int stage = 0;
    uint32_t phase = 0;
    uint64_t t_last = ptx::globaltimer_ns();
#pragma unroll 1
    while (np < n_heads) {
      if (np < ns && poll(&ctl->p_ready, np & 1)) {
        ptx::tc_fence_after();
        // O[128 q][64 d] = P V, as k_attn_enc: A = P (K-major over keys), B = V (MN-major, one 1024-byte atom per 8 keys)
#pragma unroll
        for (int k = 0; k < 8; ++k)
          ptx::mma_bf16_e(tmem + kSCol, ptx::make_smem_desc(qa + (k >> 2) * kUnit + (k & 3) * 32, 128),
                          ptx::make_smem_desc(va + k * 2048, 128), idesc_o, k != 0);
        ptx::mma_commit_e(&ctl->o_full);
        ++np;
        t_last = ptx::globaltimer_ns();
        continue;
      }
      // qkv_ready(h) also says O(h - 1) has been read out of the S / O columns
      if (ns < n_heads && ns == np && poll(&ctl->qkv_ready, ns & 1)) {
        ptx::tc_fence_after();
#pragma unroll
        for (int k = 0; k < 4; ++k)
          ptx::mma_bf16_e(tmem + kSCol, ptx::make_smem_desc(qa + k * 32, 128), ptx::make_smem_desc(ka + k * 32, 128), idesc_s, k != 0);
        ptx::mma_commit_e(&ctl->s_full);
        ++ns;
        t_last = ptx::globaltimer_ns();
        continue;
      }
      // acc[ph & 1] was last drained by g = ph - 2: its qkv_ready was seen when S(ph - 2) was issued; a crop's first head
      // waits for its rows
      if (ph < n_heads && ns >= ph - 1 && (ph % H != 0 || poll(&ctl->x_full[pk], (ph / H) & 1)) && poll(&ctl->full[stage], phase)) {
        ptx::tc_fence_after();
        const uint32_t wa = ptx::smem_u32(ring + stage * kSlot);
        const uint32_t d = tmem + (ph & 1) * kAccCols;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          ptx::mma_bf16_e(d, ptx::make_smem_desc(xa + pk * kUnit + k * 32, 128), ptx::make_smem_desc(wa + k * 32, 128), idesc_p,
                          (pk | k) != 0);
        ptx::mma_commit_e(&ctl->empty[stage]);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
        if (++pk == KB) {
          ptx::mma_commit_e(&ctl->acc_full[ph & 1]);
          if (ph % H == H - 1) ptx::mma_commit_e(&ctl->x_empty);   // sX may take the next crop's rows
          pk = 0;
          ++ph;
        }
        t_last = ptx::globaltimer_ns();
        continue;
      }
      if (ptx::globaltimer_ns() - t_last > 4000000000ull) __trap();
    }
  } else {
    // ----------------------------------------------------------------- row owners
    const int q = warp & 3;                  // TMEM lane quadrant this warp may read
    const int r = q * 32 + lane;             // token == TMEM lane
    const uint32_t t_lane = tmem + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t q_row = ptx::smem_u32(sQ) + r * 128;
    const int sw = r & 7;
#pragma unroll 1
    for (int it = 0; it < n_crops; ++it) {
      const int crop = blockIdx.x + it * gridDim.x;
      // LayerNorm statistics of the row: exactly the consumer epilogue of gemm_tc.cu (same partial order, same formula)
      uint64_t ln_a, ln_b;
      {
        constexpr int kLnMaxParts = 4;
        const float2* st = stats + (static_cast<long long>(crop) * 128 + r) * parts;
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int pp = 0; pp < kLnMaxParts; ++pp) {
          const float2 v = pp < parts ? __ldg(st + pp) : make_float2(0.f, 0.f);
          s1 += v.x; s2 += v.y;
        }
        const float inv_d = 1.f / static_cast<float>(D);
        const float mu = s1 * inv_d;
        const float rstd = rsqrtf(fmaxf(s2 * inv_d - mu * mu, 0.f) + eps);
        ln_a = pk2(rstd, rstd);
        ln_b = pk2(-rstd * mu, -rstd * mu);
      }
#pragma unroll 1
      for (int h = 0; h < H; ++h) {
        const int g = it * H + h;
        ptx::mbar_wait(&ctl->acc_full[g & 1], (g >> 1) & 1);
        ptx::tc_fence_after();
        if (g > 0) {   // the TMA store of the previous O has finished reading this warp's rows of sQ
          if (ptx::elect_one()) ptx::bulk_wait_read<0>();
          __syncwarp();
        }
        const uint32_t t_acc = t_lane + (g & 1) * kAccCols;
#pragma unroll 1
        for (int part = 0; part < 3; ++part) {   // q | k | v of head h -> its [128][64] tile
          uint32_t raw[2][32];
          ptx::tmem_ld<32>(t_acc + part * 64, raw[0]);
          ptx::tmem_ld<32>(t_acc + part * 64 + 32, raw[1]);
          ptx::tmem_ld_wait(raw[0]);
          ptx::tmem_ld_wait(raw[1]);
          const int col0 = part * D + h * 64;
          const uint32_t dst = q_row + part * kUnit;
#pragma unroll
          for (int u = 0; u < 8; ++u) {   // 16-byte unit u = columns [8u, 8u + 8)
            const float4 b0 = __ldg(reinterpret_cast<const float4*>(c0 + col0 + 8 * u));
            const float4 b1 = __ldg(reinterpret_cast<const float4*>(c0 + col0 + 8 * u + 4));
            const float4 e0 = __ldg(reinterpret_cast<const float4*>(c1 + col0 + 8 * u));
            const float4 e1 = __ldg(reinterpret_cast<const float4*>(c1 + col0 + 8 * u + 4));
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
            const float ee[8] = {e0.x, e0.y, e0.z, e0.w, e1.x, e1.y, e1.z, e1.w};
            uint32_t o[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {   // rstd * acc - rstd * mean * c1 + c0
              const uint32_t* a = &raw[u >> 2][(u & 3) * 8 + 2 * e];
              const uint64_t v = fma2(pk2u(a[0], a[1]), ln_a, fma2(ln_b, pk2(ee[2 * e], ee[2 * e + 1]), pk2(bb[2 * e], bb[2 * e + 1])));
              float v0, v1;
              upk2(v, v0, v1);
              o[e] = pack_bf16(v0, v1);
            }
            ptx::sts128(dst + ((u ^ sw) << 4), make_uint4(o[0], o[1], o[2], o[3]));
          }
        }
        ptx::fence_proxy_async();
        ptx::tc_fence_before();
        ptx::mbar_arrive(&ctl->qkv_ready);

        ptx::mbar_wait(&ctl->s_full, g & 1);
        ptx::tc_fence_after();
        const float sum = attn_softmax_onepass(t_lane + kSCol, sQ, r, scale_log2e);
        ptx::fence_proxy_async();
        ptx::tc_fence_before();
        ptx::mbar_arrive(&ctl->p_ready);

        ptx::mbar_wait(&ctl->o_full, g & 1);
        ptx::tc_fence_after();
        {
          const float inv = 1.f / sum;
          uint32_t raw[2][32];
          ptx::tmem_ld<32>(t_lane + kSCol, raw[0]);
          ptx::tmem_ld<32>(t_lane + kSCol + 32, raw[1]);
          ptx::tmem_ld_wait(raw[0]);
          ptx::tmem_ld_wait(raw[1]);
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            uint32_t o[4];
#pragma unroll
            for (int e = 0; e < 4; ++e)
              o[e] = pack_bf16(__uint_as_float(raw[u >> 2][(u & 3) * 8 + 2 * e]) * inv,
                               __uint_as_float(raw[u >> 2][(u & 3) * 8 + 2 * e + 1]) * inv);
            ptx::sts128(q_row + ((u ^ sw) << 4), make_uint4(o[0], o[1], o[2], o[3]));
          }
        }
        ptx::fence_proxy_async();
        __syncwarp();
        ptx::tma_store_2d_e(&tm_att, sQ + q * 32 * 128, h * 64, crop * 128 + q * 32);
        ptx::bulk_commit_e();
      }
    }
    if (ptx::elect_one()) ptx::bulk_wait<0>();
    __syncwarp();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem, kTmemCols);
  }
}

bool make_map(CUtensorMap* m, const void* base, long long rows, int cols, int box_rows) {
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(cols) * 2};
  const cuuint32_t box[2] = {64, static_cast<cuuint32_t>(box_rows)};
  return make_tmap_bf16(m, base, 2, dims, strides, box, 128);
}

template <int D>
cudaError_t launch(const CUtensorMap& tm_hi, const CUtensorMap& tm_w, const CUtensorMap& tm_att, const float* stats, int parts,
                   const float* c0, const float* c1, int crops, float eps, float scale_log2e, cudaStream_t s) {
  constexpr int kSmem = smem_bytes<D>();
  static_assert(kSmem <= 227 * 1024, "shared memory budget");
  TT_CUDA_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(k_enc_qkv_attn<D>), kSmem));
  static const int sms = [] {
    int dev = 0, n = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    return n;
  }();
  k_enc_qkv_attn<D><<<std::min(crops, sms), kThreads, kSmem, s>>>(tm_hi, tm_w, tm_att, reinterpret_cast<const float2*>(stats), parts,
                                                                 c0, c1, crops, eps, scale_log2e);
  return cudaSuccess;
}

}  // namespace

bool enc_qkv_attn_supported(int D, int heads) { return (D == 384 || D == 192) && heads * 64 == D; }

cudaError_t enc_qkv_attn_forward(const __nv_bfloat16* hi, const float* stats, int parts, const __nv_bfloat16* wf,
                                 const float* c0, const float* c1, __nv_bfloat16* att, int crops, int D, int heads, float eps,
                                 cudaStream_t s) {
  if (crops <= 0) return cudaSuccess;
  if (!enc_qkv_attn_supported(D, heads) || parts < 1 || parts > 4) {
    set_error("enc_qkv_attn: built for head dim 64 with D = 384 or 192 and 1..4 LayerNorm partials per row");
    return cudaErrorInvalidValue;
  }
  if ((reinterpret_cast<uintptr_t>(c0) | reinterpret_cast<uintptr_t>(c1)) & 15) {
    set_error("enc_qkv_attn: per-column vectors must be 16-byte aligned");
    return cudaErrorInvalidValue;
  }
  const long long M = static_cast<long long>(crops) * 128;
  CUtensorMap tm_hi, tm_w, tm_att;
  if (!make_map(&tm_hi, hi, M, D, 128) || !make_map(&tm_w, wf, 3LL * D, D, 64) || !make_map(&tm_att, att, M, D, 32))
    return cudaErrorInvalidValue;
  const float scale_log2e = 0.125f * 1.4426950408889634f;  // head_dim^-0.5 * log2(e), as attention_enc
  char tag[64];
  if (prof_enabled()) {
    std::snprintf(tag, sizeof(tag), "qkv+attn M%lld D%d", M, D);
    prof_record(s, true, 0, 0);
  }
  if (D == 384) TT_CUDA_TRY(launch<384>(tm_hi, tm_w, tm_att, stats, parts, c0, c1, crops, eps, scale_log2e, s));
  else TT_CUDA_TRY(launch<192>(tm_hi, tm_w, tm_att, stats, parts, c0, c1, crops, eps, scale_log2e, s));
  // the qkv projection's FLOPs (the attention's own are not counted, as for k_attn_enc), so tensor-core totals stay comparable
  prof_record(s, false, 2.0 * static_cast<double>(M) * D * 3 * D, 0, tag);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

}  // namespace tt
