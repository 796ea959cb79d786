// Softmax of one 128-key encoder score row, shared by the encoder attention kernels (nn_kernels.cu k_attn_enc and
// enc_qkv_attn.cu k_enc_qkv_attn): both must produce the same P bits from the same scores.
#pragma once
#include <math.h>
#include <stdint.h>

#include "epi_math.cuh"
#include "ptx.cuh"

namespace tt {

// P as the A operand of O = P V: K-major SWIZZLE_128B, keys [64b, 64b+64) in the 16 KB atom block b at sP + b * 16384.
// Stores keys [16 ch, 16 ch + 16) of row r.
__device__ __forceinline__ void attn_store_p16(uint8_t* sP, int r, int ch, const float (&p)[16]) {
  uint8_t* blk = sP + (ch >> 2) * 16384 + r * 128;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int chunk = ((ch & 3) * 2 + h) ^ (r & 7);
    uint4 u;
    u.x = pack_bf16(p[8 * h + 0], p[8 * h + 1]); u.y = pack_bf16(p[8 * h + 2], p[8 * h + 3]);
    u.z = pack_bf16(p[8 * h + 4], p[8 * h + 5]); u.w = pack_bf16(p[8 * h + 6], p[8 * h + 7]);
    *reinterpret_cast<uint4*>(blk + chunk * 16) = u;
  }
}

// One-pass softmax: the thread's whole S row (128 fp32 at TMEM address t_row) is pulled out of TMEM once and kept in
// registers for the maximum and the exponentials; exp2((s - max) * scale) -> bf16 P row r in sP.  Returns the row's
// sum of the (fp32) exponentials.
__device__ __forceinline__ float attn_softmax_onepass(uint32_t t_row, uint8_t* sP, int r, float scale_log2e) {
  uint32_t raw[4][32];
#pragma unroll
  for (int b = 0; b < 4; ++b) ptx::tmem_ld<32>(t_row + b * 32, raw[b]);
#pragma unroll
  for (int b = 0; b < 4; ++b) ptx::tmem_ld_wait(raw[b]);
  float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
  for (int b = 0; b < 4; ++b)
#pragma unroll
    for (int i = 0; i < 32; ++i) m4[i & 3] = fmaxf(m4[i & 3], __uint_as_float(raw[b][i]));
  const float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
  const float nms = -mx * scale_log2e;
  float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int ch = 0; ch < 8; ++ch) {
    float p[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      // exp2((s - mx) * scale) as one FFMA + one MUFU (arguments <= 0: no range fix-up needed)
      const float a = fmaf(__uint_as_float(raw[ch >> 1][(ch & 1) * 16 + i]), scale_log2e, nms);
      asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(p[i]) : "f"(a));
      s4[i & 3] += p[i];
    }
    attn_store_p16(sP, r, ch, p);
  }
  return (s4[0] + s4[1]) + (s4[2] + s4[3]);
}

}  // namespace tt
