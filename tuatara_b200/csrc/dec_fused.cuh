// Fused dense kernels of the PARSeq decoder's autoregressive loop (dec_fused.cu).
//
// One AR step of the query stream (upstream PARSeq DecoderLayer.forward_stream, SURVEY App. B; the reference reaches it
// through the TorchScript forward at tuatara.cpp:307) is, per crop, a chain of row-local operations around the two
// attentions:
//     ab  = SelfAttn(q_i, K/V of the content tokens)                              nn_kernels.cu (K/V from the lookup table)
//     t   = pos_queries[i] + out_proj(ab);  qc = q_proj(LN1(t))                   dec_dense_a2   (this file)
//     ab2 = CrossAttn(qc, memory K|V)                                             nn_kernels.cu (HBM-bound stream)
//     t  += ca_out(ab2);  t += W2 GELU(W1 LN2(t));  logits = head(LN(t)); argmax  dec_dense_b    (this file)
// The unfused path ran these as 11 launches whose GEMMs have M = crops (75 tiles for a 32-page group: two waves of
// latency-bound tiles at 17-190 TFLOP/s).  Here a CTA owns 128 crops for the whole chain: the fp32 row `t` lives in
// TMEM (tcgen05.mma accumulates the residual updates onto it in place), LayerNorm runs in registers (thread = row =
// TMEM lane, no shuffles), the normalised / GELU'd rows are written straight into swizzled smem as the next MMA's A
// operand, and the weights stream through a TMA ring in a static order.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "nn_kernels.cuh"

namespace tt {

struct DecDenseWeights {
  CUtensorMap tm_wo, tm_wq, tm_wco, tm_w1, tm_w2, tm_wh;   // bf16 [N][K] weights, box {64 k, min(128, N) rows}
  const float *bo = nullptr, *bq = nullptr, *bco = nullptr, *b1 = nullptr, *b2 = nullptr, *bh = nullptr;
  const float *n1_g = nullptr, *n1_b = nullptr, *n2_g = nullptr, *n2_b = nullptr, *nf_g = nullptr, *nf_b = nullptr;
  const float* posq = nullptr;   // [L][D]
  // the kernels' per-column vectors packed in smem order (device memory owned by this struct's user, see dec_dense_pack):
  //   vec_b  [6 D + mlp + 128]: bco | n2_g | n2_b | b1 | b2 | nf_g | nf_b | bh (zero padded to 128)
  //   vec_a2 [L][4 D]         : bo + posq[step] | n1_g | n1_b | bq
  float* vec_b = nullptr;
  float* vec_a2 = nullptr;
  int D = 0, mlp = 0, n_cls = 0, ncp = 0, L = 0;
  bool ready = false;
};

// Encodes the weight tensor maps (once per device).  wq = rows [0, D) of cross_attn.in_proj.
bool dec_dense_init(DecDenseWeights* w, int D, int mlp, int n_cls, int ncp, int L, const __nv_bfloat16* wo,
                    const __nv_bfloat16* wq, const __nv_bfloat16* wco, const __nv_bfloat16* w1, const __nv_bfloat16* w2,
                    const __nv_bfloat16* wh);
bool dec_dense_supported(int D, int mlp, int ncp);
// After the bias / LayerNorm / posq pointers are set: allocates and fills vec_b / vec_a2 on the current device
// (dec_dense_free releases them).
cudaError_t dec_dense_pack(DecDenseWeights* w, cudaStream_t s);
void dec_dense_free(DecDenseWeights* w);

// fp32 scratch the two kernels hand the residual row through: [ceil(n/128)][D][128] (column-major per 128-crop tile).
size_t dec_dense_scratch_floats(int n, int D);

// ab [n][D] bf16 (self-attention output of step `step`) -> t_scratch (t = posq[step] + out_proj(ab)), q_out [n][D] bf16
// (active, n_act): the early-exit AR pass's slot -> crop list and its device-side length (nn_kernels.cuh DecoderStep); the
// rows of ab / q_out / t_scratch are slots, logits and tokens are indexed by crop.  Null: n rows, slot == crop.
cudaError_t dec_dense_a2(const DecDenseWeights& w, const __nv_bfloat16* ab, int n, int step, float* t_scratch,
                         __nv_bfloat16* q_out, cudaStream_t s, const int* active = nullptr, const int* n_act = nullptr);
// ab2 [n][D] bf16 (cross-attention output of step `step`), t_scratch -> logits [n][L][ncp] row `step` (fp32) and the next
// token: tokens[crop][step + 1] = forced ? forced[crop][step] : argmax over the first n_cls logits (first max wins).
// mask (nullable): class masks [n][4] uint32 (16-byte aligned, indexed by crop like tokens): the argmax runs over the
// classes whose bit (c & 31 of word c >> 5) is set; the logits are written unmasked.
// lex (nullable; mask is then unused): the mask of crop c is the allow row of its state (lex->root[c] at first_step,
// else lex->state[c], indexed by crop like tokens); an all-NaN row takes the lowest allowed class and lex->state[c]
// becomes the chosen class's successor.
cudaError_t dec_dense_b(const DecDenseWeights& w, const __nv_bfloat16* ab2, int n, int step, const float* t_scratch,
                        float* logits, int* tokens, const int* forced, cudaStream_t s, const int* active = nullptr,
                        const int* n_act = nullptr, const uint32_t* mask = nullptr, const LexDev* lex = nullptr,
                        bool first_step = false);

}  // namespace tt
