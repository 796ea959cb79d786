// Everything in the two networks that is not a GEMM: pooling / upsampling for CRAFT,
// LayerNorm, encoder attention (tcgen05) and the small decoder kernels for PARSeq.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tt {

// ---- CRAFT (NHWC bf16) -------------------------------------------------------------------
// conv1_1 + BN + ReLU from the u8 page [B][H][W][3] (already channel-swapped, raw 0..255): wt bf16 [64][32] with
// k = tap * 3 + c and the 1/255 folded in (weights.py "c1_1.w"), out bf16 NHWC [B][H][W][64]
cudaError_t conv1_1_u8(const uint8_t* img, int B, int H, int W, const __nv_bfloat16* wt, const float* bias, __nv_bfloat16* out,
                       cudaStream_t s);
// MaxPool2d(2, 2): [B][H][W][C] -> [B][H/2][W/2][C]           (vgg16_bn features 6/13/23/33)
cudaError_t maxpool2x2(const __nv_bfloat16* in, __nv_bfloat16* out, int B, int H, int W, int C, cudaStream_t s);
// MaxPool2d(3, stride 1, pad 1)                                 (slice5[0])
cudaError_t maxpool3x3s1(const __nv_bfloat16* in, __nv_bfloat16* out, int B, int H, int W, int C, cudaStream_t s);
// F.interpolate(scale 2, bilinear, align_corners=False): [B][H][W][C] -> [B][2H][2W][C]
cudaError_t upsample2x(const __nv_bfloat16* in, __nv_bfloat16* out, int B, int H, int W, int C, cudaStream_t s);

// A request's lexicon automata on the device (lexicon.h: state 0 is the done state) and the walk state of its crops.
struct LexDev {
  const uint4* allow = nullptr;   // [S] class mask of each state
  const int* first = nullptr;     // [S] index of the state's first successor in next
  const int* next = nullptr;      // [E] successor of the state's k-th allowed class at next[first + k]
  const int* root = nullptr;      // [n] root state of each crop
  int* state = nullptr;           // [n] each crop's current state in the AR loop
};

// ---- PARSeq ------------------------------------------------------------------------------
// LayerNorm over the last dim D (multiple of 32, <= 1024) of fp32 rows -> bf16 (and/or fp32) rows.
// rows_mod > 0: input row = row % rows_mod (broadcast table, e.g. pos_queries).
cudaError_t layernorm(const float* x, int rows, int D, const float* gamma, const float* beta, float eps,
                      __nv_bfloat16* out_bf16, float* out_f32, int rows_mod, cudaStream_t s);

// Encoder self-attention for T = 128 tokens, head dim 64: qkv bf16 [crops*128][3*D] (timm layout
// q|k|v, head-major inside each) -> out bf16 [crops*128][D].  One CTA per (head, crop); QK^T and PV
// on tcgen05 with S/O in TMEM, softmax in registers.  onepass: the S row is read from TMEM once (k_attn_enc<true>, the
// default); false selects the two-pass kernel.
cudaError_t attention_enc(const __nv_bfloat16* qkv, __nv_bfloat16* out, int crops, int D, int heads, bool onepass,
                          cudaStream_t s);

struct DecoderStep {
  int n_crops;
  int D, heads;     // 384, 12 (head dim 32)
  int L;            // 26 positions
  int p0, np;       // query positions [p0, p0+np) handled by this pass
  int refine;       // 0: AR causal mask (keys 0..p); 1: cloze mask + key padding after the first EOS
  // AR pass with per-crop early exit (nets.cpp): the step works on the first *n_act entries of `active` (slot -> crop).
  // Per-step activations (q, attention outputs) are indexed by slot; tokens, memory K|V and logits by crop.
  // Both null: every crop is active and slot == crop.
  const int* active = nullptr;
  const int* n_act = nullptr;
};
// content embedding of position `pos` (bos at 0, else pos_queries[pos-1] + sqrt(D)*E[tok]) -> LN_c -> bf16 [n][D]
cudaError_t dec_context(const int* tokens, const float* embed, const float* posq, const float* g, const float* b,
                        float eps, int pos, int n_crops, int D, int L, __nv_bfloat16* out, cudaStream_t s);
// self attention of the query stream over the content K/V.  With one decoder layer the content stream's K|V at
//   position j depend only on (j, token): kv_table bf16 [L][n_tok][2D] (K | V) is built once per engine
//   (DeviceCtx::init) and key j of a crop is row (j, tokens[crop][j]) -- no per-crop cache, no per-step K/V GEMM.
//   q_table fp32 [L][D] (already projected, crop independent), tokens int32 [n][L], out bf16 [n*np][D].
//   sc_table fp32 [L][L][n_tok][heads] (nullable): the AR pass's scores as a lookup, see dec_score_table.
cudaError_t dec_self_attn(const DecoderStep& st, const float* q_table, const float* sc_table, const __nv_bfloat16* kv_table,
                          const int* tokens, int eos_id, int n_tok, __nv_bfloat16* out, cudaStream_t s);
// sc_table[i][j][token][head] = q_table[i][head] . K(j, token)[head] / sqrt(32)   (built once per engine)
cudaError_t dec_score_table(const float* q_table, const __nv_bfloat16* kv_table, int L, int n_tok, int D, int heads,
                            float* out, cudaStream_t s);
// cross attention over the encoder memory: q bf16 [n*np][D], mem_kv bf16 [n][128][2D] -> out bf16 [n*np][D]
cudaError_t dec_cross_attn(const DecoderStep& st, const __nv_bfloat16* q, const __nv_bfloat16* mem_kv,
                           __nv_bfloat16* out, cudaStream_t s);
// argmax over the first n_cls of ld logits per row (first max wins) -> ids[row*ids_stride]; when
// `forced` != null the value written to next_tokens comes from forced instead of the argmax.
// mask (nullable, device [rows / rows_per_mask][4] uint32, 16-byte aligned): the class mask of each group of
// rows_per_mask consecutive rows (1: row = crop; L: row = crop * L + t); only classes whose bit is set compete.
// lex (nullable, rows = crops; mask is then unused): the allowed classes of crop c are the allow row of its state
// (lex->root[c] when first_step, else lex->state[c]); lex->state[c] becomes the chosen class's successor.  An all-NaN row
// takes the state's lowest allowed class.
cudaError_t argmax_rows(const float* logits, int rows, int n_cls, int ld, int* ids, int ids_stride,
                        int* next_tokens, int next_stride, const int* forced, int forced_stride, cudaStream_t s,
                        const uint32_t* mask = nullptr, int rows_per_mask = 1, const LexDev* lex = nullptr,
                        bool first_step = false);
// argmax_rows' ids (same tie and NaN rules, bit-identical) fused with the largest softmax probability of the row,
// pmax[row] = 1 / sum_c exp(logits[row][c] - max) in fp32 (deterministic; NaN for a row holding a NaN).  ids, pmax [rows].
// mask as in argmax_rows: the max and the sum run over the allowed classes only.
cudaError_t argmax_conf_rows(const float* logits, int rows, int n_cls, int ld, int* ids, float* pmax, cudaStream_t s,
                             const uint32_t* mask = nullptr, int rows_per_mask = 1);
// Refinement head of a lexicon request (INTEGRATION.md section 9): per crop, a walk over its L rows of logits [n][L][ld]
// from lex.root[crop]; each row's id is the argmax over its state's allowed classes (argmax_conf_rows' rules; an all-NaN
// row takes the lowest allowed class) and p the probability renormalised over them.  ids [n][L], pmax (nullable) [n][L].
cudaError_t lexicon_walk(const float* logits, int n, int L, int n_cls, int ld, const LexDev& lex, int* ids, float* pmax,
                         cudaStream_t s);
// u8 crops [n][32][128][3] -> bf16 patch rows [n*128][96] (raw 0..255), k = c*32 + (y%4)*8 + x%8
cudaError_t tokens_init(int* tokens, int n, int L, int bos, int pad, cudaStream_t s);
// AR early exit: the crops of (active_in, *n_in) -- null: all n crops -- whose token at position `pos` is not EOS, in the
// same order -> active_out, *n_out.  A crop that has produced EOS leaves the AR loop: upstream PARSeq stops a batch when
// every sequence has one, and nothing after a crop's first EOS reaches the refinement pass (its keys are masked from
// there on) or the decoded string.
cudaError_t dec_compact(const int* active_in, const int* n_in, int n, const int* tokens, int L, int pos, int eos_id,
                        int* active_out, int* n_out, cudaStream_t s);
// x fp32 [n] -> hi = bf16(x), lo = bf16(x - hi)  (split residual stream, gemm_tc.cuh RES_SPLIT)
cudaError_t split_f32(const float* x, long long n, __nv_bfloat16* hi, __nv_bfloat16* lo, cudaStream_t s);
cudaError_t patchify_u8(const uint8_t* crops, int n, __nv_bfloat16* out, cudaStream_t s);

}  // namespace tt
