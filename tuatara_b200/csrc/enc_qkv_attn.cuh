// First half of a PARSeq encoder block (timm Block: attn(LN1(x)) up to the output projection, reached by the reference
// through TorchScript at tuatara.cpp:307) in ONE kernel: the LayerNorm-folded qkv projection and the self attention,
// head by head, so the [rows][3D] qkv tensor never leaves the SM.  See enc_qkv_attn.cu for the layout.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace tt {

// PARSeq-base (D = 384, 6 heads) and PARSeq-tiny (D = 192, 3 heads): head dim 64, 128 tokens per crop.
bool enc_qkv_attn_supported(int D, int heads);

// att[crops*128][D] (bf16) = attention of q | k | v = LN(x) Wqkv^T + b, computed as the LayerNorm-consumer GEMM epilogue
// does (gemm_tc.cuh, Epilogue::ln_*): hi = bf16(x) [crops*128][D]; stats: per row `parts` (1..4) partial
// (sum x, sum x^2) float2 over D columns in total; wf = Wqkv * gamma (bf16 [3D][D]); c0 = b + Wqkv beta, c1 = row sums of
// wf (fp32 [3D]).  Bit for bit the output of that GEMM (qkv, bf16) followed by attention_enc(onepass).
cudaError_t enc_qkv_attn_forward(const __nv_bfloat16* hi, const float* stats, int parts, const __nv_bfloat16* wf,
                                 const float* c0, const float* c1, __nv_bfloat16* att, int crops, int D, int heads, float eps,
                                 cudaStream_t s);

}  // namespace tt
