// CRAFT and PARSeq forward passes assembled from the tcgen05 GEMM kernel (gemm_tc.cu) and the
// auxiliary kernels (nn_kernels.cu).  These replace `detector_model.forward` (tuatara.cpp:376) and
// `model.forward` inside infer() (tuatara.cpp:307); the graphs are the upstream architectures the
// reference's TorchScript files encode (SURVEY.md App. A / B; oracle/models.py is the fp32 oracle).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <stdexcept>
#include <vector>

#include "common.h"
#include "dec_fused.cuh"
#include "enc_mlp.cuh"
#include "enc_qkv_attn.cuh"
#include "engine.h"
#include "gemm_tc.cuh"
#include "nn_kernels.cuh"
#include "resize.cuh"

namespace tt {

// ------------------------------------------------------------------------------ WeightFile
WeightFile::~WeightFile() {
  if (arena_) cudaFree(arena_);
}

bool WeightFile::load(const std::string& path, std::vector<int>* meta_out) {
  std::ifstream f(path, std::ios::binary | std::ios::ate);
  if (!f) { set_error("cannot open weight file " + path); return false; }
  const size_t size = static_cast<size_t>(f.tellg());
  f.seekg(0);
  std::vector<char> buf(size);
  f.read(buf.data(), static_cast<std::streamsize>(size));
  if (size < 8 || std::memcmp(buf.data(), "TTW1", 4) != 0) { set_error("bad weight file " + path); return false; }
  uint32_t n;
  std::memcpy(&n, buf.data() + 4, 4);
  // the directory must lie inside the file before anything in it is trusted
  if (static_cast<uint64_t>(n) > (size - 8) / 120) { set_error("bad weight file " + path + " (directory larger than the file)"); return false; }
  if (cudaMalloc(&arena_, size) != cudaSuccess) { set_error("cudaMalloc failed for " + path); return false; }
  if (cudaMemcpy(arena_, buf.data(), size, cudaMemcpyHostToDevice) != cudaSuccess) {
    set_error("weight upload failed for " + path);
    return false;
  }
  for (uint32_t i = 0; i < n; ++i) {
    const char* e = buf.data() + 8 + static_cast<size_t>(i) * 120;
    char name[65] = {0};
    std::memcpy(name, e, 64);
    uint32_t dt, nd;
    uint64_t dims[4], off, nb;
    std::memcpy(&dt, e + 64, 4);
    std::memcpy(&nd, e + 68, 4);
    std::memcpy(dims, e + 72, 32);
    std::memcpy(&off, e + 104, 8);
    std::memcpy(&nb, e + 112, 8);
    if (off > size || nb > size - off) { set_error("truncated weight file " + path); return false; }   // no uint64 wrap
    if (dt > 2 || nd > 4 || off % 16 != 0) { set_error("bad weight file " + path + " (tensor '" + name + "')"); return false; }
    if (meta_out && std::strcmp(name, "meta") == 0) {
      if (nb % 4 != 0) { set_error("bad weight file " + path + " (meta tensor)"); return false; }
      meta_out->resize(nb / 4);
      std::memcpy(meta_out->data(), buf.data() + off, nb);
    }
    WTensor t;
    t.ptr = static_cast<char*>(arena_) + off;
    t.dtype = static_cast<int>(dt);
    t.nbytes = nb;
    for (uint32_t k = 0; k < nd; ++k) t.dims.push_back(static_cast<long long>(dims[k]));
    t_[name] = t;
  }
  return true;
}

const WTensor& WeightFile::get(const std::string& name) const {
  auto it = t_.find(name);
  if (it == t_.end()) throw std::runtime_error("weight tensor '" + name + "' missing");
  return it->second;
}

// ----------------------------------------------------------------------------------- Arena
Arena::~Arena() {
  if (base_) cudaFree(base_);
}
cudaError_t Arena::reserve(size_t bytes) {
  off_ = 0;
  if (bytes <= cap_) return cudaSuccess;
  if (base_) { cudaFree(base_); base_ = nullptr; cap_ = 0; }
  bytes = (bytes + (size_t(1) << 26)) & ~((size_t(1) << 20) - 1);  // +64 MiB slack, MiB granularity
  TT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&base_), bytes));
  cap_ = bytes;
  return cudaSuccess;
}
void* Arena::alloc(size_t bytes) {
  const size_t a = (off_ + 1023) & ~size_t(1023);
  if (a + bytes > cap_) return nullptr;
  off_ = a + bytes;
  return base_ + a;
}

#define ARENA_GET(var, T, n)                                                       \
  T* var = arena.get<T>(static_cast<size_t>(n));                                   \
  if (!var) { set_error("arena exhausted (" #var ")"); return cudaErrorMemoryAllocation; }

// ----------------------------------------------------------------------------------- CRAFT
size_t DeviceCtx::craft_bytes(int B, int H, int W) const {
  // bf16 elements per input pixel over every activation kept (no buffer reuse), see craft_forward
  const double per_px = 32 + 64 + 64 + 64 / 4.0 + 128 / 4.0 + 128 / 4.0 + 128 / 16.0 + 3 * 256 / 16.0 + 256 / 64.0 +
                        3 * 512 / 64.0 + 512 / 256.0 + 3 * 512 / 256.0 + 2 * 1024 / 256.0 + (512 + 256) / 256.0 +
                        256 / 64.0 + (256 + 128) / 64.0 + 128 / 16.0 + (128 + 64) / 16.0 + 64 / 4.0 +
                        (64 + 32) / 4.0 + 2 * 32 / 4.0;
  const size_t px = static_cast<size_t>(B) * H * W;
  return static_cast<size_t>(per_px * 2.0 * px) + px * 2 /*fp32 maps: 2 ch * 4 B / 4*/ + (64u << 10) * 64;
}

cudaError_t DeviceCtx::craft_forward(const uint8_t* in, int B, int H, int W, float** maps_out) {
  using bf = __nv_bfloat16;
  if (H % 32 || W % 32) { set_error("craft_forward: input must be padded to a multiple of 32"); return cudaErrorInvalidValue; }
  const size_t px = static_cast<size_t>(B) * H * W;
  const int H2 = H / 2, W2 = W / 2, H4 = H / 4, W4 = W / 4, H8 = H / 8, W8 = W / 8, H16 = H / 16, W16 = W / 16;
  cudaStream_t s = stream;

  // pooled != nullptr: the 2x2 max-pool that follows the conv runs in its epilogue (out == nullptr: only the pooled
  // tensor is written).  TT_CRAFT_POOLFUSE=0 keeps the separate pooling kernel (A/B runs).
  const char* pool_env = std::getenv("TT_CRAFT_POOLFUSE");   // read per call: the parity test flips it in-process
  const bool pool_fuse = !(pool_env && std::atoi(pool_env) == 0);
  auto conv = [&](const char* name, const bf* a, int Ca, const bf* b, int Cb, int hh, int ww, int taps, int dil, int cout,
                  bool relu, bf* out, bf* pooled = nullptr) -> cudaError_t {
    ConvProblem c;
    c.batch = B; c.H = hh; c.W = ww;
    c.src[0] = ConvSrc{a, Ca, Ca};
    c.nsrc = 1;
    if (b) { c.src[1] = ConvSrc{b, Cb, Cb}; c.nsrc = 2; }
    c.taps = taps; c.dil = dil; c.Cout = cout;
    if (Ca == 32 && taps == 1 && cout == 64) c.algo_k = 27;  // conv1_1: 3x3x3 taps stored padded to 32
    c.weight = w->craft.bf(std::string(name) + ".w");
    Epilogue e;
    e.bias = w->craft.f32(std::string(name) + ".b");
    e.act = relu ? ACT_RELU : ACT_NONE;
    e.out = out; e.out_type = OUT_BF16; e.ldc = cout;
    if (pooled) { e.pool_out = pooled; e.pool_mode = out ? 2 : 1; }
    return conv_forward(c, e, s);
  };
  // conv + ReLU followed by MaxPool2d(2, 2); `full` (nullable) also keeps the un-pooled tensor
  auto conv_pool = [&](const char* name, const bf* a, int Ca, int hh, int ww, int cout, bf* full, bf* pooled) -> cudaError_t {
    if (pool_fuse) return conv(name, a, Ca, nullptr, 0, hh, ww, 9, 1, cout, true, full, pooled);
    bf* tmp = full;
    if (!tmp) {
      tmp = arena.get<bf>(static_cast<size_t>(B) * hh * ww * cout);
      if (!tmp) { set_error("arena exhausted (conv_pool)"); return cudaErrorMemoryAllocation; }
    }
    if (cudaError_t e1 = conv(name, a, Ca, nullptr, 0, hh, ww, 9, 1, cout, true, tmp)) return e1;
    return maxpool2x2(tmp, pooled, B, hh, ww, cout, s);
  };
#define CV(...) do { cudaError_t _e = conv(__VA_ARGS__); if (_e != cudaSuccess) return _e; } while (0)
#define RUN(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) return _e; } while (0)

  ARENA_GET(a1, bf, px * 64);
  const char* c11_env = std::getenv("TT_CRAFT_C11");   // 0: the round-1 path (im2col tensor + K=32 tcgen05 GEMM), A/B runs
  if (c11_env && std::atoi(c11_env) == 0) {
    ARENA_GET(x0, bf, px * 32);
    RUN(page_im2col(in, B, H, W, x0, s));
    CV("c1_1", x0, 32, nullptr, 0, H, W, 1, 1, 64, true, a1);  // 3x3 conv as a K=32 GEMM over the im2col'd pixels
  } else {
    RUN(conv1_1_u8(in, B, H, W, w->craft.bf("c1_1.w"), w->craft.f32("c1_1.b"), a1, s));   // straight from the u8 page
  }
  ARENA_GET(p1, bf, px / 4 * 64);
  RUN(conv_pool("c1_2", a1, 64, H, W, 64, nullptr, p1));
  ARENA_GET(b1, bf, px / 4 * 128);
  CV("c2_1", p1, 64, nullptr, 0, H2, W2, 9, 1, 128, true, b1);
  ARENA_GET(s1, bf, px / 4 * 128);  // relu2_2 (ReLU'd through upstream's in-place aliasing)
  ARENA_GET(p2, bf, px / 16 * 128);
  RUN(conv_pool("c2_2", b1, 128, H2, W2, 128, s1, p2));
  ARENA_GET(c1, bf, px / 16 * 256);
  CV("c3_1", p2, 128, nullptr, 0, H4, W4, 9, 1, 256, true, c1);
  ARENA_GET(s2, bf, px / 16 * 256);  // relu3_2
  CV("c3_2", c1, 256, nullptr, 0, H4, W4, 9, 1, 256, true, s2);
  ARENA_GET(p3, bf, px / 64 * 256);
  RUN(conv_pool("c3_3", s2, 256, H4, W4, 256, nullptr, p3));
  ARENA_GET(d1, bf, px / 64 * 512);
  CV("c4_1", p3, 256, nullptr, 0, H8, W8, 9, 1, 512, true, d1);
  ARENA_GET(s3, bf, px / 64 * 512);  // "relu4_3" (really conv4_2)
  CV("c4_2", d1, 512, nullptr, 0, H8, W8, 9, 1, 512, true, s3);
  ARENA_GET(p4, bf, px / 256 * 512);
  RUN(conv_pool("c4_3", s3, 512, H8, W8, 512, nullptr, p4));
  ARENA_GET(e1, bf, px / 256 * 512);
  CV("c5_1", p4, 512, nullptr, 0, H16, W16, 9, 1, 512, true, e1);
  ARENA_GET(s4, bf, px / 256 * 512);  // "relu5_3": conv5_2 + BN, NOT ReLU'd (slice5 starts with a MaxPool)
  CV("c5_2", e1, 512, nullptr, 0, H16, W16, 9, 1, 512, false, s4);
  ARENA_GET(m5, bf, px / 256 * 512);
  RUN(maxpool3x3s1(s4, m5, B, H16, W16, 512, s));
  ARENA_GET(f6, bf, px / 256 * 1024);
  CV("fc6", m5, 512, nullptr, 0, H16, W16, 9, 6, 1024, false, f6);
  ARENA_GET(f7, bf, px / 256 * 1024);
  CV("fc7", f6, 1024, nullptr, 0, H16, W16, 1, 1, 1024, false, f7);
  // U-net head: double_conv(cat[y, skip]) with the concat fused into the 1x1 conv's K loop
  ARENA_GET(u1a, bf, px / 256 * 512);
  CV("up1a", f7, 1024, s4, 512, H16, W16, 1, 1, 512, true, u1a);
  ARENA_GET(y1, bf, px / 256 * 256);
  CV("up1b", u1a, 512, nullptr, 0, H16, W16, 9, 1, 256, true, y1);
  ARENA_GET(y1u, bf, px / 64 * 256);
  RUN(upsample2x(y1, y1u, B, H16, W16, 256, s));
  ARENA_GET(u2a, bf, px / 64 * 256);
  CV("up2a", y1u, 256, s3, 512, H8, W8, 1, 1, 256, true, u2a);
  ARENA_GET(y2, bf, px / 64 * 128);
  CV("up2b", u2a, 256, nullptr, 0, H8, W8, 9, 1, 128, true, y2);
  ARENA_GET(y2u, bf, px / 16 * 128);
  RUN(upsample2x(y2, y2u, B, H8, W8, 128, s));
  ARENA_GET(u3a, bf, px / 16 * 128);
  CV("up3a", y2u, 128, s2, 256, H4, W4, 1, 1, 128, true, u3a);
  ARENA_GET(y3, bf, px / 16 * 64);
  CV("up3b", u3a, 128, nullptr, 0, H4, W4, 9, 1, 64, true, y3);
  ARENA_GET(y3u, bf, px / 4 * 64);
  RUN(upsample2x(y3, y3u, B, H4, W4, 64, s));
  ARENA_GET(u4a, bf, px / 4 * 64);
  CV("up4a", y3u, 64, s1, 128, H2, W2, 1, 1, 64, true, u4a);
  ARENA_GET(y4, bf, px / 4 * 32);
  CV("up4b", u4a, 64, nullptr, 0, H2, W2, 9, 1, 32, true, y4);
  ARENA_GET(k1, bf, px / 4 * 32);
  CV("cls1", y4, 32, nullptr, 0, H2, W2, 9, 1, 32, true, k1);
  ARENA_GET(k2, bf, px / 4 * 32);
  CV("cls2", k1, 32, nullptr, 0, H2, W2, 9, 1, 32, true, k2);
  ARENA_GET(maps, float, px / 4 * 2);
  {
    // cls3 (3x3 32->16 + ReLU) with cls4 (1x1 16->16 + ReLU) and cls5 (1x1 16->2) in its epilogue,
    // writing the (H/2, W/2, 2) fp32 channels-last map the reference reads (tuatara.cpp:377-394)
    ConvProblem c;
    c.batch = B; c.H = H2; c.W = W2;
    c.src[0] = ConvSrc{k2, 32, 32};
    c.taps = 9; c.dil = 1; c.Cout = 16;
    c.weight = w->craft.bf("cls3.w");
    Epilogue e;
    e.bias = w->craft.f32("cls3.b");
    e.act = ACT_RELU;
    e.out = maps; e.out_type = OUT_CLS_TAIL; e.ldc = 2;
    e.tail = w->craft.f32("cls.tail");
    RUN(conv_forward(c, e, s));
  }
  *maps_out = maps;
  // SURVEY 8d: per-slice parity (names as the oracle's taps: oracle/models.py CRAFT.forward)
  craft_taps = {{"relu2_2", s1, 128, H2, W2}, {"relu3_2", s2, 256, H4, W4}, {"relu4_3", s3, 512, H8, W8},
                {"relu5_3", s4, 512, H16, W16}, {"fc7", f7, 1024, H16, W16}, {"up1", y1, 256, H16, W16},
                {"up2", y2, 128, H8, W8}, {"up3", y3, 64, H4, W4}, {"up4", y4, 32, H2, W2}};
  return cudaSuccess;
}

// ---------------------------------------------------------------------------------- PARSeq
// LayerNorm fused away (see parseq_forward); TT_ENC_LNFUSE=0 keeps the standalone LayerNorm.  Read per call: the parity
// test flips it in-process.
static bool enc_ln_fused(const WeightFile& wf) {
  const char* e = std::getenv("TT_ENC_LNFUSE");
  return !(e && std::atoi(e) == 0) && wf.has("b0.qkv.wf") && wf.has("dec.ca.kvf.wf");
}
static bool enc_attn_onepass() {   // TT_ATTN_ONEPASS=0: the two-pass encoder attention (A/B runs)
  static const bool v = !(std::getenv("TT_ATTN_ONEPASS") && std::atoi(std::getenv("TT_ATTN_ONEPASS")) == 0);
  return v;
}
// qkv projection + attention as one kernel (enc_qkv_attn.cu): the LayerNorm-fused stream only, no qkv buffer then
static bool enc_qkv_attn_fused(const WeightFile& wf, const ParseqDims& pd) {
  return enc_ln_fused(wf) && enc_attn_onepass() && enc_qkv_attn_supported(pd.D, pd.enc_heads);
}

size_t DeviceCtx::parseq_bytes(int n) const {
  const ParseqDims& pd = w->pd;
  const size_t M = static_cast<size_t>(n) * 128, D = pd.D;
  const size_t qkv = enc_qkv_attn_fused(w->parseq, pd) ? 0 : M * 3 * D * 2;
  size_t b = M * D * 4 + M * D * 2 + qkv + M * D * 2 + M * pd.mlp * 2 + M * D * 2 + M * 32 + M * 2 * D * 2;  // encoder
  const size_t R = static_cast<size_t>(n) * pd.L;
  b += R * 4 + R * D * (4 + 2 + 2 + 2) + R * pd.mlp * 2 + 2 * R * pd.n_cls_pad * 4 + 2 * R * 4;
  b += dec_dense_scratch_floats(n, pd.D) * 4;
  b += (static_cast<size_t>(2) * n + 2 * pd.L) * 4;   // early exit: slot -> crop lists and their lengths
  return b + (1u << 20);
}

static cudaError_t lin(cudaStream_t s, const __nv_bfloat16* A, int lda, int M, int K, const __nv_bfloat16* W, int N,
                       const float* bias, int act, const void* res, int res_type, int ldr, int res_mod, void* out,
                       int out_type, int ldc) {
  LinearProblem l;
  l.A = A; l.lda = lda; l.M = M; l.K = K; l.W = W; l.N = N;
  if (N == 96) l.algo_n = 95;  // head: 95 classes stored padded to 96
  Epilogue e;
  e.bias = bias; e.act = act; e.residual = res; e.res_type = res_type; e.ldr = ldr; e.res_mod = res_mod;
  e.out = out; e.out_type = out_type; e.ldc = ldc;
  return linear_forward(l, e, s);
}

cudaError_t DeviceCtx::parseq_forward(const __nv_bfloat16* patches, int n, const int* forced, float** logits_out,
                                      int** ids_out, float* pmax_dev, const uint32_t* mask_dev, const LexDev* lex) {
  using bf = __nv_bfloat16;
  const ParseqDims& pd = w->pd;
  const WeightFile& wf = w->parseq;
  const int D = pd.D, L = pd.L, M = n * 128, NC = pd.n_cls_pad;
  cudaStream_t s = stream;

  // Encoder, in chunks of crops: every intermediate (residual stream, LayerNorm output, qkv, attention
  // output, MLP hidden) lives in chunk-sized buffers that are reused chunk after chunk, so a producer's
  // output is still in the 126 MB L2 when its consumer reads it; only the cross-attention K|V of the
  // memory (what the decoder needs) is written per crop.  At the full batch the same tensors are
  // 7.5 GB of HBM traffic per block and the encoder is HBM-bound (profiles/r1_launches_a5feb26.md).
  static const int chunk_env = std::getenv("TT_ENC_CHUNK") ? std::atoi(std::getenv("TT_ENC_CHUNK")) : 0;
  const int chunk = chunk_env > 0 ? std::min(chunk_env, n) : n;
  const size_t Mc = static_cast<size_t>(chunk) * 128;
  // LayerNorm fused away (gemm_tc.cuh, Epilogue::ln_*): the residual stream x is kept as a bf16 pair (hi, lo) with
  // x = hi + lo (same bytes as fp32, ~2^-17 relative); the residual GEMMs (patch embedding, proj, fc2) update it in
  // fp32 and emit the rows' (sum, sum of squares); qkv / fc1 / the memory K|V projection read `hi` (= bf16(x)) with
  // gamma folded into their weights and apply (mean, rstd) in the epilogue.  Needs the folded tensors of the current
  // weights.py; TT_ENC_LNFUSE=0 keeps the fp32 stream and the standalone LayerNorm kernel (A/B runs, parity test).
  const bool lnf = enc_ln_fused(wf);
  // LN1 + qkv + attention in one kernel whenever the stream is LayerNorm-fused: qkv never reaches HBM (enc_qkv_attn.cu)
  const bool qkv_attn = enc_qkv_attn_fused(wf, pd);
  // fc1 + GELU + fc2 + residual as one kernel (enc_mlp.cu; PARSeq-base dims, split stream): the hidden activations stay
  // on the SM.  TT_ENC_MLPFUSE=0 keeps the two GEMM launches (A/B runs, parity test); PARSeq-tiny always takes them.
  const char* mf_env = std::getenv("TT_ENC_MLPFUSE");   // read per call: the parity test flips it in-process
  const bool mlp_fuse = lnf && !(mf_env && std::atoi(mf_env) == 0) && enc_mlp_supported(D, pd.mlp);
  const char* pf_env = std::getenv("TT_ENC_PROJFUSE");   // 0: the attention output projection stays a GEMM launch (A/B runs)
  const bool proj_fuse = !(pf_env && std::atoi(pf_env) == 0);
  const bool attn_onepass = enc_attn_onepass();
  ARENA_GET(x, float, Mc * D);       // fp32 residual stream (unfused) / the lo half of the split stream (fused; first half of the buffer)
  ARENA_GET(h, bf, Mc * D);          // LayerNorm output (unfused) / the hi half of the split stream = bf16(x) (fused)
  bf* const x_lo = reinterpret_cast<bf*>(x);
  bf* qkv = nullptr;
  if (!qkv_attn) { ARENA_GET(qkv_buf, bf, Mc * 3 * D); qkv = qkv_buf; }
  ARENA_GET(att, bf, Mc * D);
  ARENA_GET(hid, bf, Mc * pd.mlp);
  ARENA_GET(mem, bf, Mc * D);
  ARENA_GET(lnstats, float, Mc * 8);  // fused: per row up to 4 partial (sum, sum of squares)
  ARENA_GET(mem_kv, bf, static_cast<size_t>(M) * 2 * D);

  // residual GEMM x (+)= A W^T + b [+ table]; fused mode: also bf16(x) -> h and the LayerNorm partial sums
  int ln_parts = 0;
  // res == nullptr: the stream itself (in place); else a positional table (fp32 unfused / split pair fused) of res_mod rows
  auto res_gemm = [&](const bf* A, int lda, int Mi, int K, const bf* W, const float* bias, const float* res, int res_mod) -> cudaError_t {
    LinearProblem l;
    l.A = A; l.lda = lda; l.M = Mi; l.K = K; l.W = W; l.N = D;
    Epilogue e;
    e.bias = bias; e.ldr = D; e.res_mod = res_mod; e.ldc = D;
    if (lnf) {
      const bf* tab = w->pos_split;
      e.res_type = RES_SPLIT; e.out_type = OUT_SPLIT;
      e.residual = res ? tab : h; e.residual_lo = res ? tab + static_cast<size_t>(res_mod) * D : x_lo;
      e.out = h; e.out_lo = x_lo;
      e.ln_stats_out = lnstats; e.ln_parts_out = &ln_parts;
    } else {
      e.residual = res ? res : x; e.res_type = RES_F32;
      e.out = x; e.out_type = OUT_F32;
    }
    return linear_forward(l, e, s);
  };
  // y = Linear(LN(x)) [GELU]: fused mode reads h = bf16(x) with the folded weights `name`.wf / .c0 / .c1
  auto ln_gemm = [&](const std::string& name, int Mi, int N, int act, bf* out) -> cudaError_t {
    LinearProblem l;
    l.A = h; l.lda = D; l.M = Mi; l.K = D; l.W = wf.bf(name + (lnf ? ".wf" : ".w")); l.N = N;
    Epilogue e;
    e.bias = wf.f32(name + (lnf ? ".c0" : ".b")); e.act = act;
    e.out = out; e.out_type = OUT_BF16; e.ldc = N;
    if (lnf) { e.ln_stats_in = lnstats; e.ln_c1 = wf.f32(name + ".c1"); e.ln_parts = ln_parts; e.ln_dim = D; e.ln_eps = 1e-6f; }
    return linear_forward(l, e, s);
  };

  stage_begin(s);
  for (int c0 = 0; c0 < n; c0 += chunk) {
    const int nc = std::min(chunk, n - c0);
    const int Mi = nc * 128;
    const bf* pch = patches + static_cast<size_t>(c0) * 128 * 96;
    // patch embedding (Conv2d k=s=(4,8) as a K=96 GEMM) + bias + pos_embed
    RUN(res_gemm(pch, 96, Mi, 96, wf.bf("pe.w"), wf.f32("pe.b"), wf.f32("pos"), 128));
    for (int i = 0; i < pd.depth; ++i) {
      const std::string p = "b" + std::to_string(i) + ".";
      if (!lnf) RUN(layernorm(x, Mi, D, wf.f32(p + "ln1.g"), wf.f32(p + "ln1.b"), 1e-6f, h, nullptr, 0, s));
      if (qkv_attn) {
        RUN(enc_qkv_attn_forward(h, lnstats, ln_parts, wf.bf(p + "qkv.wf"), wf.f32(p + "qkv.c0"), wf.f32(p + "qkv.c1"), att, nc, D,
                                 pd.enc_heads, 1e-6f, s));
      } else {
        RUN(ln_gemm(p + "qkv", Mi, 3 * D, ACT_NONE, qkv));
        RUN(attention_enc(qkv, att, nc, D, pd.enc_heads, attn_onepass, s));
      }
      if (mlp_fuse && proj_fuse) {
        // proj + residual + fc1 -> GELU -> fc2 + residual in one kernel: x1 never leaves the SM either (enc_mlp.cu)
        EncMlpWeights mw;
        mw.w1 = wf.bf(p + "fc1.wf"); mw.c0 = wf.f32(p + "fc1.c0"); mw.c1 = wf.f32(p + "fc1.c1");
        mw.w2 = wf.bf(p + "fc2.w"); mw.b2 = wf.f32(p + "fc2.b");
        EncProj pj;
        pj.att = att; pj.wp = wf.bf(p + "proj.w"); pj.bp = wf.f32(p + "proj.b");
        RUN(enc_mlp_forward(mw, h, x_lo, lnstats, 2, Mi, D, pd.mlp, 1e-6f, s, &pj));
        ln_parts = 2;
        continue;
      }
      RUN(res_gemm(att, D, Mi, D, wf.bf(p + "proj.w"), wf.f32(p + "proj.b"), nullptr, 0));
      if (mlp_fuse && ln_parts == 2) {
        // fc1 -> GELU -> fc2 -> residual in one kernel: the hidden activations stay on the SM (enc_mlp.cu)
        EncMlpWeights mw;
        mw.w1 = wf.bf(p + "fc1.wf"); mw.c0 = wf.f32(p + "fc1.c0"); mw.c1 = wf.f32(p + "fc1.c1");
        mw.w2 = wf.bf(p + "fc2.w"); mw.b2 = wf.f32(p + "fc2.b");
        RUN(enc_mlp_forward(mw, h, x_lo, lnstats, ln_parts, Mi, D, pd.mlp, 1e-6f, s));
        continue;
      }
      if (!lnf) RUN(layernorm(x, Mi, D, wf.f32(p + "ln2.g"), wf.f32(p + "ln2.b"), 1e-6f, h, nullptr, 0, s));
      RUN(ln_gemm(p + "fc1", Mi, pd.mlp, ACT_GELU, hid));
      RUN(res_gemm(hid, pd.mlp, Mi, pd.mlp, wf.bf(p + "fc2.w"), wf.f32(p + "fc2.b"), nullptr, 0));
    }
    // cross-attention K/V of the memory = rows D.. of cross_attn.in_proj applied to the encoder's final LayerNorm, once per crop
    bf* mkv = mem_kv + static_cast<size_t>(c0) * 128 * 2 * D;
    if (lnf) {
      RUN(ln_gemm("dec.ca.kvf", Mi, 2 * D, ACT_NONE, mkv));
    } else {
      RUN(layernorm(x, Mi, D, wf.f32("enc.ln.g"), wf.f32("enc.ln.b"), 1e-6f, mem, nullptr, 0, s));
      RUN(lin(s, mem, D, Mi, D, wf.bf("dec.ca.in.w") + static_cast<size_t>(D) * D, 2 * D, wf.f32("dec.ca.in.b") + D, ACT_NONE,
              nullptr, RES_NONE, 0, 0, mkv, OUT_BF16, 2 * D));
    }
  }

  stage_end(s, "parseq_encoder", 5.75e9 * n, 0.0);  // SURVEY 8a row 9: 2 x 2.874 GMAC per crop
  // ---- decoder: 26 autoregressive steps + one cloze refinement (SURVEY App. B)
  // Content-stream K|V come from the (position, token) table built at init, so a step is: self attention ->
  // [out_proj, norm1, q_proj] -> cross attention -> [ca.out, norm2, MLP, norm, head, argmax].  The two bracketed groups
  // are one fused tcgen05 kernel each (dec_fused.cu); TT_DEC_FUSED=0 runs them as separate GEMM / LayerNorm launches.
  const int R = n * L;
  const char* fused_env = std::getenv("TT_DEC_FUSED");   // read per call: the parity test flips it in-process
  const bool fused = !(fused_env && std::atoi(fused_env) == 0) && w->dd.ready;
  ARENA_GET(tokens, int, static_cast<size_t>(R));
  ARENA_GET(t, float, static_cast<size_t>(R) * D);
  ARENA_GET(hb, bf, static_cast<size_t>(R) * D);
  ARENA_GET(qc, bf, static_cast<size_t>(R) * D);
  ARENA_GET(ab, bf, static_cast<size_t>(R) * D);
  ARENA_GET(dh, bf, static_cast<size_t>(R) * pd.mlp);
  ARENA_GET(logits_ar, float, static_cast<size_t>(R) * NC);
  ARENA_GET(logits, float, static_cast<size_t>(R) * NC);
  ARENA_GET(ids, int, static_cast<size_t>(R));
  ARENA_GET(t_scratch, float, dec_dense_scratch_floats(n, D));
  ARENA_GET(act, int, static_cast<size_t>(2) * n);       // early exit: two generations of the slot -> crop lists (both halves)
  ARENA_GET(act_n, int, static_cast<size_t>(2) * L);     // live crops of half h before step i at [h * L + i]
  const char* ee_env = std::getenv("TT_DEC_EARLY_EXIT");   // read per call: the parity test flips it in-process
  const bool early = fused && forced == nullptr && !(ee_env && std::atoi(ee_env) == 0);
  int ar_counts_h[64];
  double ar_passes = static_cast<double>(n) * L;           // crop-steps of the AR pass
  RUN(tokens_init(tokens, n, L, pd.bos_id, pd.pad_id, s));
  const float* posq = wf.f32("posq");
  const bf* kv_table = w->kv_table;
  stage_begin(s);
  auto stream_tail = [&](const DecoderStep& st, int rows, float* logits_dst, int ldl) -> cudaError_t {
    // t = posq[p] + out_proj(self_attn); t += cross_attn(norm1(t)); t += mlp(norm2(t)); head(norm(t))
    RUN(dec_self_attn(st, w->q_sa_table, w->sc_table, kv_table, tokens, pd.eos_id, pd.n_tok, ab, s));
    RUN(lin(s, ab, D, rows, D, wf.bf("dec.sa.out.w"), D, wf.f32("dec.sa.out.b"), ACT_NONE, posq + static_cast<size_t>(st.p0) * D,
            RES_F32, D, st.np, t, OUT_F32, D));
    RUN(layernorm(t, rows, D, wf.f32("dec.n1.g"), wf.f32("dec.n1.b"), 1e-5f, hb, nullptr, 0, s));
    RUN(lin(s, hb, D, rows, D, wf.bf("dec.ca.in.w"), D, wf.f32("dec.ca.in.b"), ACT_NONE, nullptr, RES_NONE, 0, 0, qc, OUT_BF16, D));
    RUN(dec_cross_attn(st, qc, mem_kv, ab, s));
    RUN(lin(s, ab, D, rows, D, wf.bf("dec.ca.out.w"), D, wf.f32("dec.ca.out.b"), ACT_NONE, t, RES_F32, D, 0, t, OUT_F32, D));
    RUN(layernorm(t, rows, D, wf.f32("dec.n2.g"), wf.f32("dec.n2.b"), 1e-5f, hb, nullptr, 0, s));
    RUN(lin(s, hb, D, rows, D, wf.bf("dec.l1.w"), pd.mlp, wf.f32("dec.l1.b"), ACT_GELU, nullptr, RES_NONE, 0, 0, dh, OUT_BF16, pd.mlp));
    RUN(lin(s, dh, pd.mlp, rows, pd.mlp, wf.bf("dec.l2.w"), D, wf.f32("dec.l2.b"), ACT_NONE, t, RES_F32, D, 0, t, OUT_F32, D));
    RUN(layernorm(t, rows, D, wf.f32("dec.norm.g"), wf.f32("dec.norm.b"), 1e-5f, hb, nullptr, 0, s));
    RUN(lin(s, hb, D, rows, D, wf.bf("head.w"), NC, wf.f32("head.b"), ACT_NONE, nullptr, RES_NONE, 0, 0, logits_dst, OUT_F32, ldl));
    return cudaSuccess;
  };
  if (fused) {
    // The AR loop is crop-local, so the batch runs as two independent halves on two streams: the dense kernels of one
    // half (128 crops per CTA: 75 CTAs for a 32-page group, latency / L2 bound) overlap the HBM-bound cross attention
    // of the other.  Small batches stay on one stream.
    const int n0 = (n >= 512 && stream2) ? ((n / 2 + 127) / 128) * 128 : n;
    // Per-crop early exit: a crop whose step produced EOS leaves the loop (dec_compact keeps the slot -> crop list of the
    // crops still decoding, its length stays on the device: the grids cover all crops, surplus blocks return at once).
    // Upstream PARSeq stops a batch once every sequence has an EOS and the reference feeds it 4 crops at a time
    // (tuatara.cpp:452-475); nothing after a crop's first EOS reaches the refinement pass -- its keys are masked from
    // there on -- or the decoded string, so the outputs are the ones of the full schedule.  Off under teacher forcing
    // (the parity tests compare every position) and with TT_DEC_EARLY_EXIT=0.
    for (int h = 0; h < 2; ++h)
      for (int i = 0; i < L; ++i) ar_counts_h[h * L + i] = 0;
    auto ar_step = [&](int i, int c0, int nc, int half, cudaStream_t hs) -> cudaError_t {
      int* tok_h = tokens + static_cast<size_t>(c0) * L;
      bf* ab_h = ab + static_cast<size_t>(c0) * D;
      bf* qc_h = qc + static_cast<size_t>(c0) * D;
      float* ts_h = t_scratch + static_cast<size_t>(c0) * D;   // c0 is a multiple of 128: whole tiles
      float* la_h = logits_ar + static_cast<size_t>(c0) * L * NC;
      const int* forced_h = forced ? forced + static_cast<size_t>(c0) * (L - 1) : nullptr;
      const bf* mkv_h = mem_kv + static_cast<size_t>(c0) * 128 * 2 * D;
      const uint32_t* mask_h = mask_dev ? mask_dev + static_cast<size_t>(c0) * 4 : nullptr;
      LexDev lex_h{};   // the half's crops' walk state; under teacher forcing the AR steps do not consult the automaton
      if (lex && !forced) {
        lex_h = *lex;
        lex_h.root += c0;
        lex_h.state += c0;
      }
      // lists hold crop indices relative to the half; step 0 works on all of them (no list)
      int* const cnt = act_n + half * L;
      const int* cur = (early && i > 0) ? act + static_cast<size_t>(i & 1) * n + c0 : nullptr;
      const int* cur_n = (early && i > 0) ? cnt + i : nullptr;
      DecoderStep st{nc, D, pd.dec_heads, L, i, 1, 0};
      st.active = cur; st.n_act = cur_n;
      RUN(dec_self_attn(st, w->q_sa_table, w->sc_table, kv_table, tok_h, pd.eos_id, pd.n_tok, ab_h, hs));
      RUN(dec_dense_a2(w->dd, ab_h, nc, i, ts_h, qc_h, hs, cur, cur_n));
      RUN(dec_cross_attn(st, qc_h, mkv_h, ab_h, hs));
      RUN(dec_dense_b(w->dd, ab_h, nc, i, ts_h, la_h, tok_h, forced_h, hs, cur, cur_n, mask_h, lex_h.root ? &lex_h : nullptr,
                      i == 0));
      if (early && i + 1 < L)
        RUN(dec_compact(cur, cur_n, nc, tok_h, L, i + 1, pd.eos_id, act + static_cast<size_t>((i + 1) & 1) * n + c0, cnt + i + 1, hs));
      return cudaSuccess;
    };
    if (n0 < n) {
      TT_CUDA_TRY(cudaEventRecord(ev_fork, s));
      TT_CUDA_TRY(cudaStreamWaitEvent(stream2, ev_fork, 0));
      for (int i = 0; i < L; ++i) {   // launches interleaved so that neither stream's queue runs dry
        RUN(ar_step(i, 0, n0, 0, s));
        RUN(ar_step(i, n0, n - n0, 1, stream2));
      }
      TT_CUDA_TRY(cudaEventRecord(ev_join, stream2));
      TT_CUDA_TRY(cudaStreamWaitEvent(s, ev_join, 0));
    } else {
      for (int i = 0; i < L; ++i) RUN(ar_step(i, 0, n, 0, s));
    }
    if (early && prof_enabled()) {   // the stage's algorithmic work is what the live crops did: read the counts back (profiling passes only)
      TT_CUDA_TRY(cudaMemcpyAsync(ar_counts_h, act_n, sizeof(int) * 2 * L, cudaMemcpyDeviceToHost, s));
      TT_CUDA_TRY(stream_sync(s));
      ar_passes = static_cast<double>(n);   // step 0: every crop
      for (int h = 0; h < (n0 < n ? 2 : 1); ++h)
        for (int i = 1; i < L; ++i) ar_passes += ar_counts_h[h * L + i];
    }
  } else {
    for (int i = 0; i < L; ++i) {
      DecoderStep st{n, D, pd.dec_heads, L, i, 1, 0};
      RUN(stream_tail(st, n, logits_ar + static_cast<size_t>(i) * NC, L * NC));
      if (i + 1 < L)
        RUN(argmax_rows(logits_ar + static_cast<size_t>(i) * NC, n, pd.n_cls, L * NC, nullptr, 0, tokens + i + 1, L,
                        forced ? forced + i : nullptr, L - 1, s, mask_dev, 1, forced ? nullptr : lex, i == 0));
    }
  }
  DecoderStep st{n, D, pd.dec_heads, L, 0, L, 1};
  RUN(stream_tail(st, R, logits, NC));
  if (lex)   // lexicons: each crop walks its positions in order from its root (the ids, and pmax when requested)
    RUN(lexicon_walk(logits, n, L, pd.n_cls, NC, *lex, ids, pmax_dev, s));
  else if (pmax_dev)   // scores requested: the same ids plus each position's largest softmax probability, in the same launch
    RUN(argmax_conf_rows(logits, R, pd.n_cls, NC, ids, pmax_dev, s, mask_dev, L));
  else
    RUN(argmax_rows(logits, R, pd.n_cls, NC, ids, 1, nullptr, 0, nullptr, 0, s, mask_dev, L));
  // decoder: 2 x 0.153 GMAC per crop over L + 1 passes; its floor is one read of the crop's memory K|V (128 x 768 bf16) per
  // pass the crop takes part in: L AR steps (fewer with the early exit) + the refinement
  {
    const double passes = ar_passes + n;
    stage_end(s, "parseq_decoder", 0.306e9 / (L + 1) * passes, passes * 128 * 768 * 2);
  }
  // test hook (tests/test_models_gpu.py): hand back the AR pass's logits instead of the refinement's
  const char* ar_env = std::getenv("TT_PARSEQ_AR_LOGITS");
  *logits_out = (ar_env && std::atoi(ar_env) != 0) ? logits_ar : logits;
  *ids_out = ids;
  return cudaSuccess;
}

// ------------------------------------------------------------------------------- DeviceCtx
DeviceWeights::~DeviceWeights() {
  cudaSetDevice(device);
  if (q_sa_table) cudaFree(q_sa_table);
  if (kv_table) cudaFree(kv_table);
  if (sc_table) cudaFree(sc_table);
  if (pos_split) cudaFree(pos_split);
  dec_dense_free(&dd);
}

DeviceCtx::~DeviceCtx() {
  cudaSetDevice(device);
  post_workspace_free(&post);
  if (patch_buf) cudaFree(patch_buf);
  if (lex_buf) cudaFree(lex_buf);
  if (pinned) cudaFreeHost(pinned);
  if (ev_fork) cudaEventDestroy(ev_fork);
  if (ev_join) cudaEventDestroy(ev_join);
  if (stream2) cudaStreamDestroy(stream2);
  if (stream) cudaStreamDestroy(stream);
}

cudaError_t DeviceCtx::ensure_pinned(size_t bytes) {
  if (bytes <= pinned_bytes) return cudaSuccess;
  if (pinned) cudaFreeHost(pinned);
  pinned = nullptr;
  pinned_bytes = 0;
  TT_CUDA_TRY(cudaMallocHost(reinterpret_cast<void**>(&pinned), bytes));
  pinned_bytes = bytes;
  return cudaSuccess;
}

cudaError_t DeviceCtx::init(const std::string& dir, std::shared_ptr<DeviceWeights> shared) {
  TT_CUDA_TRY(cudaSetDevice(device));
  TT_CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  TT_CUDA_TRY(cudaStreamCreateWithFlags(&stream2, cudaStreamNonBlocking));
  TT_CUDA_TRY(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
  TT_CUDA_TRY(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
  if (shared) {
    w = std::move(shared);
    return cudaSuccess;
  }
  w = std::make_shared<DeviceWeights>();
  w->device = device;
  ParseqDims& pd = w->pd;
  std::vector<int> meta;
  if (!w->craft.load(dir + "/craft.ttw")) return cudaErrorInvalidValue;
  if (!w->parseq.load(dir + "/parseq.ttw", &meta)) return cudaErrorInvalidValue;
  if (meta.size() >= 8) {
    pd.D = meta[0]; pd.depth = meta[1]; pd.enc_heads = meta[2]; pd.dec_heads = meta[3]; pd.mlp = meta[4];
    pd.n_cls = meta[5]; pd.L = meta[6]; pd.n_tok = meta[7];
    pd.n_cls_pad = (pd.n_cls + 15) / 16 * 16;
    pd.eos_id = 0; pd.bos_id = pd.n_tok - 2; pd.pad_id = pd.n_tok - 1;
  }
  // PARSeq-base (384 / 6 / 12 heads) and PARSeq-tiny (192 / 3 / 6): head dims are 64 (encoder) and 32 (decoder) in both
  if (!(pd.D == 384 || pd.D == 192) || pd.enc_heads * 64 != pd.D || pd.dec_heads * 32 != pd.D || pd.L > 32 || pd.mlp % 128 != 0) {
    set_error("unsupported PARSeq dimensions (built for embed_dim 384 and 192, head dims 64 / 32, <= 32 positions)");
    return cudaErrorInvalidValue;
  }
  // self-attention queries: W_q LN_q(pos_queries) + b_q, identical for every crop
  const WeightFile& wf = w->parseq;
  const int D = pd.D, L = pd.L, NT = pd.n_tok;
  TT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&w->q_sa_table), sizeof(float) * L * D));
  TT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&w->kv_table), sizeof(__nv_bfloat16) * L * NT * 2 * D));
  TT_CUDA_TRY(arena.reserve((4u << 20) + static_cast<size_t>(NT) * (L * 4 + D * 2)));
  arena.reset();
  __nv_bfloat16* qn = arena.get<__nv_bfloat16>(static_cast<size_t>(L) * D);
  RUN(layernorm(wf.f32("posq"), L, D, wf.f32("dec.nq.g"), wf.f32("dec.nq.b"), 1e-5f, qn, nullptr, 0, stream));
  RUN(lin(stream, qn, D, L, D, wf.bf("dec.sa.in.w"), D, wf.f32("dec.sa.in.b"), ACT_NONE, nullptr,
          RES_NONE, 0, 0, w->q_sa_table, OUT_F32, D));
  // Content-stream K|V of every (position, token): rows D.. of self_attn.in_proj applied to
  // LN_c(sqrt(D) E[token] + pos_queries[position - 1]) (bos sits at position 0 without a positional term).  One decoder
  // layer => these 26 x 97 rows are all the self-attention keys / values any crop can ever have.
  {
    std::vector<int> tok(static_cast<size_t>(NT) * L);
    for (int c = 0; c < NT; ++c)
      for (int j = 0; j < L; ++j) tok[static_cast<size_t>(c) * L + j] = c;
    int* tok_d = arena.get<int>(tok.size());
    __nv_bfloat16* ctx = arena.get<__nv_bfloat16>(static_cast<size_t>(NT) * D);
    if (!tok_d || !ctx) { set_error("arena exhausted (kv table)"); return cudaErrorMemoryAllocation; }
    TT_CUDA_TRY(cudaMemcpyAsync(tok_d, tok.data(), tok.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
    for (int j = 0; j < L; ++j) {
      RUN(dec_context(tok_d, wf.f32("embed"), wf.f32("posq"), wf.f32("dec.nc.g"), wf.f32("dec.nc.b"), 1e-5f, j, NT, D, L, ctx, stream));
      RUN(lin(stream, ctx, D, NT, D, wf.bf("dec.sa.in.w") + static_cast<size_t>(D) * D, 2 * D, wf.f32("dec.sa.in.b") + D, ACT_NONE,
              nullptr, RES_NONE, 0, 0, w->kv_table + static_cast<size_t>(j) * NT * 2 * D, OUT_BF16, 2 * D));
    }
    TT_CUDA_TRY(stream_sync(stream));   // `tok` must outlive the copy
  }
  TT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&w->pos_split), sizeof(__nv_bfloat16) * 2 * 128 * D));
  RUN(split_f32(wf.f32("pos"), 128LL * D, w->pos_split, w->pos_split + 128 * D, stream));
  TT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&w->sc_table), sizeof(float) * L * L * NT * pd.dec_heads));
  RUN(dec_score_table(w->q_sa_table, w->kv_table, L, NT, D, pd.dec_heads, w->sc_table, stream));
  // fused decoder kernels: weight tensor maps + per-column vectors
  {
    DecDenseWeights& dd = w->dd;
    if (!dec_dense_init(&dd, D, pd.mlp, pd.n_cls, pd.n_cls_pad, L, wf.bf("dec.sa.out.w"), wf.bf("dec.ca.in.w"), wf.bf("dec.ca.out.w"),
                        wf.bf("dec.l1.w"), wf.bf("dec.l2.w"), wf.bf("head.w")))
      return cudaErrorInvalidValue;
    dd.bo = wf.f32("dec.sa.out.b"); dd.bq = wf.f32("dec.ca.in.b"); dd.bco = wf.f32("dec.ca.out.b");
    dd.b1 = wf.f32("dec.l1.b"); dd.b2 = wf.f32("dec.l2.b"); dd.bh = wf.f32("head.b");
    dd.n1_g = wf.f32("dec.n1.g"); dd.n1_b = wf.f32("dec.n1.b"); dd.n2_g = wf.f32("dec.n2.g"); dd.n2_b = wf.f32("dec.n2.b");
    dd.nf_g = wf.f32("dec.norm.g"); dd.nf_b = wf.f32("dec.norm.b");
    dd.posq = wf.f32("posq");
    RUN(dec_dense_pack(&dd, stream));
  }
  TT_CUDA_TRY(stream_sync(stream));
  return cudaSuccess;
}

}  // namespace tt
