// The engine behind tt_engine_*: per-GPU weight replicas, streams and workspaces; pages are
// sharded over GPUs by one host worker thread per device, results gathered on the host.
// Replaces the orchestration of image_to_data (tuatara.cpp:314-512).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "dec_fused.cuh"
#include "detect.h"
#include "postprocess.cuh"
#include "tuatara_c.h"

namespace tt {

struct WTensor {
  void* ptr = nullptr;
  int dtype = 0;  // 0 f32, 1 bf16, 2 i32
  std::vector<long long> dims;
  size_t nbytes = 0;
};

// A .ttw file resident on one device (tuatara_b200/weights.py documents the format).
class WeightFile {
 public:
  ~WeightFile();
  bool load(const std::string& path, std::vector<int>* meta_out = nullptr);
  const WTensor& get(const std::string& name) const;  // throws std::runtime_error when missing
  bool has(const std::string& name) const { return t_.find(name) != t_.end(); }
  const __nv_bfloat16* bf(const std::string& name) const { return static_cast<const __nv_bfloat16*>(get(name).ptr); }
  const float* f32(const std::string& name) const { return static_cast<const float*>(get(name).ptr); }

 private:
  std::map<std::string, WTensor> t_;
  void* arena_ = nullptr;
};

// Grow-only device scratch: reset() at the start of a forward pass, alloc() bumps.
class Arena {
 public:
  ~Arena();
  cudaError_t reserve(size_t bytes);
  void reset() { off_ = 0; }
  size_t offset() const { return off_; }
  void reset_to(size_t off) { off_ = off; }  // drop everything allocated after a mark taken with offset()
  void* alloc(size_t bytes);  // nullptr when exhausted (caller reserved too little)
  template <class T> T* get(size_t n) { return static_cast<T*>(alloc(n * sizeof(T))); }
  size_t capacity() const { return cap_; }

 private:
  uint8_t* base_ = nullptr;
  size_t cap_ = 0, off_ = 0;
};

struct ParseqDims {
  int D = 384, depth = 12, enc_heads = 6, dec_heads = 12, mlp = 1536, n_cls = 95, L = 26, n_tok = 97;
  int n_cls_pad = 96;
  int eos_id = 0, bos_id = 95, pad_id = 96;
};

// Read-only state shared by the execution slots of one GPU: the two weight files and what is derived from them.
struct DeviceWeights {
  int device = 0;
  WeightFile craft, parseq;
  ParseqDims pd;
  float* q_sa_table = nullptr;  // [L][D] fp32: self-attn queries of the 26 positions (crop independent)
  __nv_bfloat16* kv_table = nullptr;  // [L][n_tok][2D] bf16: content-stream K|V of every (position, token) pair
  __nv_bfloat16* pos_split = nullptr;  // [2][128][D] bf16: pos_embed as a (hi, lo) pair, the patch embedding's split residual
  float* sc_table = nullptr;    // [L][L][n_tok][dec_heads] fp32: AR self-attention scores as a lookup (nn_kernels.cuh)
  DecDenseWeights dd;           // tensor maps + vectors of the fused decoder kernels (dec_fused.cu)
  ~DeviceWeights();
};

// One execution slot: a stream with its own scratch arena and workspaces.  Each GPU runs up to kSlotsPerDevice
// of them from separate host threads so that one slot's host-side phases (box geometry, result
// assembly, D2H waits) and its latency-bound kernels (the decoder's AR loop) are covered by the other slots' kernels.
// Measured on the 512-page bench: 1 slot 211, 2 slots 245, 3 slots 251, 4 slots 252 pages/s.
constexpr int kSlotsPerDevice = 4;   // upper bound; tt_config.slots_per_gpu picks how many run (0 = default 3)

// A named CRAFT activation of the most recent craft_forward (arena memory: valid until the slot's next call).
struct CraftTap { const char* name; const __nv_bfloat16* ptr; int C, H, W; };

struct DeviceCtx {
  int device = 0;
  std::vector<CraftTap> craft_taps;   // per-slice parity test (tt_craft_tap): image 0 of the batch
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;  // second half of a recognition batch's AR loop (overlaps the first half's cross attention)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  std::shared_ptr<DeviceWeights> w;
  Arena arena;
  PostWorkspace post;           // sized lazily for (batch, H, W)
  __nv_bfloat16* patch_buf = nullptr;  // recognition batch: bf16 patch rows [crops * 128][96] of the crops awaiting PARSeq
  size_t patch_cap = 0;                //   capacity in crops
  void* lex_buf = nullptr;             // the automaton table of the lexicon request this slot runs (lexicon.h layout)
  size_t lex_cap = 0;                  //   capacity in bytes
  LexDev lex_view;                     //   its table pointers (root / state unset)
  uint8_t* pinned = nullptr;    // host staging for D2H of post results / ids
  size_t pinned_bytes = 0;
  std::mutex mu;                // one request at a time per device

  ~DeviceCtx();
  // shared == nullptr: load the weights; otherwise become another slot on the same GPU
  cudaError_t init(const std::string& weights_dir, std::shared_ptr<DeviceWeights> shared);
  cudaError_t ensure_pinned(size_t bytes);
  // CRAFT: device u8 [B][H][W][3] (already swapped/padded) -> device fp32 maps [B][H/2][W/2][2] (arena memory)
  cudaError_t craft_forward(const uint8_t* input_dev, int B, int H, int W, float** maps_out);
  size_t craft_bytes(int B, int H, int W) const;
  // PARSeq: device bf16 patches [n*128][96] -> device fp32 logits [n][L][n_cls_pad] + int ids [n][L] (arena).
  // pmax_dev (nullable, device [n][L]): also the largest softmax probability of each refinement position.
  // mask_dev (nullable, device [n][4] uint32, 16-byte aligned): per-crop class masks (tt_char_filter_mask); every greedy
  // choice -- each AR step's fed-back token and the refinement's ids -- and pmax run over the allowed classes only.  The
  // logits are not masked.
  // lex (nullable; mask_dev is then null): the state path of a lexicon request (INTEGRATION.md section 9).  Every AR
  // step feeds back the argmax over the classes its crop's state allows (from lex->root, advancing lex->state [n]);
  // without forced_dev only.  The refinement's ids and pmax are a second walk from lex->root (lexicon_walk).
  cudaError_t parseq_forward(const __nv_bfloat16* patches_dev, int n, const int* forced_dev, float** logits_out,
                             int** ids_out, float* pmax_dev = nullptr, const uint32_t* mask_dev = nullptr,
                             const LexDev* lex = nullptr);
  size_t parseq_bytes(int n) const;
};

}  // namespace tt

struct tt_engine {
  tt_config cfg;
  std::atomic<int> slots{0};   // live value of cfg.slots_per_gpu (tt_engine_set_slots may change it between calls)
  int n_devices = 0;
  std::vector<std::unique_ptr<tt::DeviceCtx>> devs;  // [device g][slot s] at g * kSlotsPerDevice + s
};
