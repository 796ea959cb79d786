// extern "C" surface (include/tuatara_c.h).  No exceptions cross this boundary.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "common.h"
#include "contrast.cuh"
#include "detect.h"
#include "enc_mlp.cuh"
#include "enc_qkv_attn.cuh"
#include "engine.h"
#include "lexicon.h"
#include "gemm_tc.cuh"
#include "geometry.h"
#include "nn_kernels.cuh"
#include "orient.cuh"
#include "postprocess.cuh"
#include "resize.cuh"
#include "tokenizer.h"
#include "trace.h"
#include "tuatara_c.h"

using namespace tt;

namespace {

template <class F>
int guarded(F&& f) {
  try {
    return f();
  } catch (const std::exception& ex) {
    set_error(std::string("exception: ") + ex.what());
    return 1;
  } catch (...) {
    set_error("unknown exception");
    return 1;
  }
}

struct DevBuf {
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  cudaError_t alloc(size_t n) { return cudaMalloc(&p, n ? n : 1); }
  template <class T> T* as() { return static_cast<T*>(p); }
};

#define TT_TRY_INT(expr)                        \
  do {                                          \
    if ((expr) != cudaSuccess) return 1;        \
  } while (0)
#define TT_CUDA_INT(expr)                                                          \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) {                                                       \
      set_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e));        \
      return 1;                                                                    \
    }                                                                              \
  } while (0)

RotatedRect to_rect(const float r[5]) { return RotatedRect{r[0], r[1], r[2], r[3], r[4]}; }
void from_rect(const RotatedRect& r, float o[5]) { o[0] = r.cx; o[1] = r.cy; o[2] = r.w; o[3] = r.h; o[4] = r.angle; }

}  // namespace

extern "C" {

void tt_config_default(tt_config* cfg) {
  cfg->canvas_size = 1024.f;
  cfg->mag_ratio = 1.0f;
  cfg->text_threshold = 0.7f;
  cfg->link_threshold = 0.4f;
  cfg->low_text = 0.4f;
  cfg->min_area = 10;
  cfg->max_batch_pages = 0;
  cfg->slots_per_gpu = 0;
  cfg->rectify = 0;
}

const char* tt_last_error(void) { return last_error(); }
unsigned long long tt_launch_count(void) { return g_launches.load(); }

int tt_debug_trace_report(char* buf, int cap) {
  const std::string r = trace_report();
  if (!buf || cap <= 0) return static_cast<int>(r.size());
  const size_t n = std::min(r.size(), static_cast<size_t>(cap - 1));
  std::memcpy(buf, r.data(), n);
  buf[n] = 0;
  return static_cast<int>(r.size());
}

int tt_resize_plan(int rows, int cols, float canvas_size, float mag_ratio, int* target_h, int* target_w, int* h32,
                   int* w32, float* ratio) {
  if (rows <= 0 || cols <= 0) { set_error("tt_resize_plan: empty image"); return 1; }
  resize_plan(rows, cols, canvas_size, mag_ratio, target_h, target_w, h32, w32, ratio);
  return 0;
}

int tt_preprocess(const tt_image* image, float canvas_size, float mag_ratio, uint8_t* out) {
  return guarded([&]() -> int {
    if (!image || !image->data || image->channels != 3) { set_error("tt_preprocess: need a 3-channel image"); return 1; }
    int th, tw, h32, w32; float ratio;
    resize_plan(image->rows, image->cols, canvas_size, mag_ratio, &th, &tw, &h32, &w32, &ratio);
    DevBuf src, dst;
    const size_t src_bytes = image->step * image->rows;
    TT_CUDA_INT(src.alloc(src_bytes));
    TT_CUDA_INT(dst.alloc(static_cast<size_t>(h32) * w32 * 3));
    TT_CUDA_INT(cudaMemcpy(src.p, image->data, src_bytes, cudaMemcpyHostToDevice));
    TT_TRY_INT(page_resize_pad(src.as<uint8_t>(), image->rows, image->cols, image->step, dst.as<uint8_t>(), th, tw, h32,
                               w32, 0));
    TT_CUDA_INT(cudaMemcpy(out, dst.p, static_cast<size_t>(h32) * w32 * 3, cudaMemcpyDeviceToHost));
    return 0;
  });
}

int tt_postprocess(const float* maps, int H, int W, const tt_config* cfg_in, int32_t* labels_out, int32_t* stats_out,
                   int stats_cap, int* n_labels, float* rects_out, int32_t* rect_labels_out, int rect_cap,
                   int* n_rects) {
  return guarded([&]() -> int {
    tt_config cfg;
    if (cfg_in) cfg = *cfg_in; else tt_config_default(&cfg);
    const size_t hw = static_cast<size_t>(H) * W;
    if (hw == 0) { set_error("tt_postprocess: empty map"); return 1; }
    DevBuf dmaps;
    TT_CUDA_INT(dmaps.alloc(hw * 2 * sizeof(float)));
    TT_CUDA_INT(cudaMemcpy(dmaps.p, maps, hw * 2 * sizeof(float), cudaMemcpyHostToDevice));
    // stage-level call: size the compact block for the worst case so it never overflows
    const int comp_cap = static_cast<int>(hw / 2 + 2), row_cap = static_cast<int>(hw);
    PostWorkspace ws;
    TT_TRY_INT(post_workspace_alloc(&ws, 1, H, W, comp_cap, row_cap, labels_out != nullptr));
    PostParams pp;
    pp.low_text = cfg.low_text;
    pp.link_threshold = cfg.link_threshold;
    int rc = 0;
    std::vector<uint8_t> block(ws.result_stride);
    if (post_run(ws, dmaps.as<float>(), pp, 0) != cudaSuccess) rc = 1;
    if (!rc && cudaMemcpy(block.data(), ws.result, ws.result_stride, cudaMemcpyDeviceToHost) != cudaSuccess) {
      set_error("tt_postprocess: result copy failed"); rc = 1;
    }
    if (!rc && labels_out &&
        cudaMemcpy(labels_out, ws.labels, hw * sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) {
      set_error("tt_postprocess: label copy failed"); rc = 1;
    }
    post_workspace_free(&ws);
    if (rc) return rc;
    const PostHeader* h = reinterpret_cast<const PostHeader*>(block.data());
    const PostComp* comps = reinterpret_cast<const PostComp*>(block.data() + sizeof(PostHeader));
    if (n_labels) *n_labels = h->n_comp + 1;
    if (stats_out) {
      // row 0 (background) is not produced on the GPU: bbox of all background pixels is not needed
      // by the reference; report zeros with the background area.
      long long fg = 0;
      for (int j = 0; j < h->n_comp; ++j) fg += comps[j].area;
      if (stats_cap > 0) {
        stats_out[0] = 0; stats_out[1] = 0; stats_out[2] = 0; stats_out[3] = 0;
        stats_out[4] = static_cast<int32_t>(static_cast<long long>(hw) - fg);
      }
      for (int j = 0; j < h->n_comp && j + 1 < stats_cap; ++j) {
        int32_t* r = stats_out + static_cast<size_t>(j + 1) * 5;
        r[0] = comps[j].left; r[1] = comps[j].top;
        r[2] = comps[j].right - comps[j].left + 1; r[3] = comps[j].bottom - comps[j].top + 1;
        r[4] = comps[j].area;
      }
    }
    std::vector<DetBox> boxes;
    if (!collect_boxes(block.data(), comp_cap, row_cap, H, W, cfg, &boxes)) {
      set_error("tt_postprocess: internal capacity overflow"); return 1;
    }
    if (n_rects) *n_rects = static_cast<int>(boxes.size());
    for (size_t i = 0; i < boxes.size() && static_cast<int>(i) < rect_cap; ++i) {
      if (rects_out) from_rect(boxes[i].rect, rects_out + i * 5);
      if (rect_labels_out) rect_labels_out[i] = boxes[i].label;
    }
    return 0;
  });
}

int tt_crop_resize(const tt_image* image, const int32_t* rects_xywh, int n, uint8_t* out) {
  return guarded([&]() -> int {
    if (!image || !image->data || image->channels != 3) { set_error("tt_crop_resize: need a 3-channel image"); return 1; }
    if (n <= 0) return 0;
    DevBuf src, dpages, dboxes, dout;
    const size_t src_bytes = image->step * image->rows;
    TT_CUDA_INT(src.alloc(src_bytes));
    TT_CUDA_INT(cudaMemcpy(src.p, image->data, src_bytes, cudaMemcpyHostToDevice));
    PageRef pr{src.as<uint8_t>(), image->rows, image->cols, image->step};
    TT_CUDA_INT(dpages.alloc(sizeof(PageRef)));
    TT_CUDA_INT(cudaMemcpy(dpages.p, &pr, sizeof(pr), cudaMemcpyHostToDevice));
    std::vector<CropBox> boxes(n);
    for (int i = 0; i < n; ++i) {
      const int32_t* r = rects_xywh + 4 * i;
      if (r[0] < 0 || r[1] < 0 || r[2] < 0 || r[3] < 0 || r[0] + r[2] > image->cols || r[1] + r[3] > image->rows) {
        set_error("tt_crop_resize: rect " + std::to_string(i) + " leaves the image (clamp it first)");
        return 1;
      }
      boxes[i] = CropBox{0, r[0], r[1], r[2], r[3]};
    }
    TT_CUDA_INT(dboxes.alloc(sizeof(CropBox) * n));
    TT_CUDA_INT(cudaMemcpy(dboxes.p, boxes.data(), sizeof(CropBox) * n, cudaMemcpyHostToDevice));
    const size_t out_bytes = static_cast<size_t>(n) * 32 * 128 * 3;
    TT_CUDA_INT(dout.alloc(out_bytes));
    TT_TRY_INT(crop_resize(dpages.as<PageRef>(), dboxes.as<CropBox>(), n, dout.as<uint8_t>(), nullptr, 0));
    TT_CUDA_INT(cudaMemcpy(out, dout.p, out_bytes, cudaMemcpyDeviceToHost));
    return 0;
  });
}

int tt_crop_resize_rotated(const tt_image* image, const int32_t* rects_xywh, const int32_t* angles, int n, uint8_t* out) {
  return guarded([&]() -> int {
    if (!image || !image->data || image->channels != 3) { set_error("tt_crop_resize_rotated: need a 3-channel image"); return 1; }
    if (n <= 0) return 0;
    if (!rects_xywh || !angles || !out) { set_error("tt_crop_resize_rotated: null rects, angles or output"); return 1; }
    std::vector<CropBox> boxes(n);
    std::vector<uint8_t> rot(n);
    for (int i = 0; i < n; ++i) {
      const int32_t* r = rects_xywh + 4 * i;
      if (r[0] < 0 || r[1] < 0 || r[2] < 0 || r[3] < 0 || r[0] + r[2] > image->cols || r[1] + r[3] > image->rows) {
        set_error("tt_crop_resize_rotated: rect " + std::to_string(i) + " leaves the image (clamp it first)");
        return 1;
      }
      const int a = angles[i];
      if (a != 0 && a != 90 && a != 180 && a != 270) {
        set_error("tt_crop_resize_rotated: angle " + std::to_string(a) + " of crop " + std::to_string(i) +
                  "; the angles are 0, 90, 180 and 270");
        return 1;
      }
      boxes[i] = CropBox{0, r[0], r[1], r[2], r[3]};
      rot[i] = static_cast<uint8_t>(a / 90);
    }
    DevBuf src, dpages, dboxes, drot, dout;
    const size_t src_bytes = image->step * image->rows;
    TT_CUDA_INT(src.alloc(src_bytes));
    TT_CUDA_INT(cudaMemcpy(src.p, image->data, src_bytes, cudaMemcpyHostToDevice));
    PageRef pr{src.as<uint8_t>(), image->rows, image->cols, image->step};
    TT_CUDA_INT(dpages.alloc(sizeof(PageRef)));
    TT_CUDA_INT(cudaMemcpy(dpages.p, &pr, sizeof(pr), cudaMemcpyHostToDevice));
    TT_CUDA_INT(dboxes.alloc(sizeof(CropBox) * n));
    TT_CUDA_INT(cudaMemcpy(dboxes.p, boxes.data(), sizeof(CropBox) * n, cudaMemcpyHostToDevice));
    TT_CUDA_INT(drot.alloc(n));
    TT_CUDA_INT(cudaMemcpy(drot.p, rot.data(), n, cudaMemcpyHostToDevice));
    const size_t out_bytes = static_cast<size_t>(n) * 32 * 128 * 3;
    TT_CUDA_INT(dout.alloc(out_bytes));
    TT_TRY_INT(crop_resize_rot(dpages.as<PageRef>(), dboxes.as<CropBox>(), drot.as<uint8_t>(), 1, n, dout.as<uint8_t>(), nullptr, 0));
    TT_CUDA_INT(cudaMemcpy(out, dout.p, out_bytes, cudaMemcpyDeviceToHost));
    return 0;
  });
}

int tt_crop_warp(const tt_image* image, const float* quads, int n, uint8_t* out) {
  return guarded([&]() -> int {
    if (!image || !image->data || image->channels != 3 || !quads || !out) { set_error("tt_crop_warp: need a 3-channel image, quads and an output"); return 1; }
    if (n <= 0) return 0;
    DevBuf src, dpages, dboxes, dout;
    const size_t src_bytes = image->step * image->rows;
    TT_CUDA_INT(src.alloc(src_bytes));
    TT_CUDA_INT(cudaMemcpy(src.p, image->data, src_bytes, cudaMemcpyHostToDevice));
    PageRef pr{src.as<uint8_t>(), image->rows, image->cols, image->step};
    TT_CUDA_INT(dpages.alloc(sizeof(PageRef)));
    TT_CUDA_INT(cudaMemcpy(dpages.p, &pr, sizeof(pr), cudaMemcpyHostToDevice));
    std::vector<WarpBox> boxes(n);
    for (int i = 0; i < n; ++i) {
      Pt2f q[4];
      for (int k = 0; k < 4; ++k) q[k] = Pt2f{quads[8 * i + 2 * k], quads[8 * i + 2 * k + 1]};
      boxes[i].page = quad_to_warp(q, boxes[i].m) ? 0 : -1;
      boxes[i].pad_ = 0;
    }
    TT_CUDA_INT(dboxes.alloc(sizeof(WarpBox) * n));
    TT_CUDA_INT(cudaMemcpy(dboxes.p, boxes.data(), sizeof(WarpBox) * n, cudaMemcpyHostToDevice));
    const size_t out_bytes = static_cast<size_t>(n) * 32 * 128 * 3;
    TT_CUDA_INT(dout.alloc(out_bytes));
    TT_TRY_INT(crop_warp(dpages.as<PageRef>(), dboxes.as<WarpBox>(), n, dout.as<uint8_t>(), nullptr, 0));
    TT_CUDA_INT(cudaMemcpy(out, dout.p, out_bytes, cudaMemcpyDeviceToHost));
    return 0;
  });
}

int tt_contrast_adjust(const uint8_t* crops, int n, float adjust_contrast, uint8_t* out, int32_t* stretched) {
  return guarded([&]() -> int {
    if (!std::isfinite(adjust_contrast) || !(adjust_contrast > 0.f) || adjust_contrast > 1.f) {
      char v[32];
      std::snprintf(v, sizeof v, "%g", adjust_contrast);
      set_error(std::string("tt_contrast_adjust: adjust_contrast is ") + v + "; it must be finite and in (0, 1]");
      return 1;
    }
    if (n < 0 || (n > 0 && (!crops || !out))) { set_error("tt_contrast_adjust: null crops or output, or n < 0"); return 1; }
    if (n == 0) return 0;
    const size_t bytes = static_cast<size_t>(n) * 32 * 128 * 3;
    DevBuf din, dpatch, dflag, dlr, dlist, dcount, dout;
    TT_CUDA_INT(din.alloc(bytes));
    TT_CUDA_INT(dout.alloc(bytes));
    TT_CUDA_INT(dpatch.alloc(static_cast<size_t>(n) * 128 * 96 * sizeof(__nv_bfloat16)));
    TT_CUDA_INT(dflag.alloc(sizeof(int) * n));
    TT_CUDA_INT(dlr.alloc(sizeof(double2) * n));
    TT_CUDA_INT(dlist.alloc(sizeof(int) * n));
    TT_CUDA_INT(dcount.alloc(sizeof(int)));
    TT_CUDA_INT(cudaMemcpy(din.p, crops, bytes, cudaMemcpyHostToDevice));
    TT_CUDA_INT(cudaMemcpy(dout.p, din.p, bytes, cudaMemcpyDeviceToDevice));   // crops that are not stretched stay as given
    const OrientSet upright{1, {0, 0, 0, 0}};
    TT_TRY_INT(patchify_u8(din.as<uint8_t>(), n, dpatch.as<__nv_bfloat16>(), 0));
    TT_TRY_INT(contrast_stats(nullptr, nullptr, n, TT_MAX_LABEL_LEN, 0.f, adjust_contrast, dpatch.as<__nv_bfloat16>(), 1,
                              nullptr, upright, dflag.as<int>(), dlr.as<double2>(), 0));
    TT_TRY_INT(contrast_compact(dflag.as<int>(), n, dlist.as<int>(), dcount.as<int>(), 0));
    int m = 0;
    TT_CUDA_INT(cudaMemcpy(&m, dcount.p, sizeof(int), cudaMemcpyDeviceToHost));
    TT_TRY_INT(contrast_apply(dlist.as<int>(), m, dpatch.as<__nv_bfloat16>(), 1, nullptr, upright, dlr.as<double2>(), nullptr,
                              dout.as<uint8_t>(), nullptr, nullptr, nullptr, nullptr, 0));
    TT_CUDA_INT(cudaMemcpy(out, dout.p, bytes, cudaMemcpyDeviceToHost));
    if (stretched) TT_CUDA_INT(cudaMemcpy(stretched, dflag.p, sizeof(int) * n, cudaMemcpyDeviceToHost));
    return 0;
  });
}

int tt_rect_to_quad(const float rect[5], float quad_out[8]) {
  return guarded([&]() -> int {
    Pt2f q[4];
    rect_to_quad(RotatedRect{rect[0], rect[1], rect[2], rect[3], rect[4]}, q);
    for (int k = 0; k < 4; ++k) { quad_out[2 * k] = q[k].x; quad_out[2 * k + 1] = q[k].y; }
    return 0;
  });
}

int tt_decode(const int32_t* ids, int n, int len, char* out, int out_stride) {
  return guarded([&]() -> int {
    for (int i = 0; i < n; ++i) {
      const std::string s = decode_ids(ids + static_cast<size_t>(i) * len, len);
      if (static_cast<int>(s.size()) + 1 > out_stride) { set_error("tt_decode: out_stride too small"); return 1; }
      std::memcpy(out + static_cast<size_t>(i) * out_stride, s.c_str(), s.size() + 1);
    }
    return 0;
  });
}

int tt_decode_scores(const int32_t* ids, const float* pmax, int n, int len, char* out, int out_stride, float* conf_out,
                     float* char_conf_out) {
  return guarded([&]() -> int {
    std::string s;
    std::vector<float> cc;
    for (int i = 0; i < n; ++i) {
      float conf = 0.f;
      decode_ids_scored(ids + static_cast<size_t>(i) * len, pmax + static_cast<size_t>(i) * len, len, &s, &cc, &conf);
      if (static_cast<int>(s.size()) + 1 > out_stride) { set_error("tt_decode_scores: out_stride too small"); return 1; }
      std::memcpy(out + static_cast<size_t>(i) * out_stride, s.c_str(), s.size() + 1);
      if (conf_out) conf_out[i] = conf;
      if (char_conf_out) {
        float* row = char_conf_out + static_cast<size_t>(i) * len;
        std::fill(row, row + len, 0.f);
        std::copy(cc.begin(), cc.end(), row);
      }
    }
    return 0;
  });
}

int tt_char_filter_mask(const tt_char_filter* f, uint32_t mask_out[4]) {
  if (!f || !mask_out) { set_error("tt_char_filter_mask: null argument"); return 1; }
  char_filter_mask(f->allow, f->block, mask_out);
  return 0;
}

int tt_tokenizer_table(char* itos_out, int* eos_id, int* bos_id, int* pad_id) {
  const TokenizerTable& t = tokenizer_table();
  std::memcpy(itos_out, t.itos.c_str(), t.itos.size() + 1);
  if (eos_id) *eos_id = t.eos_id;
  if (bos_id) *bos_id = t.bos_id;
  if (pad_id) *pad_id = t.pad_id;
  return 0;
}

int tt_convex_hull_i32(const int32_t* xy, int n, int32_t* idx_out, int* n_out) {
  return guarded([&]() -> int {
    const std::vector<int> h = convex_hull_i(reinterpret_cast<const Pt2i*>(xy), n);
    for (size_t i = 0; i < h.size(); ++i) idx_out[i] = h[i];
    *n_out = static_cast<int>(h.size());
    return 0;
  });
}
int tt_convex_hull_f32(const float* xy, int n, int32_t* idx_out, int* n_out) {
  return guarded([&]() -> int {
    const std::vector<int> h = convex_hull_f(reinterpret_cast<const Pt2f*>(xy), n);
    for (size_t i = 0; i < h.size(); ++i) idx_out[i] = h[i];
    *n_out = static_cast<int>(h.size());
    return 0;
  });
}
int tt_min_area_rect_i32(const int32_t* xy, int n, float rect_out[5]) {
  return guarded([&]() -> int { from_rect(min_area_rect_i(reinterpret_cast<const Pt2i*>(xy), n), rect_out); return 0; });
}
int tt_min_area_rect_f32(const float* xy, int n, float rect_out[5]) {
  return guarded([&]() -> int { from_rect(min_area_rect_f(reinterpret_cast<const Pt2f*>(xy), n), rect_out); return 0; });
}
int tt_rect_points(const float rect[5], float pts_out[8]) {
  Pt2f p[4];
  rect_points(to_rect(rect), p);
  for (int i = 0; i < 4; ++i) { pts_out[2 * i] = p[i].x; pts_out[2 * i + 1] = p[i].y; }
  return 0;
}
int tt_rect_bounding(const float rect[5], int32_t o[4]) {
  const RectI r = rect_bounding(to_rect(rect));
  o[0] = r.x; o[1] = r.y; o[2] = r.w; o[3] = r.h;
  return 0;
}
int tt_adjust_rect(const float rect[5], float ratio_w, float ratio_h, float ratio_net, float rect_out[5]) {
  return guarded([&]() -> int { from_rect(adjust_rect(to_rect(rect), ratio_w, ratio_h, ratio_net), rect_out); return 0; });
}
int tt_rect_to_bbox(const float rect[5], float bbox_out[4]) {
  rect_to_bbox(to_rect(rect), bbox_out);
  return 0;
}

int tt_linear_dev(const void* A, int lda, int M, int K, const void* W, int N, const float* bias, int act,
                  const void* residual, int res_f32, int ldr, void* out, int out_f32, int ldc, int BN, int resident,
                  void* stream) {
  return guarded([&]() -> int {
    LinearProblem l;
    l.A = static_cast<const __nv_bfloat16*>(A); l.lda = lda; l.M = M; l.K = K;
    l.W = static_cast<const __nv_bfloat16*>(W); l.N = N; l.BN = BN; l.resident = BN ? (resident & 1) : -1;
    l.pair = BN ? ((resident >> 1) & 1) : ((resident & 4) ? 1 : (resident & 8) ? 0 : -1);
    Epilogue e;
    e.bias = bias; e.act = act;
    e.residual = residual; e.res_type = residual ? (res_f32 ? RES_F32 : RES_BF16) : RES_NONE; e.ldr = ldr;
    e.out = out; e.out_type = out_f32 ? OUT_F32 : OUT_BF16; e.ldc = ldc;
    return linear_forward(l, e, static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : 1;
  });
}

int tt_linear_ln_pair_dev(const void* A, int M, int K1, const void* W1, const float* b1, int D, void* x_hi, void* x_lo,
                          float* stats, const void* W2f, const float* c0, const float* c1, int N2, int act, float eps,
                          void* out, void* stream) {
  return guarded([&]() -> int {
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int parts = 0;
    {  // producer: x += A W1^T + b1 on the split (hi, lo) stream, plus the rows' partial (sum, sum of squares)
      LinearProblem l;
      l.A = static_cast<const __nv_bfloat16*>(A); l.lda = K1; l.M = M; l.K = K1;
      l.W = static_cast<const __nv_bfloat16*>(W1); l.N = D;
      Epilogue e;
      e.bias = b1; e.residual = x_hi; e.residual_lo = x_lo; e.res_type = RES_SPLIT; e.ldr = D;
      e.out = x_hi; e.out_lo = x_lo; e.out_type = OUT_SPLIT; e.ldc = D;
      e.ln_stats_out = stats; e.ln_parts_out = &parts;
      if (linear_forward(l, e, s) != cudaSuccess) return 1;
    }
    {  // consumer: out = act(Linear(LN(x))) from hi = bf16(x), the folded weights and the statistics
      LinearProblem l;
      l.A = static_cast<const __nv_bfloat16*>(x_hi); l.lda = D; l.M = M; l.K = D;
      l.W = static_cast<const __nv_bfloat16*>(W2f); l.N = N2;
      Epilogue e;
      e.bias = c0; e.act = act; e.out = out; e.out_type = OUT_BF16; e.ldc = N2;
      e.ln_stats_in = stats; e.ln_c1 = c1; e.ln_parts = parts; e.ln_dim = D; e.ln_eps = eps;
      if (linear_forward(l, e, s) != cudaSuccess) return 1;
    }
    return 0;
  });
}

int tt_linear_ln_dev(const void* A, int M, int K, const void* Wf, const float* c0, const float* c1, int N, const float* stats,
                     int parts, float eps, void* out, void* stream) {
  return guarded([&]() -> int {
    LinearProblem l;
    l.A = static_cast<const __nv_bfloat16*>(A); l.lda = K; l.M = M; l.K = K;
    l.W = static_cast<const __nv_bfloat16*>(Wf); l.N = N;
    Epilogue e;
    e.bias = c0; e.out = out; e.out_type = OUT_BF16; e.ldc = N;
    e.ln_stats_in = stats; e.ln_c1 = c1; e.ln_parts = parts; e.ln_dim = K; e.ln_eps = eps;
    return linear_forward(l, e, static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : 1;
  });
}

int tt_enc_mlp_dev(void* x_hi, void* x_lo, float* stats, long long M, const void* att, const void* Wp, const float* bp,
                   const void* W1f, const float* c0, const float* c1, const void* W2, const float* b2, float eps, void* stream) {
  return guarded([&]() -> int {
    EncMlpWeights w;
    w.w1 = static_cast<const __nv_bfloat16*>(W1f); w.c0 = c0; w.c1 = c1;
    w.w2 = static_cast<const __nv_bfloat16*>(W2); w.b2 = b2;
    EncProj pj;
    pj.att = static_cast<const __nv_bfloat16*>(att); pj.wp = static_cast<const __nv_bfloat16*>(Wp); pj.bp = bp;
    return enc_mlp_forward(w, static_cast<__nv_bfloat16*>(x_hi), static_cast<__nv_bfloat16*>(x_lo), stats, 2, M, 384, 1536, eps,
                           static_cast<cudaStream_t>(stream), att ? &pj : nullptr) == cudaSuccess ? 0 : 1;
  });
}

int tt_enc_qkv_attn_dev(const void* x_hi, const float* stats, int parts, const void* Wf, const float* c0, const float* c1, void* att,
                        int crops, int D, int heads, float eps, void* stream) {
  return guarded([&]() -> int {
    return enc_qkv_attn_forward(static_cast<const __nv_bfloat16*>(x_hi), stats, parts, static_cast<const __nv_bfloat16*>(Wf), c0, c1,
                                static_cast<__nv_bfloat16*>(att), crops, D, heads, eps, static_cast<cudaStream_t>(stream)) == cudaSuccess
               ? 0 : 1;
  });
}

int tt_conv_dev(const void* src0, int C0, const void* src1, int C1, int batch, int H, int W, int taps, int dil,
                const void* weight, const float* bias, int Cout, int relu, void* out, int BN, int resident,
                void* stream) {
  return guarded([&]() -> int {
    ConvProblem c;
    c.batch = batch; c.H = H; c.W = W;
    c.src[0] = ConvSrc{static_cast<const __nv_bfloat16*>(src0), C0, C0};
    c.nsrc = 1;
    if (src1) { c.src[1] = ConvSrc{static_cast<const __nv_bfloat16*>(src1), C1, C1}; c.nsrc = 2; }
    c.taps = taps; c.dil = dil;
    c.weight = static_cast<const __nv_bfloat16*>(weight); c.Cout = Cout; c.BN = BN; c.resident = BN ? (resident & 1) : -1;
    c.pair = BN ? ((resident >> 1) & 1) : ((resident & 4) ? 1 : (resident & 8) ? 0 : -1);
    Epilogue e;
    e.bias = bias; e.act = relu ? ACT_RELU : ACT_NONE; e.out = out; e.out_type = OUT_BF16; e.ldc = Cout;
    return conv_forward(c, e, static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : 1;
  });
}

int tt_attn_enc_dev(const void* qkv, void* out, int crops, int D, int heads, int onepass, void* stream) {
  return guarded([&]() -> int {
    return attention_enc(static_cast<const __nv_bfloat16*>(qkv), static_cast<__nv_bfloat16*>(out), crops, D, heads,
                         onepass != 0, static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : 1;
  });
}

int tt_dec_score_table_dev(const float* q_table, const void* kv_table, int L, int n_tok, int D, int heads, float* out,
                           void* stream) {
  return guarded([&]() -> int {
    return dec_score_table(q_table, static_cast<const __nv_bfloat16*>(kv_table), L, n_tok, D, heads, out,
                           static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : 1;
  });
}

int tt_dec_self_attn_dev(int n_crops, int D, int heads, int L, int p0, int np, int refine, const int32_t* active,
                         const int32_t* n_act, const float* q_table, const float* sc_table, const void* kv_table,
                         const int32_t* tokens, int eos_id, int n_tok, void* out, void* stream) {
  return guarded([&]() -> int {
    DecoderStep st{n_crops, D, heads, L, p0, np, refine};
    st.active = active; st.n_act = n_act;
    return dec_self_attn(st, q_table, sc_table, static_cast<const __nv_bfloat16*>(kv_table), tokens, eos_id, n_tok,
                         static_cast<__nv_bfloat16*>(out), static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : 1;
  });
}

int tt_orient_select_dev(const int32_t* ids, const float* pmax, int n_words, const int32_t* angles, int n_candidates,
                         int32_t* ids_out, float* pmax_out, int32_t* angle_out, void* stream) {
  return guarded([&]() -> int {
    if (n_candidates < 1 || n_candidates > 4 || !angles) {
      set_error("tt_orient_select_dev: n_candidates must be 1..4 with its angles, got " + std::to_string(n_candidates));
      return 1;
    }
    OrientSet set{n_candidates, {0, 0, 0, 0}};
    for (int r = 0; r < n_candidates; ++r) set.angle[r] = angles[r];
    return orient_select(ids, pmax, n_words, TT_MAX_LABEL_LEN, set, ids_out, pmax_out, angle_out,
                         static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : 1;
  });
}

int tt_contrast_select_dev(int32_t* ids, float* pmax, const int32_t* list, int n_listed, const int32_t* ids2, const float* pmax2,
                           void* stream) {
  return guarded([&]() -> int {
    if (n_listed < 0 || (n_listed > 0 && (!ids || !pmax || !list || !ids2 || !pmax2))) {
      set_error("tt_contrast_select_dev: null argument or n_listed < 0");
      return 1;
    }
    return contrast_select(ids, pmax, TT_MAX_LABEL_LEN, list, n_listed, ids2, pmax2, static_cast<cudaStream_t>(stream)) ==
                   cudaSuccess ? 0 : 1;
  });
}

int tt_lexicon_walk_dev(const tt_lexicon* lex, const float* logits, int n, int32_t* ids_out, float* pmax_out, void* stream) {
  return guarded([&]() -> int {
    if (!lex || !ids_out || n < 0 || (n > 0 && !logits)) { set_error("tt_lexicon_walk_dev: null argument or n < 0"); return 1; }
    if (n == 0) return 0;
    LexTableBuilder table;
    const std::vector<int> roots(n, table.append(lex->trie));
    const std::vector<uint32_t> words = table.words();
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    DevBuf tab, root, state;
    TT_CUDA_INT(tab.alloc(sizeof(uint32_t) * words.size()));
    TT_CUDA_INT(root.alloc(sizeof(int) * n));
    TT_CUDA_INT(state.alloc(sizeof(int) * n));
    TT_CUDA_INT(cudaMemcpyAsync(tab.p, words.data(), sizeof(uint32_t) * words.size(), cudaMemcpyHostToDevice, s));
    TT_CUDA_INT(cudaMemcpyAsync(root.p, roots.data(), sizeof(int) * n, cudaMemcpyHostToDevice, s));
    LexDev lx;
    lx.allow = tab.as<const uint4>();
    lx.first = tab.as<const int>() + 4 * static_cast<size_t>(table.n_states());
    lx.next = lx.first + table.n_states();
    lx.root = root.as<int>();
    lx.state = state.as<int>();
    TT_TRY_INT(lexicon_walk(logits, n, TT_MAX_LABEL_LEN, TT_NUM_CLASSES, TT_NUM_CLASSES, lx, ids_out, pmax_out, s));
    TT_CUDA_INT(cudaStreamSynchronize(s));   // the table and the roots are freed on return
    return 0;
  });
}

int tt_dec_cross_attn_dev(int n_crops, int D, int heads, int L, int p0, int np, const int32_t* active, const int32_t* n_act,
                          const void* q, const void* mem_kv, void* out, void* stream) {
  return guarded([&]() -> int {
    DecoderStep st{n_crops, D, heads, L, p0, np, 0};
    st.active = active; st.n_act = n_act;
    return dec_cross_attn(st, static_cast<const __nv_bfloat16*>(q), static_cast<const __nv_bfloat16*>(mem_kv),
                          static_cast<__nv_bfloat16*>(out), static_cast<cudaStream_t>(stream)) == cudaSuccess ? 0 : 1;
  });
}

}  // extern "C"
