// Page pipeline and the engine half of the C ABI: image_to_data (tuatara.cpp:314-512) for a batch
// of pages, sharded data-parallel over the engine's GPUs (one host worker thread per device, no
// collective: pages are independent), results gathered on the host in page order.
#include "engine.h"

#include <algorithm>
#include <array>
#include <atomic>
#include <map>
#include <tuple>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "common.h"
#include "contrast.cuh"
#include "gemm_tc.cuh"
#include "lexicon.h"
#include "nn_kernels.cuh"
#include "orient.cuh"
#include "resize.cuh"
#include "tokenizer.h"

using namespace tt;

namespace {

constexpr int kCompCap = 2048;   // compact per-page result block: components
constexpr int kRowCap = 32768;   //                                row extents
constexpr int kMaxCropsPerPass = 32768;
constexpr int kCraftSubBatch = 8;   // pages per CRAFT / post-processing pass inside a group

#define E_TRY(expr)                                   \
  do {                                                \
    cudaError_t _e = (expr);                          \
    if (_e != cudaSuccess) return 1;                  \
  } while (0)
#define E_CUDA(expr)                                                               \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) {                                                       \
      set_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e));        \
      return 1;                                                                    \
    }                                                                              \
  } while (0)

struct PageOut {
  std::vector<std::string> text;
  std::vector<std::array<float, 4>> bbox;
  // tt_ocr_options.with_scores only (empty otherwise); definitions at tt_item_scores
  std::vector<float> det;                        // per item: the component's maximum normalised text score
  std::vector<float> conf;                       // per item: word confidence, -1 until recognised
  std::vector<std::vector<float>> char_conf;     // per item: one probability per character of text
  // with rotation candidates only (empty otherwise): per item the winning candidate's angle, -1 until recognised
  std::vector<int> angle;
};

// What tt_ocr_pages_ex returns: the public tt_result first (the caller only ever sees its address), the scores in a
// block of their own so that tt_item / tt_page_result / tt_result keep their layout.
struct ResultBlock {
  tt_result r;
  std::vector<PageOut>* scores;   // null without with_scores; text / bbox already copied into r
  std::vector<std::vector<int>>* angles;   // null without rotation candidates; per page, per item (tt_item_angle)
};

cudaError_t ensure_post(DeviceCtx& d, int batch, int H, int W, int comp_cap, int row_cap) {
  if (d.post.parent && d.post.batch >= batch && d.post.H == H && d.post.W == W && d.post.comp_cap == comp_cap &&
      d.post.row_cap == row_cap)
    return cudaSuccess;
  post_workspace_free(&d.post);
  return post_workspace_alloc(&d.post, batch, H, W, comp_cap, row_cap, false);
}

// Runs post-processing for `batch` maps on the device and returns the boxes per page (host).
int detect_boxes(DeviceCtx& d, const tt_config& cfg, const float* maps_dev, int batch, int H, int W,
                 std::vector<std::vector<DetBox>>* out) {
  int comp_cap = kCompCap, row_cap = kRowCap;
  for (int attempt = 0; attempt < 2; ++attempt) {
    E_TRY(ensure_post(d, batch, H, W, comp_cap, row_cap));
    PostWorkspace ws = d.post;
    ws.batch = batch;
    PostParams pp;
    pp.low_text = cfg.low_text;
    pp.link_threshold = cfg.link_threshold;
    const size_t bytes = ws.result_stride * batch;
    E_TRY(d.ensure_pinned(bytes));
    stage_begin(d.stream);
    E_TRY(post_run(ws, maps_dev, pp, d.stream));
    E_CUDA(cudaMemcpyAsync(d.pinned, ws.result, bytes, cudaMemcpyDeviceToHost, d.stream));
    stage_end(d.stream, "postprocess", 0.0, 24.0 * batch * H * W);  // 24 B per map pixel (SURVEY 8d); kernels + the result D2H
    E_TRY(stream_sync(d.stream));
    g_d2h_bytes += bytes;
    out->assign(batch, {});
    bool ok = true;
    for (int b = 0; b < batch && ok; ++b)
      ok = collect_boxes(d.pinned + b * ws.result_stride, comp_cap, row_cap, H, W, cfg, &(*out)[b]);
    if (ok) return 0;
    comp_cap = H * W / 2 + 2;  // pathological map: worst-case capacities
    row_cap = H * W;
  }
  set_error("post-process: capacity overflow");
  return 1;
}

// ---------------------------------------------------------------------------------------------------------------
// Scheduling (SURVEY 8e).  A request is cut into DETECTION UNITS: up to kCraftSubBatch pages of one size (pages of equal
// size are bucketed wherever they sit in the request).  Units go into work queues that the execution slots of all GPUs
// drain with an atomic counter: words per page vary, so static page -> GPU assignment would leave GPUs idle.  A slot
//   1. runs a unit: upload, resize, CRAFT, post-processing, one small D2H, host geometry, then the crop kernel, which
//      appends the unit's crops (bf16 patch rows) to the slot's RECOGNITION BATCH -- pages of any size mix there;
//   2. runs PARSeq over the batch once it holds `max_batch_pages` pages' worth of crops (or the queues are empty):
//      the decoder's 27 passes are latency bound, their cost per crop falls with the batch.
// Two slots per GPU by default: one slot's host phases (geometry, result assembly, D2H waits) are covered by the other
// slot's kernels.
struct Unit {
  std::vector<int> pages;   // indices into the request, all of one size
};

struct CropOwner { int page, box; };

// What a request asks for besides its pages, checked by make_request; every tt_ocr_pages* entry point builds one.
struct Request {
  tt_ocr_options opt{0, 0, nullptr, 0, 0};   // zeroed when the caller passes none
  std::vector<ClassMask> masks;              // one class mask per page; empty when no page has a filter
  OrientSet orient{1, {0, 0, 0, 0}};         // the rotation candidates; n == 1 (angle 0 alone) without
  // lexicon requests only (both empty otherwise; masks is then empty too, the filters being folded into the automata):
  std::vector<int> roots;                    // the root state of every page's automaton
  std::vector<uint32_t> lex_table;           // the request's automata, LexTableBuilder::words()
  int lex_states = 0;                        //   its number of states
  float contrast_ths = 0.f;                  // the contrast re-read (INTEGRATION.md section 10); 0 = off
  float adjust_contrast = 0.5f;
};

// The request's automaton table in the slot's lex_buf, uploaded at most once per slot per request; -> its device view.
int upload_lex_table(DeviceCtx& d, const std::vector<uint32_t>& table, int n_states, LexDev* lx) {
  const size_t bytes = sizeof(uint32_t) * table.size();
  if (bytes > d.lex_cap) {
    if (d.lex_buf) {
      E_TRY(stream_sync(d.stream));
      cudaFree(d.lex_buf);
      d.lex_buf = nullptr;
      d.lex_cap = 0;
    }
    E_CUDA(cudaMalloc(&d.lex_buf, bytes));
    d.lex_cap = bytes;
  }
  stage_begin(d.stream);
  E_CUDA(cudaMemcpyAsync(d.lex_buf, table.data(), bytes, cudaMemcpyHostToDevice, d.stream));
  stage_end(d.stream, "lexicon_table", 0.0, static_cast<double>(bytes));
  g_h2d_bytes += bytes;
  const uint32_t* base = static_cast<const uint32_t*>(d.lex_buf);   // allow [S][4] | first [S] | next [E]
  lx->allow = reinterpret_cast<const uint4*>(base);
  lx->first = reinterpret_cast<const int*>(base + 4 * static_cast<size_t>(n_states));
  lx->next = lx->first + n_states;
  return 0;
}

// crops waiting for recognition in one slot (device patch rows live in DeviceCtx::patch_buf)
struct Pending {
  std::vector<CropOwner> owner;
  int pages = 0;
};

cudaError_t ensure_patch_buf(DeviceCtx& d, size_t crops, size_t keep_crops) {
  if (crops <= d.patch_cap) return cudaSuccess;
  size_t cap = std::max<size_t>(crops + crops / 2, 4096);
  __nv_bfloat16* nb = nullptr;
  TT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&nb), cap * 128 * 96 * sizeof(__nv_bfloat16)));
  if (d.patch_buf && keep_crops)
    TT_CUDA_TRY(cudaMemcpyAsync(nb, d.patch_buf, keep_crops * 128 * 96 * sizeof(__nv_bfloat16), cudaMemcpyDeviceToDevice, d.stream));
  if (d.patch_buf) {
    TT_CUDA_TRY(stream_sync(d.stream));
    cudaFree(d.patch_buf);
  }
  d.patch_buf = nb;
  d.patch_cap = cap;
  return cudaSuccess;
}

// Detection + cropping of one unit (tuatara.cpp:349-418, :437-441).  Fills bbox of every page of the unit, sizes its
// text vector, appends the crops to the slot's recognition batch.  Every word gets R = req.orient.n crops, candidate r
// turned req.orient.angle[r] degrees counter-clockwise, stored word-major (crop = word * R + r).
int detect_unit(DeviceCtx& d, const tt_config& cfg, const tt_image* pages, const Unit& u, const Request& req,
                std::vector<PageOut>* results, Pending* pend) {
  const tt_ocr_options& opt = req.opt;
  const cudaMemcpyKind page_kind = opt.pages_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  const int nb = static_cast<int>(u.pages.size());
  const tt_image& first = pages[u.pages[0]];
  int th, tw, h32, w32;
  float ratio;
  resize_plan(first.rows, first.cols, cfg.canvas_size, cfg.mag_ratio, &th, &tw, &h32, &w32, &ratio);
  const size_t page_bytes = static_cast<size_t>(first.rows) * first.cols * 3;
  const size_t in_bytes = static_cast<size_t>(h32) * w32 * 3;
  const size_t page_stride = (page_bytes + 255) & ~size_t(255);
  const size_t need = d.craft_bytes(nb, h32, w32) + nb * (page_stride + 4096 + in_bytes) + (8u << 20);
  if (need > d.arena.capacity()) E_TRY(stream_sync(d.stream));   // growing frees the old block: nothing may still use it
  E_TRY(d.arena.reserve(need));
  d.arena.reset();
  uint8_t* pages_dev = d.arena.get<uint8_t>(nb * page_stride);
  uint8_t* craft_in = d.arena.get<uint8_t>(nb * in_bytes);
  if (!pages_dev || !craft_in) { set_error("arena exhausted (pages)"); return 1; }
  std::vector<PageRef> refs(nb);
  stage_begin(d.stream);
  for (int b = 0; b < nb; ++b) {
    const tt_image& im = pages[u.pages[b]];
    uint8_t* dst = pages_dev + b * page_stride;
    if (opt.pages_on_device) {
      refs[b] = PageRef{im.data, im.rows, im.cols, im.step};  // already resident: read in place
    } else {
      E_CUDA(cudaMemcpy2DAsync(dst, static_cast<size_t>(im.cols) * 3, im.data, im.step, static_cast<size_t>(im.cols) * 3, im.rows,
                               page_kind, d.stream));
      g_h2d_bytes += page_bytes;
      refs[b] = PageRef{dst, im.rows, im.cols, static_cast<size_t>(im.cols) * 3};
    }
    E_TRY(page_resize_pad(refs[b].data, im.rows, im.cols, refs[b].step, craft_in + b * in_bytes, th, tw, h32, w32, d.stream));
  }
  stage_end(d.stream, "preprocess", 0.0, static_cast<double>(nb) * (page_bytes + in_bytes));
  float* maps = nullptr;
  stage_begin(d.stream);
  E_TRY(d.craft_forward(craft_in, nb, h32, w32, &maps));
  // 27 convolutions of CRAFT: 711.4 FLOP per input pixel (= 746.0 GFLOP at 1024 x 1024, SURVEY 8d)
  stage_end(d.stream, "craft", 746.0e9 / (1024.0 * 1024.0) * nb * h32 * w32, 0.0);
  if (opt.score_override) {
    const size_t map_elems = static_cast<size_t>(h32 / 2) * (w32 / 2) * 2;
    for (int b = 0; b < nb; ++b)
      if (opt.score_override[u.pages[b]]) {
        E_CUDA(cudaMemcpyAsync(maps + b * map_elems, opt.score_override[u.pages[b]], map_elems * sizeof(float),
                               opt.override_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, d.stream));
        if (!opt.override_on_device) g_h2d_bytes += map_elems * sizeof(float);
      }
  }
  std::vector<std::vector<DetBox>> det;
  if (detect_boxes(d, cfg, maps, nb, h32 / 2, w32 / 2, &det)) return 1;

  // host: rescale boxes, bounding rects, output bboxes (tuatara.cpp:406-418, :256-274)
  const float inv = 1.f / ratio;  // ratio_w == ratio_h (tuatara.cpp:360-361)
  std::vector<CropBox> crops;
  std::vector<WarpBox> warps;   // cfg.rectify: one perspective warp per box instead of the axis-aligned crop
  const bool rectify = cfg.rectify != 0;
  const int R = req.orient.n;
  for (int b = 0; b < nb; ++b) {
    PageOut& po = (*results)[u.pages[b]];
    const tt_image& im = pages[u.pages[b]];
    int k = 0;
    for (const DetBox& db : det[b]) {
      const RotatedRect adj = adjust_rect(db.rect, inv, inv, 2.f);
      std::array<float, 4> bb;
      rect_to_bbox(adj, bb.data());
      po.bbox.push_back(bb);
      if (opt.with_scores) po.det.push_back(db.score);
      const RectI r = rect_bounding(adj);  // the reference throws when this leaves the image; we clamp
      const int x0 = std::max(r.x, 0), y0 = std::max(r.y, 0);
      const int x1 = std::min(r.x + r.w, im.cols), y1 = std::min(r.y + r.h, im.rows);
      crops.push_back(CropBox{b, x0, y0, std::max(x1 - x0, 0), std::max(y1 - y0, 0)});
      if (rectify) {
        Pt2f quad[4];
        rect_to_quad(adj, quad);
        for (int r = 0; r < R; ++r) {   // candidate angle a: the corners shifted cyclically by a / 90
          const int sh = req.orient.angle[r] / 90;
          const Pt2f q[4] = {quad[sh & 3], quad[(sh + 1) & 3], quad[(sh + 2) & 3], quad[(sh + 3) & 3]};
          WarpBox wb{};
          wb.page = quad_to_warp(q, wb.m) ? b : -1;
          warps.push_back(wb);
        }
      }
      pend->owner.push_back(CropOwner{u.pages[b], k++});
    }
    po.text.resize(po.bbox.size());   // zero boxes: the reference crashes in torch::cat({}) (tuatara.cpp:485); we return no items
    if (opt.with_scores) {
      po.conf.assign(po.bbox.size(), -1.f);
      po.char_conf.resize(po.bbox.size());
    }
    if (R > 1) po.angle.assign(po.bbox.size(), -1);
  }
  const int n = static_cast<int>(crops.size());
  if (opt.detect_only) {   // boxes only: nothing joins the recognition batch
    pend->owner.resize(pend->owner.size() - n);
    return 0;
  }
  pend->pages += nb;
  if (n == 0) return 0;
  const size_t have = (pend->owner.size() - n) * R;   // crops already in the batch
  const int nc = n * R;
  E_TRY(ensure_patch_buf(d, have + nc, have));
  PageRef* refs_dev = d.arena.get<PageRef>(nb);
  CropBox* boxes_dev = d.arena.get<CropBox>(n);
  if (!refs_dev || !boxes_dev) { set_error("arena exhausted (crops)"); return 1; }
  E_CUDA(cudaMemcpyAsync(refs_dev, refs.data(), sizeof(PageRef) * nb, cudaMemcpyHostToDevice, d.stream));
  E_CUDA(cudaMemcpyAsync(boxes_dev, crops.data(), sizeof(CropBox) * n, cudaMemcpyHostToDevice, d.stream));
  g_h2d_bytes += sizeof(PageRef) * nb + sizeof(CropBox) * n;
  stage_begin(d.stream);
  if (rectify) {
    WarpBox* warps_dev = d.arena.get<WarpBox>(nc);
    if (!warps_dev) { set_error("arena exhausted (warps)"); return 1; }
    E_CUDA(cudaMemcpyAsync(warps_dev, warps.data(), sizeof(WarpBox) * nc, cudaMemcpyHostToDevice, d.stream));
    g_h2d_bytes += sizeof(WarpBox) * nc;
    E_TRY(crop_warp(refs_dev, warps_dev, nc, nullptr, d.patch_buf + have * 128 * 96, d.stream));
  } else if (R > 1) {
    std::vector<uint8_t> rot(nc);
    for (int c = 0; c < nc; ++c) rot[c] = static_cast<uint8_t>(req.orient.angle[c % R] / 90);
    uint8_t* rot_dev = d.arena.get<uint8_t>(nc);
    if (!rot_dev) { set_error("arena exhausted (rotations)"); return 1; }
    E_CUDA(cudaMemcpyAsync(rot_dev, rot.data(), nc, cudaMemcpyHostToDevice, d.stream));
    g_h2d_bytes += nc;
    E_TRY(crop_resize_rot(refs_dev, boxes_dev, rot_dev, R, nc, nullptr, d.patch_buf + have * 128 * 96, d.stream));
  } else {
    E_TRY(crop_resize(refs_dev, boxes_dev, n, nullptr, d.patch_buf + have * 128 * 96, d.stream));
  }
  double src = 0;
  for (const CropBox& c : crops) src += 3.0 * c.w * c.h;
  stage_end(d.stream, "crop_resize", 0.0, src + static_cast<double>(nc) * 128 * 96 * 2);  // source rect + bf16 patch rows
  return 0;
}

// The contrast re-read's per-pass buffers in the arena, below the first read's end (so the second forward leaves them).
struct ContrastBufs {
  int* ids = nullptr;           // R == 1: the first read's ids [nw][L] (with R > 1 orient_select's output is kept)
  int* flag = nullptr;          // [nw]
  double2* lr = nullptr;        // [nw] (low, ratio)
  int* list = nullptr;          // [nw] the words read again
  int* count = nullptr;         //   their number
  __nv_bfloat16* patches = nullptr;   // [nw * 128][96] their stretched crops
  float* p2 = nullptr;          // [nw][L] the second read's pmax
  uint32_t* mask = nullptr;     // [nw][4] with filters
  int* root = nullptr;          // [nw] with lexicons, and as many walk states
  int* state = nullptr;
  int get(Arena& a, int nw, int L, bool own_ids, bool masked, bool lexed) {
    const size_t n = static_cast<size_t>(nw);
    if (own_ids) ids = a.get<int>(n * L);
    flag = a.get<int>(n);
    lr = a.get<double2>(n);
    list = a.get<int>(n);
    count = a.get<int>(1);
    patches = a.get<__nv_bfloat16>(n * 128 * 96);
    p2 = a.get<float>(n * L);
    if (masked) mask = a.get<uint32_t>(4 * n);
    if (lexed) {
      root = a.get<int>(n);
      state = a.get<int>(n);
    }
    if ((own_ids && !ids) || !flag || !lr || !list || !count || !patches || !p2 || (masked && !mask) ||
        (lexed && (!root || !state))) {
      set_error("arena exhausted (contrast)");
      return 1;
    }
    return 0;
  }
};

// The contrast re-read of one pass (INTEGRATION.md section 10): ids / pmax [nw][L] hold the first read of every word (the
// winner of its candidates; angle [nw] its angle, null without rotation candidates) and end up holding the kept read.
// mask / lex: the first forward's per-crop class masks or lexicon roots (null without).
int reread_contrast(DeviceCtx& d, const Request& req, const __nv_bfloat16* patches, int nw, const int* angle,
                    const uint32_t* mask, const LexDev* lex, const ContrastBufs& cb, size_t first_read_end, int* ids,
                    float* pmax) {
  const int L = d.w->pd.L, R = req.orient.n;
  stage_begin(d.stream);
  E_TRY(contrast_stats(ids, pmax, nw, L, req.contrast_ths, req.adjust_contrast, patches, R, angle, req.orient, cb.flag, cb.lr,
                       d.stream));
  E_TRY(contrast_compact(cb.flag, nw, cb.list, cb.count, d.stream));
  E_CUDA(cudaMemcpyAsync(d.pinned, cb.count, sizeof(int), cudaMemcpyDeviceToHost, d.stream));
  stage_end(d.stream, "contrast_stats", 0.0, static_cast<double>(nw) * (L * 8 + 16));
  g_d2h_bytes += sizeof(int);
  E_TRY(stream_sync(d.stream));
  const int m = *reinterpret_cast<const int*>(d.pinned);
  if (m == 0) return 0;
  stage_begin(d.stream);
  E_TRY(contrast_apply(cb.list, m, patches, R, angle, req.orient, cb.lr, cb.patches, nullptr, mask, cb.mask,
                       lex ? lex->root : nullptr, cb.root, d.stream));
  stage_end(d.stream, "contrast_apply", 0.0, static_cast<double>(m) * 128 * 96 * 4);
  d.arena.reset_to(first_read_end);
  LexDev lx2{};
  if (lex) {
    lx2 = *lex;
    lx2.root = cb.root;
    lx2.state = cb.state;
  }
  float* logits = nullptr;
  int* ids2 = nullptr;
  E_TRY(d.parseq_forward(cb.patches, m, nullptr, &logits, &ids2, cb.p2, mask ? cb.mask : nullptr, lex ? &lx2 : nullptr));
  stage_begin(d.stream);
  E_TRY(contrast_select(ids, pmax, L, cb.list, m, ids2, cb.p2, d.stream));
  stage_end(d.stream, "contrast_select", 0.0, static_cast<double>(m) * L * 16);
  return 0;
}

// PARSeq + tokenizer over the slot's recognition batch (tuatara.cpp:450-505), which holds R = req.orient.n crops per
// word.  A pass takes whole words (at most kMaxCropsPerPass crops).  With scores the refinement head also writes each
// position's largest softmax probability, copied back next to the ids and decoded into conf / char_conf.  With
// rotation candidates (R > 1) it always writes them, and orient_select leaves one candidate per word on the device, so
// the copy back is the same ids (and pmax with scores) per word plus its 4-byte angle.  With filters (req.masks) each
// crop decodes under its page's class mask, uploaded per pass as [nc][4] words.  With lexicons (req.roots) each crop
// walks its page's automaton instead: the table goes to the slot once per request (*lex_ready), the crops' roots with
// each pass as [nc] words.  With the contrast re-read (req.contrast_ths > 0) the refinement head always writes pmax, and
// after the first read (and orient_select) the contrast kernels pick the low-confidence, low-contrast words on the device;
// the host reads their 4-byte count, runs PARSeq once more on their stretched crops, and contrast_select leaves the more
// confident read in the per-word ids / pmax, which then go back as without it.
int recognise(DeviceCtx& d, std::vector<PageOut>* results, Pending* pend, const Request& req, bool* lex_ready) {
  const int n = static_cast<int>(pend->owner.size());
  const bool lexed = !req.roots.empty();
  LexDev lx{};
  if (lexed && n > 0 && !*lex_ready) {
    if (upload_lex_table(d, req.lex_table, req.lex_states, &d.lex_view)) return 1;
    *lex_ready = true;
  }
  if (lexed) lx = d.lex_view;
  const int L = d.w->pd.L, R = req.orient.n;
  const bool scores = req.opt.with_scores != 0;
  const bool contrast = req.contrast_ths > 0.f;
  const int words_per_pass = kMaxCropsPerPass / R;
  for (int w0 = 0; w0 < n; w0 += words_per_pass) {
    const int nw = std::min(words_per_pass, n - w0);
    const int nc = nw * R;
    const size_t bytes = sizeof(int) * static_cast<size_t>(nw) * L;   // ids per word; with scores as many bytes of pmax
    const size_t angle_bytes = R > 1 ? sizeof(int) * static_cast<size_t>(nw) : 0;
    const size_t pmax_bytes = scores || R > 1 || contrast ? sizeof(float) * static_cast<size_t>(nc) * L : 0;
    const size_t mask_bytes = req.masks.empty() ? 0 : sizeof(ClassMask) * nc;
    const size_t root_bytes = lexed ? sizeof(int) * static_cast<size_t>(nc) : 0;   // and as many for the walk state
    // contrast: the first read's ids (R == 1), flag, (low, ratio), list, count, the second batch's patch rows, its pmax,
    // class masks and roots / walk states -- at most nw words, so the second forward fits in parseq_bytes(nc)
    const size_t contrast_bytes =
        contrast ? (R == 1 ? bytes : 0) + static_cast<size_t>(nw) * (4 + 16 + 4 + 128 * 96 * 2 + 4 * L) + 4 +
                       (req.masks.empty() ? 0 : sizeof(ClassMask) * nw) + (lexed ? 8 * static_cast<size_t>(nw) : 0)
                 : 0;
    const size_t need = d.parseq_bytes(nc) + (4u << 20) + pmax_bytes + (R > 1 ? 2 * bytes + angle_bytes : 0) + mask_bytes +
                        2 * root_bytes + contrast_bytes;
    if (need > d.arena.capacity()) E_TRY(stream_sync(d.stream));
    E_TRY(d.arena.reserve(need));
    d.arena.reset();
    float* pmax = pmax_bytes ? d.arena.get<float>(static_cast<size_t>(nc) * L) : nullptr;
    if (pmax_bytes && !pmax) { set_error("arena exhausted (pmax)"); return 1; }
    int* win_ids = nullptr;   // R > 1: the winning candidate of every word
    float* win_p = nullptr;
    int* win_angle = nullptr;
    if (R > 1) {
      win_ids = d.arena.get<int>(static_cast<size_t>(nw) * L);
      win_p = d.arena.get<float>(static_cast<size_t>(nw) * L);
      win_angle = d.arena.get<int>(nw);
      if (!win_ids || !win_p || !win_angle) { set_error("arena exhausted (orientation)"); return 1; }
    }
    // pinned staging: ids | angle | pmax on the way back, the class masks or the roots on the way in
    E_TRY(d.ensure_pinned(std::max((scores ? 2 * bytes : bytes) + angle_bytes, std::max(mask_bytes, root_bytes))));
    uint32_t* mask = nullptr;
    if (!req.masks.empty()) {
      mask = d.arena.get<uint32_t>(4 * static_cast<size_t>(nc));
      if (!mask) { set_error("arena exhausted (class masks)"); return 1; }
      ClassMask* host_mask = reinterpret_cast<ClassMask*>(d.pinned);   // the ids' D2H below is ordered after this copy
      for (int c = 0; c < nc; ++c) host_mask[c] = req.masks[pend->owner[w0 + c / R].page];
      E_CUDA(cudaMemcpyAsync(mask, host_mask, mask_bytes, cudaMemcpyHostToDevice, d.stream));
      g_h2d_bytes += mask_bytes;
    }
    if (lexed) {
      int* roots = d.arena.get<int>(nc);
      lx.state = d.arena.get<int>(nc);
      if (!roots || !lx.state) { set_error("arena exhausted (lexicon roots)"); return 1; }
      int* host_roots = reinterpret_cast<int*>(d.pinned);   // the ids' D2H below is ordered after this copy
      for (int c = 0; c < nc; ++c) host_roots[c] = req.roots[pend->owner[w0 + c / R].page];
      E_CUDA(cudaMemcpyAsync(roots, host_roots, root_bytes, cudaMemcpyHostToDevice, d.stream));
      g_h2d_bytes += root_bytes;
      lx.root = roots;
    }
    ContrastBufs cb{};
    if (contrast && cb.get(d.arena, nw, L, R == 1, !req.masks.empty(), lexed)) return 1;
    const size_t first_read_end = d.arena.offset();   // the second forward reuses the arena from here
    const __nv_bfloat16* patches = d.patch_buf + static_cast<size_t>(w0) * R * 128 * 96;
    float* logits = nullptr;
    int* ids = nullptr;
    E_TRY(d.parseq_forward(patches, nc, nullptr, &logits, &ids, pmax, mask, lexed ? &lx : nullptr));
    if (R > 1) {
      stage_begin(d.stream);
      E_TRY(orient_select(ids, pmax, nw, L, req.orient, win_ids, scores || contrast ? win_p : nullptr, win_angle, d.stream));
      stage_end(d.stream, "orient_select", 0.0, static_cast<double>(nc) * L * 8 + static_cast<double>(nw) * (L * 8 + 4));
      ids = win_ids;
      pmax = win_p;
    }
    if (contrast) {
      if (R == 1) {   // the first read's ids live in the forward's arena space, which the second forward reuses
        E_CUDA(cudaMemcpyAsync(cb.ids, ids, bytes, cudaMemcpyDeviceToDevice, d.stream));
        ids = cb.ids;
      }
      if (reread_contrast(d, req, patches, nw, R > 1 ? win_angle : nullptr, mask, lexed ? &lx : nullptr, cb,
                          first_read_end, ids, pmax))
        return 1;
    }
    E_CUDA(cudaMemcpyAsync(d.pinned, ids, bytes, cudaMemcpyDeviceToHost, d.stream));
    if (R > 1) E_CUDA(cudaMemcpyAsync(d.pinned + bytes, win_angle, angle_bytes, cudaMemcpyDeviceToHost, d.stream));
    g_d2h_bytes += bytes + angle_bytes;
    if (scores) {
      E_CUDA(cudaMemcpyAsync(d.pinned + bytes + angle_bytes, pmax, bytes, cudaMemcpyDeviceToHost, d.stream));
      g_d2h_bytes += bytes;
    }
    E_TRY(stream_sync(d.stream));
    const int* host_ids = reinterpret_cast<const int*>(d.pinned);
    const int* host_angle = reinterpret_cast<const int*>(d.pinned + bytes);
    const float* host_p = reinterpret_cast<const float*>(d.pinned + bytes + angle_bytes);
    for (int w = 0; w < nw; ++w) {   // tokenizer (tuatara.cpp:492-505)
      const CropOwner& o = pend->owner[w0 + w];
      PageOut& po = (*results)[o.page];
      if (scores)
        decode_ids_scored(host_ids + static_cast<size_t>(w) * L, host_p + static_cast<size_t>(w) * L, L, &po.text[o.box],
                          &po.char_conf[o.box], &po.conf[o.box]);
      else
        po.text[o.box] = decode_ids(host_ids + static_cast<size_t>(w) * L, L);
      if (R > 1) po.angle[o.box] = host_angle[w];
    }
  }
  pend->owner.clear();
  pend->pages = 0;
  return 0;
}

struct WorkQueues {
  std::vector<Unit> units;
  std::vector<std::vector<int>> per_dev;   // unit indices bound to a device (pages resident there)
  std::vector<int> shared;                 // unit indices any device may take (host pages)
  std::vector<std::atomic<int>> next_dev;
  std::atomic<int> next_shared{0};
  explicit WorkQueues(int G) : per_dev(G), next_dev(G) { for (auto& a : next_dev) a.store(0); }
  // next unit for a slot of device g, or -1
  int pop(int g) {
    const int i = next_dev[g].fetch_add(1);
    if (i < static_cast<int>(per_dev[g].size())) return per_dev[g][i];
    const int j = next_shared.fetch_add(1);
    if (j < static_cast<int>(shared.size())) return shared[j];
    return -1;
  }
};

// One execution slot draining the queues.
void slot_worker(tt_engine& e, int g, int sidx, int want, const tt_image* pages, const Request& req, WorkQueues* q,
                 std::vector<PageOut>* results, int* rc, std::string* err) {
  // take an idle slot of this GPU if there is one (concurrent callers spread over the slots), else queue on our own
  DeviceCtx* dp = nullptr;
  for (int k = 0; k < want && dp == nullptr; ++k) {
    DeviceCtx& c = *e.devs[g * kSlotsPerDevice + (sidx + k) % want];
    if (c.mu.try_lock()) dp = &c;
  }
  if (dp == nullptr) {
    dp = e.devs[g * kSlotsPerDevice + sidx].get();
    dp->mu.lock();
  }
  DeviceCtx& d = *dp;
  std::lock_guard<std::mutex> lock(d.mu, std::adopt_lock);
  bool lex_ready = false;   // this request's automaton table is in the slot's lex_buf
  if (cudaSetDevice(d.device) != cudaSuccess) { *err = "cudaSetDevice failed"; *rc = 1; return; }
  const tt_config& cfg = e.cfg;
  const int max_b = cfg.max_batch_pages > 0 ? cfg.max_batch_pages : 32;
  Pending pend;
  for (int ui = q->pop(g); ui >= 0; ui = q->pop(g)) {
    if (detect_unit(d, cfg, pages, q->units[ui], req, results, &pend)) { *err = last_error(); *rc = 1; return; }
    if (pend.pages >= max_b && recognise(d, results, &pend, req, &lex_ready)) { *err = last_error(); *rc = 1; return; }
  }
  if (recognise(d, results, &pend, req, &lex_ready)) { *err = last_error(); *rc = 1; return; }
}

// The last check of make_request: the contrast re-read's two values.
int set_contrast(const char* fn, float contrast_ths, float adjust_contrast, Request* req) {
  char v[32];
  if (!std::isfinite(contrast_ths) || contrast_ths < 0.f) {
    std::snprintf(v, sizeof v, "%g", contrast_ths);
    set_error(std::string(fn) + ": contrast_ths is " + v + "; it must be finite and >= 0");
    return 1;
  }
  if (!std::isfinite(adjust_contrast) || !(adjust_contrast > 0.f) || adjust_contrast > 1.f) {
    std::snprintf(v, sizeof v, "%g", adjust_contrast);
    set_error(std::string(fn) + ": adjust_contrast is " + v + "; it must be finite and in (0, 1]");
    return 1;
  }
  req->contrast_ths = contrast_ths;
  req->adjust_contrast = adjust_contrast;
  return 0;
}

// The argument checks of the tt_ocr_pages* entry points (fn: the one called, named in the messages), made before any
// device work: the rotation candidates, then the filters, turned into one class mask per page, then the lexicons, turned
// into one automaton per page with the page's filter folded in, then the contrast values.  ocr_pages checks the engine
// and the pages.
int make_request(const char* fn, const tt_ocr_options* opt, const tt_char_filter* filters, int n_filters,
                 const int* rotation_info, int n_rotations, const tt_lexicon* const* lexicons, int n_lexicons,
                 float contrast_ths, float adjust_contrast, int n_pages, Request* req) {
  try {
    if (opt) req->opt = *opt;
    if (n_rotations < 0 || (n_rotations > 0 && !rotation_info)) {
      set_error(std::string(fn) + ": rotation_info is NULL or n_rotations (" + std::to_string(n_rotations) + ") is negative");
      return 1;
    }
    bool seen[4] = {true, false, false, false};
    for (int i = 0; i < n_rotations; ++i) {
      const int a = rotation_info[i];
      if (a != 90 && a != 180 && a != 270) {
        set_error(std::string(fn) + ": rotation_info holds " + std::to_string(a) + "; the angles are 90, 180 and 270");
        return 1;
      }
      if (seen[a / 90]) { set_error(std::string(fn) + ": rotation_info holds " + std::to_string(a) + " twice"); return 1; }
      seen[a / 90] = true;
    }
    req->orient.n = 0;
    for (int q = 0; q < 4; ++q)
      if (seen[q]) req->orient.angle[req->orient.n++] = 90 * q;
    if (n_filters != 0) {
      if (!filters) { set_error(std::string(fn) + ": filters is NULL but n_filters is " + std::to_string(n_filters)); return 1; }
      if (n_filters != 1 && n_filters != n_pages) {
        set_error(std::string(fn) + ": n_filters must be 0, 1 or n_pages (" + std::to_string(n_pages) + "), got " +
                  std::to_string(n_filters));
        return 1;
      }
      req->masks.resize(std::max(n_pages, 0));
      for (int i = 0; i < n_pages; ++i) {
        const tt_char_filter& f = filters[n_filters == 1 ? 0 : i];
        char_filter_mask(f.allow, f.block, req->masks[i].data());
      }
    }
    if (n_lexicons == 0) return set_contrast(fn, contrast_ths, adjust_contrast, req);
    if (!lexicons) { set_error(std::string(fn) + ": lexicons is NULL but n_lexicons is " + std::to_string(n_lexicons)); return 1; }
    if (n_lexicons != 1 && n_lexicons != n_pages) {
      set_error(std::string(fn) + ": n_lexicons must be 0, 1 or n_pages (" + std::to_string(n_pages) + "), got " +
                std::to_string(n_lexicons));
      return 1;
    }
    // one automaton per distinct (lexicon, class mask) of the request: the lexicon's own trie when the page's filter
    // allows all its words, else a trie over the words it allows; a one-state automaton for a NULL entry
    ClassMask all;
    char_filter_mask(nullptr, nullptr, all.data());
    LexTableBuilder table;
    std::map<std::pair<const tt_lexicon*, ClassMask>, int> built;
    req->roots.resize(std::max(n_pages, 0));
    for (int i = 0; i < n_pages; ++i) {
      const tt_lexicon* lex = lexicons[n_lexicons == 1 ? 0 : i];
      const ClassMask& m = req->masks.empty() ? all : req->masks[i];
      const auto key = std::make_pair(lex, m);
      auto it = built.find(key);
      if (it == built.end()) {
        int root;
        if (!lex) {
          root = table.append(one_state(m));
        } else {
          std::vector<std::string> kept;
          for (const std::string& w : lex->words)
            if (word_allowed(w, m)) kept.push_back(w);
          if (kept.empty()) {
            set_error(std::string(fn) + ": page " + std::to_string(i) + ": its filter allows none of its lexicon's " +
                      std::to_string(lex->words.size()) + " words");
            return 1;
          }
          root = table.append(kept.size() == lex->words.size() ? lex->trie : build_trie(kept));
        }
        it = built.emplace(key, root).first;
      }
      req->roots[i] = it->second;
    }
    req->lex_table = table.words();
    req->lex_states = table.n_states();
    req->masks.clear();
    return set_contrast(fn, contrast_ths, adjust_contrast, req);
  } catch (const std::exception& ex) {
    set_error(std::string(fn) + ": " + ex.what());
    return 1;
  }
}

int ocr_pages(tt_engine* e, const tt_image* pages, int n_pages, const Request& req, tt_result** out);

}  // namespace

extern "C" {

int tt_engine_create(const char* weights_dir, const int* devices, int n_devices, const tt_config* cfg,
                     tt_engine** out) {
  try {
    if (!weights_dir || !*weights_dir) { set_error("Please provide a value for weights_dir"); return 1; }
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
      set_error("no CUDA device: this library has no CPU fallback");
      return 1;
    }
    std::unique_ptr<tt_engine> e(new tt_engine);
    if (cfg) e->cfg = *cfg; else tt_config_default(&e->cfg);
    e->slots.store(e->cfg.slots_per_gpu);
    std::vector<int> devs;
    if (devices && n_devices > 0) {
      devs.assign(devices, devices + n_devices);
    } else if (const char* ev = std::getenv("TT_DEVICES")) {   // "all" or a comma-separated list
      if (std::strcmp(ev, "all") == 0) {
        for (int i = 0; i < count; ++i) devs.push_back(i);
      } else {
        for (const char* p = ev; *p;) {
          char* end = nullptr;
          const long v = std::strtol(p, &end, 10);
          if (end == p) { set_error(std::string("TT_DEVICES: cannot parse '") + ev + "'"); return 1; }
          devs.push_back(static_cast<int>(v));
          p = (*end == ',') ? end + 1 : end;
        }
      }
    }
    if (devs.empty()) devs.push_back(0);
    for (int dv : devs) {
      if (dv < 0 || dv >= count) { set_error("invalid device index " + std::to_string(dv)); return 1; }
      std::shared_ptr<DeviceWeights> shared;
      for (int sidx = 0; sidx < kSlotsPerDevice; ++sidx) {
        std::unique_ptr<DeviceCtx> d(new DeviceCtx);
        d->device = dv;
        if (d->init(weights_dir, shared) != cudaSuccess) return 1;
        shared = d->w;
        e->devs.push_back(std::move(d));
      }
    }
    e->n_devices = static_cast<int>(devs.size());
    *out = e.release();
    return 0;
  } catch (const std::exception& ex) {
    set_error(std::string("tt_engine_create: ") + ex.what());
    return 1;
  }
}

void tt_engine_destroy(tt_engine* e) { delete e; }

int tt_device_count(void) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); return 0; }
  return count;
}

void tt_engine_set_slots(tt_engine* e, int slots) {
  if (e) e->slots.store(slots);
}

void* tt_engine_stream(tt_engine* e, int idx) {
  if (!e || idx < 0 || idx >= e->n_devices) return nullptr;
  return e->devs[idx * kSlotsPerDevice]->stream;
}
void tt_io_bytes(unsigned long long* h2d, unsigned long long* d2h) {
  if (h2d) *h2d = g_h2d_bytes.load();
  if (d2h) *d2h = g_d2h_bytes.load();
}
void tt_profile_enable(int on) { prof_enable(on != 0); }
void tt_profile_collect(double* total_ms, double* total_flops, unsigned long long* launches) {
  prof_collect(total_ms, total_flops, nullptr, launches);
}
int tt_profile_stages(char* buf, int cap) {
  const std::string csv = stage_collect();
  if (!buf || cap <= 0) return static_cast<int>(csv.size());
  const size_t n = std::min(csv.size(), static_cast<size_t>(cap - 1));
  std::memcpy(buf, csv.data(), n);
  buf[n] = 0;
  return static_cast<int>(csv.size());
}
void tt_profile_dump(const char* path, double* total_ms, double* total_flops, unsigned long long* launches) {
  prof_collect(total_ms, total_flops, nullptr, launches, path);
}

int tt_ocr_pages(tt_engine* e, const tt_image* pages, int n_pages, tt_result** out) {
  return tt_ocr_pages_ex(e, pages, n_pages, nullptr, out);
}

int tt_ocr_pages_ex(tt_engine* e, const tt_image* pages, int n_pages, const tt_ocr_options* opt, tt_result** out) {
  Request req;
  return make_request("tt_ocr_pages_ex", opt, nullptr, 0, nullptr, 0, nullptr, 0, 0.f, 0.5f, n_pages, &req)
             ? 1 : ocr_pages(e, pages, n_pages, req, out);
}

int tt_ocr_pages_filtered(tt_engine* e, const tt_image* pages, int n_pages, const tt_ocr_options* opt,
                          const tt_char_filter* filters, int n_filters, tt_result** out) {
  Request req;
  return make_request("tt_ocr_pages_filtered", opt, filters, n_filters, nullptr, 0, nullptr, 0, 0.f, 0.5f, n_pages, &req)
             ? 1 : ocr_pages(e, pages, n_pages, req, out);
}

int tt_ocr_pages_oriented(tt_engine* e, const tt_image* pages, int n_pages, const tt_ocr_options* opt,
                          const tt_char_filter* filters, int n_filters, const int* rotation_info, int n_rotations,
                          tt_result** out) {
  Request req;
  return make_request("tt_ocr_pages_oriented", opt, filters, n_filters, rotation_info, n_rotations, nullptr, 0, 0.f, 0.5f,
                      n_pages, &req)
             ? 1 : ocr_pages(e, pages, n_pages, req, out);
}

int tt_ocr_pages_lexicon(tt_engine* e, const tt_image* pages, int n_pages, const tt_ocr_options* opt,
                         const tt_char_filter* filters, int n_filters, const int* rotation_info, int n_rotations,
                         const tt_lexicon* const* lexicons, int n_lexicons, tt_result** out) {
  Request req;
  return make_request("tt_ocr_pages_lexicon", opt, filters, n_filters, rotation_info, n_rotations, lexicons, n_lexicons,
                      0.f, 0.5f, n_pages, &req)
             ? 1 : ocr_pages(e, pages, n_pages, req, out);
}

int tt_ocr_pages_contrast(tt_engine* e, const tt_image* pages, int n_pages, const tt_ocr_options* opt,
                          const tt_char_filter* filters, int n_filters, const int* rotation_info, int n_rotations,
                          const tt_lexicon* const* lexicons, int n_lexicons, float contrast_ths, float adjust_contrast,
                          tt_result** out) {
  Request req;
  return make_request("tt_ocr_pages_contrast", opt, filters, n_filters, rotation_info, n_rotations, lexicons, n_lexicons,
                      contrast_ths, adjust_contrast, n_pages, &req)
             ? 1 : ocr_pages(e, pages, n_pages, req, out);
}

}  // extern "C"

namespace {
// every tt_ocr_pages* entry point, after make_request
int ocr_pages(tt_engine* e, const tt_image* pages, int n_pages, const Request& req, tt_result** out) {
  try {
    const tt_ocr_options& opt = req.opt;
    if (!e || !out) { set_error("tt_ocr_pages: null argument"); return 1; }
    if (n_pages < 0 || (n_pages > 0 && !pages)) { set_error("tt_ocr_pages: bad page array"); return 1; }
    for (int i = 0; i < n_pages; ++i) {
      if (!pages[i].data || pages[i].rows <= 0 || pages[i].cols <= 0 || pages[i].channels != 3) {
        set_error("Error reading image from file");  // tuatara.cpp:344-347
        return 1;
      }
      if (pages[i].step < static_cast<size_t>(pages[i].cols) * 3) { set_error("tt_ocr_pages: row step smaller than cols * 3"); return 1; }
    }
    std::vector<PageOut> results(n_pages);
    const int G = e->n_devices;
    // detection units: pages of equal size, wherever they sit in the request; device-resident pages stay on their GPU
    WorkQueues q(G);
    {
      std::map<std::tuple<int, int, int>, int> open;   // (device or -1, rows, cols) -> unit being filled
      for (int i = 0; i < n_pages; ++i) {
        const int dev = opt.pages_on_device ? i % G : -1;
        const auto key = std::make_tuple(dev, pages[i].rows, pages[i].cols);
        auto it = open.find(key);
        if (it == open.end() || static_cast<int>(q.units[it->second].pages.size()) >= kCraftSubBatch) {
          q.units.emplace_back();
          const int ui = static_cast<int>(q.units.size()) - 1;
          open[key] = ui;
          if (dev >= 0) q.per_dev[dev].push_back(ui); else q.shared.push_back(ui);
          it = open.find(key);
        }
        q.units[it->second].pages.push_back(i);
      }
    }
    static const int env_slots = std::getenv("TT_SLOTS") ? std::atoi(std::getenv("TT_SLOTS")) : 0;  // development override
    const int cfg_slots = e->slots.load();
    const int want = std::max(1, std::min(cfg_slots > 0 ? cfg_slots : env_slots > 0 ? env_slots : 3, kSlotsPerDevice));
    // workers: device-major round robin, so that a short request touches every GPU before any second slot
    struct W { int g, sidx; };
    std::vector<W> ws;
    size_t shared_claimed = 0;
    for (int sidx = 0; sidx < want; ++sidx)
      for (int g = 0; g < G; ++g) {
        if (static_cast<size_t>(sidx) < q.per_dev[g].size()) ws.push_back(W{g, sidx});
        else if (shared_claimed < q.shared.size()) { ++shared_claimed; ws.push_back(W{g, sidx}); }
      }
    if (ws.empty() && n_pages > 0) ws.push_back(W{0, 0});
    std::vector<std::string> errs(ws.size());
    std::vector<int> rcs(ws.size(), 0);
    std::vector<std::thread> workers;
    for (size_t w = 1; w < ws.size(); ++w)
      workers.emplace_back([&, w] { slot_worker(*e, ws[w].g, ws[w].sidx, want, pages, req, &q, &results, &rcs[w], &errs[w]); });
    if (!ws.empty())
      slot_worker(*e, ws[0].g, ws[0].sidx, want, pages, req, &q, &results, &rcs[0], &errs[0]);
    for (auto& w : workers) w.join();
    for (size_t w = 0; w < ws.size(); ++w)
      if (rcs[w]) { set_error("device " + std::to_string(e->devs[ws[w].g * kSlotsPerDevice]->device) + ": " + errs[w]); return 1; }
    // host-side gather into the C result
    ResultBlock* rb = new ResultBlock{};
    tt_result* r = &rb->r;
    r->n_pages = n_pages;
    r->pages = new tt_page_result[n_pages];
    for (int i = 0; i < n_pages; ++i) {
      const PageOut& po = results[i];
      tt_page_result& pr = r->pages[i];
      pr.n_items = static_cast<int>(po.text.size());
      pr.items = pr.n_items ? new tt_item[pr.n_items] : nullptr;
      for (int k = 0; k < pr.n_items; ++k) {
        pr.items[k].text = new char[po.text[k].size() + 1];
        std::memcpy(pr.items[k].text, po.text[k].c_str(), po.text[k].size() + 1);
        std::memcpy(pr.items[k].bbox, po.bbox[k].data(), sizeof(float) * 4);
      }
    }
    if (req.orient.n > 1) {
      rb->angles = new std::vector<std::vector<int>>(n_pages);
      for (int i = 0; i < n_pages; ++i) (*rb->angles)[i] = std::move(results[i].angle);
    }
    if (opt.with_scores) {
      for (PageOut& po : results) {   // only the scores are kept
        po.text.clear();
        po.bbox.clear();
      }
      rb->scores = new std::vector<PageOut>(std::move(results));
    }
    *out = r;
    return 0;
  } catch (const std::exception& ex) {
    set_error(std::string("tt_ocr_pages: ") + ex.what());
    return 1;
  }
}
}  // namespace

extern "C" {

void tt_result_free(tt_result* r) {
  if (!r) return;
  for (int i = 0; i < r->n_pages; ++i) {
    for (int k = 0; k < r->pages[i].n_items; ++k) delete[] r->pages[i].items[k].text;
    delete[] r->pages[i].items;
  }
  delete[] r->pages;
  ResultBlock* rb = reinterpret_cast<ResultBlock*>(r);   // r is its first member (tt_ocr_pages_ex)
  delete rb->scores;
  delete rb->angles;
  delete rb;
}

int tt_item_angle(const tt_result* r, int page, int item, int* angle) {
  if (!r) { set_error("tt_item_angle: null result"); return 1; }
  const ResultBlock* rb = reinterpret_cast<const ResultBlock*>(r);
  if (!rb->angles) { set_error("tt_item_angle: the result was made without rotation candidates (tt_ocr_pages_oriented)"); return 1; }
  if (page < 0 || page >= r->n_pages || item < 0 || item >= r->pages[page].n_items) {
    set_error("tt_item_angle: page or item out of range");
    return 1;
  }
  if (angle) *angle = (*rb->angles)[page][item];
  return 0;
}

int tt_item_scores(const tt_result* r, int page, int item, float* conf, float* det_score, const float** char_conf,
                   int* n_chars) {
  if (!r) { set_error("tt_item_scores: null result"); return 1; }
  const ResultBlock* rb = reinterpret_cast<const ResultBlock*>(r);
  if (!rb->scores) { set_error("tt_item_scores: the result was made without tt_ocr_options.with_scores"); return 1; }
  if (page < 0 || page >= r->n_pages || item < 0 || item >= r->pages[page].n_items) {
    set_error("tt_item_scores: page or item out of range");
    return 1;
  }
  const PageOut& po = (*rb->scores)[page];
  const std::vector<float>& cc = po.char_conf[item];
  if (conf) *conf = po.conf[item];
  if (det_score) *det_score = po.det[item];
  if (char_conf) *char_conf = cc.empty() ? nullptr : cc.data();
  if (n_chars) *n_chars = static_cast<int>(cc.size());
  return 0;
}

int tt_craft_forward(tt_engine* e, const uint8_t* craft_input, int h32, int w32, float* maps_out) {
  try {
    if (!e) { set_error("tt_craft_forward: null engine"); return 1; }
    DeviceCtx& d = *e->devs[0];
    std::lock_guard<std::mutex> lock(d.mu);
    E_CUDA(cudaSetDevice(d.device));
    const size_t in_bytes = static_cast<size_t>(h32) * w32 * 3;
    E_TRY(d.arena.reserve(d.craft_bytes(1, h32, w32) + in_bytes + (8u << 20)));
    d.arena.reset();
    uint8_t* in = d.arena.get<uint8_t>(in_bytes);
    E_CUDA(cudaMemcpyAsync(in, craft_input, in_bytes, cudaMemcpyHostToDevice, d.stream));
    float* maps = nullptr;
    E_TRY(d.craft_forward(in, 1, h32, w32, &maps));
    E_CUDA(cudaMemcpyAsync(maps_out, maps, sizeof(float) * (h32 / 2) * (w32 / 2) * 2, cudaMemcpyDeviceToHost, d.stream));
    E_TRY(stream_sync(d.stream));
    return 0;
  } catch (const std::exception& ex) {
    set_error(std::string("tt_craft_forward: ") + ex.what());
    return 1;
  }
}

int tt_craft_tap(tt_engine* e, const char* name, float* out, long long capacity, int dims_out[3]) {
  try {
    if (!e || !name) { set_error("tt_craft_tap: null argument"); return 1; }
    DeviceCtx& d = *e->devs[0];
    std::lock_guard<std::mutex> lock(d.mu);
    E_CUDA(cudaSetDevice(d.device));
    for (const CraftTap& t : d.craft_taps) {
      if (std::strcmp(t.name, name) != 0) continue;
      const long long n = static_cast<long long>(t.H) * t.W * t.C;
      if (dims_out) { dims_out[0] = t.H; dims_out[1] = t.W; dims_out[2] = t.C; }
      if (!out) return 0;
      if (capacity < n) { set_error("tt_craft_tap: output buffer too small"); return 1; }
      std::vector<__nv_bfloat16> h(static_cast<size_t>(n));
      E_CUDA(cudaMemcpy(h.data(), t.ptr, sizeof(__nv_bfloat16) * n, cudaMemcpyDeviceToHost));
      for (long long i = 0; i < n; ++i) out[i] = __bfloat162float(h[static_cast<size_t>(i)]);
      return 0;
    }
    set_error(std::string("tt_craft_tap: no activation named '") + name + "' (run tt_craft_forward first)");
    return 1;
  } catch (const std::exception& ex) {
    set_error(std::string("tt_craft_tap: ") + ex.what());
    return 1;
  }
}

}  // extern "C"

namespace {
// tt_parseq_forward, tt_parseq_forward_scores, tt_parseq_forward_masked and tt_parseq_forward_lexicon (pmax_out != null:
// the refinement head also writes the probabilities; class_masks != null: [n][4] per-crop class masks; lex != null: every
// crop walks the lexicon's trie)
int parseq_stage(tt_engine* e, const uint8_t* crops, int n, const int32_t* forced_tokens, const uint32_t* class_masks,
                 const tt_lexicon* lex, float* logits_out, int32_t* ids_out, float* pmax_out) {
  try {
    if (!e) { set_error("tt_parseq_forward: null engine"); return 1; }
    if (n <= 0) return 0;
    DeviceCtx& d = *e->devs[0];
    std::lock_guard<std::mutex> lock(d.mu);
    E_CUDA(cudaSetDevice(d.device));
    const int L = d.w->pd.L, NC = d.w->pd.n_cls_pad;
    LexDev lx{};
    std::vector<int> roots;
    if (lex) {
      LexTableBuilder table;
      roots.assign(std::min(n, kMaxCropsPerPass), table.append(lex->trie));
      if (upload_lex_table(d, table.words(), table.n_states(), &lx)) return 1;
    }
    for (int c0 = 0; c0 < n; c0 += kMaxCropsPerPass) {
      const int nc = std::min(kMaxCropsPerPass, n - c0);
      const size_t crop_bytes = static_cast<size_t>(nc) * 32 * 128 * 3;
      E_TRY(d.arena.reserve(d.parseq_bytes(nc) + crop_bytes + static_cast<size_t>(nc) * (128 * 96 * 2 + 4 * L) + (8u << 20) +
                            (pmax_out ? sizeof(float) * nc * L : 0) + (class_masks ? 16 * static_cast<size_t>(nc) : 0) +
                            (lex ? 8 * static_cast<size_t>(nc) : 0)));
      d.arena.reset();
      if (lex) {
        int* root_dev = d.arena.get<int>(nc);
        lx.state = d.arena.get<int>(nc);
        E_CUDA(cudaMemcpyAsync(root_dev, roots.data(), sizeof(int) * nc, cudaMemcpyHostToDevice, d.stream));
        lx.root = root_dev;
      }
      float* pmax = pmax_out ? d.arena.get<float>(static_cast<size_t>(nc) * L) : nullptr;
      uint32_t* mask = class_masks ? d.arena.get<uint32_t>(4 * static_cast<size_t>(nc)) : nullptr;
      if (mask)
        E_CUDA(cudaMemcpyAsync(mask, class_masks + 4 * static_cast<size_t>(c0), 16 * static_cast<size_t>(nc), cudaMemcpyHostToDevice,
                               d.stream));
      uint8_t* cu8 = d.arena.get<uint8_t>(crop_bytes);
      __nv_bfloat16* patches = d.arena.get<__nv_bfloat16>(static_cast<size_t>(nc) * 128 * 96);
      int* forced = forced_tokens ? d.arena.get<int>(static_cast<size_t>(nc) * (L - 1)) : nullptr;
      E_CUDA(cudaMemcpyAsync(cu8, crops + static_cast<size_t>(c0) * 32 * 128 * 3, crop_bytes, cudaMemcpyHostToDevice, d.stream));
      if (forced)
        E_CUDA(cudaMemcpyAsync(forced, forced_tokens + static_cast<size_t>(c0) * (L - 1), sizeof(int) * nc * (L - 1),
                               cudaMemcpyHostToDevice, d.stream));
      E_TRY(patchify_u8(cu8, nc, patches, d.stream));
      float* logits = nullptr;
      int* ids = nullptr;
      E_TRY(d.parseq_forward(patches, nc, forced, &logits, &ids, pmax, mask, lex ? &lx : nullptr));
      if (logits_out)
        E_CUDA(cudaMemcpy2DAsync(logits_out + static_cast<size_t>(c0) * L * d.w->pd.n_cls, sizeof(float) * d.w->pd.n_cls, logits,
                                 sizeof(float) * NC, sizeof(float) * d.w->pd.n_cls, static_cast<size_t>(nc) * L,
                                 cudaMemcpyDeviceToHost, d.stream));
      if (ids_out)
        E_CUDA(cudaMemcpyAsync(ids_out + static_cast<size_t>(c0) * L, ids, sizeof(int) * nc * L, cudaMemcpyDeviceToHost, d.stream));
      if (pmax_out)
        E_CUDA(cudaMemcpyAsync(pmax_out + static_cast<size_t>(c0) * L, pmax, sizeof(float) * nc * L, cudaMemcpyDeviceToHost, d.stream));
      E_TRY(stream_sync(d.stream));
    }
    return 0;
  } catch (const std::exception& ex) {
    set_error(std::string("tt_parseq_forward: ") + ex.what());
    return 1;
  }
}
}  // namespace

extern "C" {

int tt_parseq_forward(tt_engine* e, const uint8_t* crops, int n, const int32_t* forced_tokens, float* logits_out,
                      int32_t* ids_out) {
  return parseq_stage(e, crops, n, forced_tokens, nullptr, nullptr, logits_out, ids_out, nullptr);
}

int tt_parseq_forward_scores(tt_engine* e, const uint8_t* crops, int n, int32_t* ids_out, float* pmax_out) {
  if (!pmax_out) { set_error("tt_parseq_forward_scores: null pmax_out"); return 1; }
  return parseq_stage(e, crops, n, nullptr, nullptr, nullptr, nullptr, ids_out, pmax_out);
}

int tt_parseq_forward_masked(tt_engine* e, const uint8_t* crops, int n, const int32_t* forced_tokens, const uint32_t* class_masks,
                             float* logits_out, int32_t* ids_out, float* pmax_out) {
  return parseq_stage(e, crops, n, forced_tokens, class_masks, nullptr, logits_out, ids_out, pmax_out);
}

int tt_parseq_forward_lexicon(tt_engine* e, const uint8_t* crops, int n, const int32_t* forced_tokens, const tt_lexicon* lex,
                              float* logits_out, int32_t* ids_out, float* pmax_out) {
  if (!lex) { set_error("tt_parseq_forward_lexicon: null lexicon"); return 1; }
  return parseq_stage(e, crops, n, forced_tokens, nullptr, lex, logits_out, ids_out, pmax_out);
}

int tt_postprocess_dev(tt_engine* e, const float* maps_dev, int batch, int H, int W, int* n_rects_total, void*) {
  try {
    if (!e) { set_error("tt_postprocess_dev: null engine"); return 1; }
    DeviceCtx& d = *e->devs[0];
    std::lock_guard<std::mutex> lock(d.mu);
    E_CUDA(cudaSetDevice(d.device));
    std::vector<std::vector<DetBox>> det;
    if (detect_boxes(d, e->cfg, maps_dev, batch, H, W, &det)) return 1;
    int total = 0;
    for (auto& v : det) total += static_cast<int>(v.size());
    if (n_rects_total) *n_rects_total = total;
    return 0;
  } catch (const std::exception& ex) {
    set_error(std::string("tt_postprocess_dev: ") + ex.what());
    return 1;
  }
}

}  // extern "C"
