/* C ABI of the B200-native Tuatara OCR hot path (libtuatara_b200.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch/OpenCV types, no
 * exceptions.  Every function returns 0 on success and non-zero on failure; the message is
 * available from tt_last_error() (thread-local).  The reference has no FFI of its own -- its
 * boundary is the C++ function image_to_data (tuatara.h:13) and the pybind11 module
 * (bindings/python.cpp:54-58); include/tuatara.h and tuatara_b200/bindings/python.cpp re-create
 * those on top of this ABI.  Each entry point cites the reference code it replaces.
 */
#ifndef TUATARA_C_H
#define TUATARA_C_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define TT_API __attribute__((visibility("default")))
#else
#define TT_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define TT_MAX_LABEL_LEN 26  /* PARSeq positions per crop (max_label_length + 1) */
#define TT_NUM_CLASSES 95    /* logits per position */

typedef struct tt_engine tt_engine;

/* A caller-owned 8-bit, 3-channel, row-major image (the cv::Mat of tuatara.h:13 without OpenCV).
 * The buffer is only read (the reference swaps channels in place at tuatara.cpp:349; here the
 * swap happens inside the kernels). */
typedef struct tt_image {
  const uint8_t* data;
  int rows, cols, channels; /* channels must be 3 */
  size_t step;              /* bytes per row */
} tt_image;

/* Every literal of the reference gathered in one struct (the TODO at tuatara.cpp:396). */
typedef struct tt_config {
  float canvas_size;    /* 1024  tuatara.cpp:352 */
  float mag_ratio;      /* 1.0   tuatara.cpp:353 */
  float text_threshold; /* 0.7   tuatara.cpp:397 */
  float link_threshold; /* 0.4   tuatara.cpp:398 */
  float low_text;       /* 0.4   tuatara.cpp:399 */
  int min_area;         /* 10    tuatara.cpp:148 */
  int max_batch_pages;  /* pages whose crops form one PARSeq batch in a slot (0 = default 32); detection runs in units of <= 8
                           equally sized pages, crops of pages of any size share the recognition batch */
  int slots_per_gpu;    /* concurrent execution slots (streams + host threads) per GPU: 0 = default 3, max 4.  More slots
                           overlap one batch's host phases and latency-bound kernels with another batch's kernels
                           (2 slots +16 %, 3 slots +19 % over 1 on the 512-page bench); 1 = strictly serial kernels */
  int rectify;          /* 0 (default) = the reference's axis-aligned boundingRect crop (tuatara.cpp:416).  1 = opt-in for the
                           TODO at tuatara.cpp:411-415: each crop is the perspective warp of its rotated box to 128 x 32
                           (cv::getPerspectiveTransform + cv::warpPerspective semantics); boxes / bboxes are unchanged */
} tt_config;

typedef struct tt_item {
  char* text;    /* NUL-terminated, owned by the result */
  float bbox[4]; /* min_x, min_y, max_x, max_y (tuatara.cpp:256-274) */
} tt_item;
typedef struct tt_page_result {
  int n_items;
  tt_item* items; /* in CCL label order (tuatara.cpp:146) */
} tt_page_result;
typedef struct tt_result {
  int n_pages;
  tt_page_result* pages;
} tt_result;

/* ---------------------------------------------------------------- whole path */
TT_API void tt_config_default(tt_config* cfg);
TT_API const char* tt_last_error(void);
/* Engine = weights resident on each listed device + streams + workspaces.  Replaces the two
 * torch::jit::load calls per image (tuatara.cpp:333-336, :423-428): weights_dir must hold
 * craft.ttw and parseq.ttw (tuatara_b200.weights exporter).  devices == NULL -> the devices named by the TT_DEVICES
 * environment variable ("0,1,2" or "all"), else {0}. */
TT_API int tt_engine_create(const char* weights_dir, const int* devices, int n_devices, const tt_config* cfg,
                     tt_engine** out);
TT_API void tt_engine_destroy(tt_engine* e);
/* CUDA devices visible to this process (0 when there is none: the library has no CPU fallback). */
TT_API int tt_device_count(void);
/* image_to_data (tuatara.cpp:314-512) for a batch of pages.  The pages are cut into detection units that the execution
 * slots of all the engine's GPUs pull from a shared work queue (no collective: pages are independent); results are
 * gathered on the host in page order. */
TT_API int tt_ocr_pages(tt_engine* e, const tt_image* pages, int n_pages, tt_result** out);
/* Same, with options the benchmark and the parity tests need.
 *  pages_on_device: tt_image.data are device pointers (page i on the GPU that gets page i, i.e.
 *    engine device i % n_devices) -- throughput with inputs already resident in HBM.
 *  score_override: NULL, or n_pages pointers (NULL entries allowed) to fp32 [h32/2][w32/2][2] maps
 *    that replace CRAFT's output for that page AFTER CRAFT has run in full (random-init weights
 *    give near-constant maps; SURVEY.md 8d).  override_on_device: those pointers are device memory.
 *  Zero-initialise the struct: fields added later default to 0. */
typedef struct tt_ocr_options {
  int pages_on_device;
  int override_on_device;
  const float* const* score_override;
  int detect_only;   /* 1: stop after the word boxes (tuatara.cpp:349-418): items carry bbox and an empty text
                        (BASELINE config "CRAFT detection only") */
  int with_scores;   /* 1: the result also holds per-item scores, read with tt_item_scores (0: none, the default) */
} tt_ocr_options;
TT_API int tt_ocr_pages_ex(tt_engine* e, const tt_image* pages, int n_pages, const tt_ocr_options* opt, tt_result** out);
TT_API void tt_result_free(tt_result* r);
/* Character filter (INTEGRATION.md section 7): restricts the characters recognition may produce.  allow / block are
 * NUL-terminated byte strings or NULL (no restriction).  Class c of the 95 prints itos[c] (tt_tokenizer_table); classes 0
 * (end of word) and 88 (dropped from the text) print nothing and are always allowed.  Any other class is allowed iff
 * (allow == NULL or allow holds its character) and (block == NULL or block does not).  Characters no class prints are
 * ignored; allow = "" is valid and gives every word an empty text.  The choice is made inside the greedy decode: at every
 * AR step (the token fed back is the best allowed class) and at the refinement.  Boxes, bboxes, det_score, item order
 * and detect_only results do not change; a filter that allows every class gives bit-identical results to no filter. */
typedef struct tt_char_filter {
  const char* allow;
  const char* block;
} tt_char_filter;
/* The filter's class mask (host only): bit c & 31 of mask_out[c >> 5] is set when class c is allowed; mask_out[3] = 0. */
TT_API int tt_char_filter_mask(const tt_char_filter* f, uint32_t mask_out[4]);
/* tt_ocr_pages_ex with character filters.  n_filters == 1: filters[0] for every page; == n_pages: filters[i] for page i;
 * == 0 (filters may be NULL): the same as tt_ocr_pages_ex.  Any other count, or filters == NULL with n_filters > 0, is an
 * error.  Every character of every item's text is in its page's allow (when given) and not in its block (when given). */
TT_API int tt_ocr_pages_filtered(tt_engine* e, const tt_image* pages, int n_pages, const tt_ocr_options* opt,
                                 const tt_char_filter* filters, int n_filters, tt_result** out);
/* Scores of item `item` of page `page` of a result made with tt_ocr_options.with_scores = 1 (an error otherwise).
 * Scale 0..1.  p[t] is the largest softmax probability of the refinement logits at position t (t = 0..25), the
 * position's id being its argmax; the end position e is the first t whose id is 0 (where the text stops), else 25.
 * With a character filter (tt_ocr_pages_filtered) the softmax is renormalised over the page's allowed classes:
 * p[t] = 1 / sum_{c allowed} exp(l[t][c] - max_{c allowed} l[t][c]), the id being the argmax over those classes.
 *  conf       = p[0] * ... * p[e] (the end position and positions of id 88 included), multiplied in double and
 *               rounded once to float; may underflow to 0.  -1 when the item was not recognised (detect_only).
 *  det_score  = the component's maximum normalised text score (tuatara.cpp:151-152), >= text_threshold.
 *  char_conf  = p[t] of each position that produced a character of the item's text, in order (*n_chars == strlen(text));
 *               memory owned by the result, valid until tt_result_free.  NULL (and 0) when not recognised.
 * Every output pointer may be NULL. */
TT_API int tt_item_scores(const tt_result* r, int page, int item, float* conf, float* det_score, const float** char_conf,
                          int* n_chars);
/* Rotation candidates (INTEGRATION.md section 8): tt_ocr_pages_filtered where every word is also read turned 90, 180 or
 * 270 degrees counter-clockwise, as listed in rotation_info (n_rotations distinct values from {90, 180, 270}, any order).
 * Candidate 0, the crop tt_ocr_pages_filtered reads, is always included; candidates are ordered 0, 90, 180, 270.  With
 * rectify == 0 candidate a is cv::resize(cv::rotate(roi, a), 128 x 32); with rectify == 1 it is the warp of the box's
 * quad with its corners shifted cyclically by a / 90.  Each candidate gets the conf of tt_item_scores (under its page's
 * filter); a later candidate replaces the best so far only when its conf is strictly greater.  The item's text (and,
 * with with_scores, conf and char_conf) are the winner's; bbox, det_score and item order do not change.  Read the angle
 * with tt_item_angle.  n_rotations == 0 (rotation_info may be NULL) is tt_ocr_pages_filtered; any other value outside
 * {90, 180, 270}, or one given twice, is an error that names it, reported before any device work. */
TT_API int tt_ocr_pages_oriented(tt_engine* e, const tt_image* pages, int n_pages, const tt_ocr_options* opt,
                                 const tt_char_filter* filters, int n_filters, const int* rotation_info, int n_rotations,
                                 tt_result** out);
/* Lexicons (INTEGRATION.md section 9): every recognised word is read from a caller's word list.  Class c of the 95 prints
 * itos[c] (tt_tokenizer_table); class 0 ends the word, class 88 prints nothing and backslash is printed by classes 69 and 87.
 *  Words: 1..25 bytes each, every byte printed by a class of 1..94 other than 88 (so not ']', '~', a control byte or a
 *    non-ASCII byte).  Anything else is an error naming the word's index and the byte (or the length); so are
 *    words == NULL and n_words < 1.  Duplicates count once.
 *  Automaton: a trie over the words.  A state allows class 0 iff a word ends there, and class c (1..94, not 88) iff a
 *    word continues with itos[c] (both backslash classes lead to the same child).  After class 0 the crop is in a done
 *    state that allows every class and loops to itself; nothing decoded there reaches the text.
 *  Greedy choice: at every AR step the token fed back is the first maximum over the classes the crop's state allows (the
 *    lowest allowed class when no allowed logit compares, i.e. all are NaN); the state then advances by it.  The ids are a
 *    second walk over the refinement logits from the root with the same rule, and with scores p[t] of tt_item_scores is
 *    renormalised over the classes the state at position t allows.  Rotation candidates are chosen by that conf.
 * A tt_lexicon is immutable: concurrent requests may share it; destroy it once they have returned. */
typedef struct tt_lexicon tt_lexicon;
TT_API int tt_lexicon_create(const char* const* words, int n_words, tt_lexicon** out);
TT_API void tt_lexicon_destroy(tt_lexicon* lex);
/* n_words: the distinct words; n_states: the states of the trie (the root included, the done state not).  Both nullable. */
TT_API int tt_lexicon_info(const tt_lexicon* lex, int* n_words, int* n_states);
/* tt_ocr_pages_oriented with lexicons.  n_lexicons == 1: lexicons[0] for every page; == n_pages: lexicons[i] for page i;
 * == 0 (lexicons may be NULL): exactly tt_ocr_pages_oriented.  Any other count, or lexicons == NULL with n_lexicons > 0, is
 * an error.  A NULL entry decodes its page under a one-state automaton allowing its filter's classes (every class without
 * a filter): its results are bit-identical to tt_ocr_pages_oriented's.  A page with a filter and a lexicon reads from the
 * lexicon's words whose every character the filter allows; none is an error naming the page.  Every check is made
 * before any device work.  Each item's text is then one of its page's words (or empty for a detect_only request);
 * bbox, det_score and item order do not change. */
TT_API int tt_ocr_pages_lexicon(tt_engine* e, const tt_image* pages, int n_pages, const tt_ocr_options* opt,
                                const tt_char_filter* filters, int n_filters, const int* rotation_info, int n_rotations,
                                const tt_lexicon* const* lexicons, int n_lexicons, tt_result** out);
/* The contrast re-read (INTEGRATION.md section 10, EasyOCR's readtext(contrast_ths, adjust_contrast)): tt_ocr_pages_lexicon
 * where a word whose first read has conf (tt_item_scores, under its page's filter or lexicon) below contrast_ths and whose
 * 128 x 32 crop has low contrast is read again from a contrast-stretched crop.  On the crop (the winning rotation candidate,
 * rectify 0 or 1): grey = cv2 BGR2GRAY of its channels in the caller's order, low / high = np.percentile(grey, 10 / 90),
 * contrast = (high - low) / max(10, high + low); low contrast iff contrast < adjust_contrast.  Then every channel value v
 * becomes uint8(clip((v - low + 25) * 200 / max(10, high - low), 0, 255)) in double (EasyOCR's adjust_contrast_grey, one
 * map for all three channels), and the crop is decoded again under the same filter or lexicon, at the same angle.  The
 * second read replaces the first only when its conf is strictly greater (ties and NaN keep the first; EasyOCR gives ties
 * to the second).  text, and with with_scores conf and char_conf, are the winner's; bbox, det_score, angle and item order
 * do not change.  contrast_ths: finite, >= 0 (0 = off: exactly tt_ocr_pages_lexicon); adjust_contrast: finite, in (0, 1]
 * (EasyOCR's defaults are 0.1 and 0.5).  Any other value is an error that names it, reported before any device work. */
TT_API int tt_ocr_pages_contrast(tt_engine* e, const tt_image* pages, int n_pages, const tt_ocr_options* opt,
                                 const tt_char_filter* filters, int n_filters, const int* rotation_info, int n_rotations,
                                 const tt_lexicon* const* lexicons, int n_lexicons, float contrast_ths, float adjust_contrast,
                                 tt_result** out);
/* The angle (0, 90, 180 or 270) of the candidate that was read for item `item` of page `page`, -1 when the item was not
 * recognised (detect_only).  An error on a result not made by tt_ocr_pages_oriented with n_rotations > 0. */
TT_API int tt_item_angle(const tt_result* r, int page, int item, int* angle);
/* Kernel launches issued by this library so far (bench.py's gpu_launches). */
TT_API unsigned long long tt_launch_count(void);

/* Change slots_per_gpu of a live engine (1 = strictly serial kernels: per-launch event timing is only
 * meaningful then). */
TT_API void tt_engine_set_slots(tt_engine* e, int slots);
/* cudaStream_t the engine's idx-th device works on (bench.py records its CUDA events there). */
TT_API void* tt_engine_stream(tt_engine* e, int idx);
/* Host<->device bytes moved by tt_ocr_pages* so far (bench.py's h2d/d2h_bytes_per_step). */
TT_API void tt_io_bytes(unsigned long long* h2d, unsigned long long* d2h);
/* Per-launch CUDA-event timing of the tensor-core GEMM/conv kernel. tt_profile_collect waits for the
 * recorded launches, returns their summed duration, algorithmic FLOPs and count, and clears the log. */
TT_API void tt_profile_enable(int on);
TT_API void tt_profile_collect(double* total_ms, double* total_flops, unsigned long long* launches);
/* Same, and appends one CSV line per launch ("tag,flops,ms") to `path` (per-layer tables in profiles/). */
TT_API void tt_profile_dump(const char* path, double* total_ms, double* total_flops, unsigned long long* launches);

/* Stage-level timings recorded while the profile is enabled: "name,count,ms,flops,bytes\n" per stage of
 * image_to_data (preprocess tuatara.cpp:206-234, craft :376, postprocess :119-204, crop_resize :416-448,
 * parseq_encoder / parseq_decoder :307), flops / bytes being the stage's algorithmic work.  Writes at most
 * cap-1 characters + NUL, returns the full length, clears the log. */
TT_API int tt_profile_stages(char* buf, int cap);

/* Development aid (TT_TRACE=1 in the environment, off otherwise): where every CTA of the TMEM-allocating kernels stands,
 * read from a host-mapped progress buffer -- callable from a watchdog thread while a kernel is stuck on the GPU.
 * Writes at most cap-1 characters + NUL, returns the full length. */
TT_API int tt_debug_trace_report(char* buf, int cap);

/* ---------------------------------------------------- stage level, host memory */
/* Size arithmetic of resize_aspect_ratio (tuatara.cpp:211-226), fp32 like the reference. */
TT_API int tt_resize_plan(int rows, int cols, float canvas_size, float mag_ratio, int* target_h, int* target_w, int* h32,
                   int* w32, float* ratio);
/* Channel swap + resize + zero pad (tuatara.cpp:349, :206-234). out: h32*w32*3 bytes. */
TT_API int tt_preprocess(const tt_image* image, float canvas_size, float mag_ratio, uint8_t* out);
/* CRAFT forward (tuatara.cpp:363-394). craft_input = tt_preprocess output; maps_out: [h32/2][w32/2][2] fp32. */
TT_API int tt_craft_forward(tt_engine* e, const uint8_t* craft_input, int h32, int w32, float* maps_out);
/* get_detected_boxes (tuatara.cpp:119-204) on one score map [H][W][2].
 *  labels_out  (nullable) [H*W] int32          == cv::connectedComponentsWithStats labels
 *  stats_out   (nullable) [stats_cap][5] int32 == its stats rows (left, top, width, height, area), row 0 = background
 *  rects_out   [rect_cap][5] fp32 (cx, cy, w, h, angle) of the kept components, rect_labels_out their labels */
TT_API int tt_postprocess(const float* maps, int H, int W, const tt_config* cfg, int32_t* labels_out, int32_t* stats_out,
                   int stats_cap, int* n_labels, float* rects_out, int32_t* rect_labels_out, int rect_cap,
                   int* n_rects);
/* Crop + resize to 128x32 (tuatara.cpp:416, :440-441). rects_xywh already clamped to the image.
 * out: [n][32][128][3] u8 in the caller's channel order. */
TT_API int tt_crop_resize(const tt_image* image, const int32_t* rects_xywh, int n, uint8_t* out);
/* tt_crop_resize with each crop turned angles[i] degrees counter-clockwise (0, 90, 180 or 270) before the resize:
 * cv::resize(cv::rotate(roi, code), (128, 32)).  Angle 0 gives tt_crop_resize's bytes. */
TT_API int tt_crop_resize_rotated(const tt_image* image, const int32_t* rects_xywh, const int32_t* angles, int n, uint8_t* out);
/* Per-slice parity of the CRAFT forward (SURVEY 8d): a named activation of the LAST tt_craft_forward call on this
 * engine as fp32 [H][W][C] (names: relu2_2, relu3_2, relu4_3, relu5_3, fc7, up1, up2, up3, up4 -- upstream CRAFT's
 * skip / U-net tensors).  out == NULL only reports dims_out = {H, W, C}.  Test entry point: not thread safe against
 * other calls on the same engine. */
TT_API int tt_craft_tap(tt_engine* e, const char* name, float* out, long long capacity, int dims_out[3]);
/* Rectified crops (tt_config.rectify): quads [n][4][2] fp32 = top-left, top-right, bottom-right, bottom-left corners in
 * image coordinates (may leave the image: border pixels are replicated).  out: [n][32][128][3] u8. */
TT_API int tt_crop_warp(const tt_image* image, const float* quads, int n, uint8_t* out);
/* The quad tt_config.rectify uses for a RotatedRect {cx, cy, w, h, angle}: 8 floats, corner order as above. */
TT_API int tt_rect_to_quad(const float rect[5], float quad_out[8]);
/* PARSeq forward (tuatara.cpp:307, 26 AR steps + 1 refinement). crops: [n][32][128][3] u8.
 * forced_tokens (nullable) [n][25]: teacher-forced AR context (parity tests).
 * logits_out (nullable) [n][26][95] fp32; ids_out (nullable) [n][26] argmax (== softmax + max, :486,:103). */
TT_API int tt_parseq_forward(tt_engine* e, const uint8_t* crops, int n, const int32_t* forced_tokens, float* logits_out,
                      int32_t* ids_out);
/* tt_parseq_forward's ids together with pmax_out [n][26]: the largest softmax probability of the refinement logits at
 * each position (the p[t] of tt_item_scores), from the same kernel that picks the ids.  ids_out [n][26]. */
TT_API int tt_parseq_forward_scores(tt_engine* e, const uint8_t* crops, int n, int32_t* ids_out, float* pmax_out);
/* tt_parseq_forward / tt_parseq_forward_scores with per-crop class masks (tt_char_filter_mask): class_masks [n][4]
 * (NULL = none).  Every AR step feeds back the argmax over the crop's allowed classes (forced_tokens, when given, still
 * win) and ids_out / pmax_out are the refinement's argmax and renormalised probability over them.  logits_out holds the
 * raw, unmasked head output.  Every output pointer may be NULL. */
TT_API int tt_parseq_forward_masked(tt_engine* e, const uint8_t* crops, int n, const int32_t* forced_tokens,
                                    const uint32_t* class_masks, float* logits_out, int32_t* ids_out, float* pmax_out);
/* tt_parseq_forward_masked with one lexicon for every crop instead of class masks: every AR step feeds back the choice of
 * the crop's trie walk (forced_tokens, when given, win and the AR steps do not consult the trie), and ids_out / pmax_out
 * are the refinement walk's.  logits_out holds the raw head output (TT_PARSEQ_AR_LOGITS=1: the AR pass's, like the other
 * forwards).  Every output pointer may be NULL. */
TT_API int tt_parseq_forward_lexicon(tt_engine* e, const uint8_t* crops, int n, const int32_t* forced_tokens,
                                     const tt_lexicon* lex, float* logits_out, int32_t* ids_out, float* pmax_out);
/* The contrast stretch of tt_ocr_pages_contrast on host crops [n][32][128][3] (tt_crop_resize's layout): out [n][32][128][3]
 * holds each crop stretched when it has low contrast for adjust_contrast (in (0, 1]), else unchanged; stretched
 * (nullable) [n] is 1 for a stretched crop, else 0.  Runs the kernels the engine runs. */
TT_API int tt_contrast_adjust(const uint8_t* crops, int n, float adjust_contrast, uint8_t* out, int32_t* stretched);
/* Tokenizer::decode + truncation (tuatara.cpp:61-116, :497-502). ids [n][len]; out [n][out_stride] chars. */
TT_API int tt_decode(const int32_t* ids, int n, int len, char* out, int out_stride);
/* tt_decode with the scores of tt_item_scores (host only).  pmax [n][len]; conf_out (nullable) [n];
 * char_conf_out (nullable) [n][len]: row i starts with the char_conf of string i, the rest of the row is 0. */
TT_API int tt_decode_scores(const int32_t* ids, const float* pmax, int n, int len, char* out, int out_stride, float* conf_out,
                            float* char_conf_out);
/* itos_out: >= 99 bytes. */
TT_API int tt_tokenizer_table(char* itos_out, int* eos_id, int* bos_id, int* pad_id);

/* ------------------------------------------------- host geometry (no GPU needed) */
TT_API int tt_convex_hull_i32(const int32_t* xy, int n, int32_t* idx_out, int* n_out);
TT_API int tt_convex_hull_f32(const float* xy, int n, int32_t* idx_out, int* n_out);
TT_API int tt_min_area_rect_i32(const int32_t* xy, int n, float rect_out[5]);
TT_API int tt_min_area_rect_f32(const float* xy, int n, float rect_out[5]);
TT_API int tt_rect_points(const float rect[5], float pts_out[8]);
TT_API int tt_rect_bounding(const float rect[5], int32_t xywh_out[4]);
TT_API int tt_adjust_rect(const float rect[5], float ratio_w, float ratio_h, float ratio_net, float rect_out[5]);
TT_API int tt_rect_to_bbox(const float rect[5], float bbox_out[4]);

/* --------------------------------------- stage level, device memory (bench / kernel tests) */
/* out[M][N] = act(A[M][K] * W[N][K]^T + bias) (+ residual). All pointers are device pointers;
 * A, W bf16; bias fp32; out bf16 (out_f32 == 0) or fp32. act: 0 none, 1 relu, 2 gelu.
 * BN: N tile (0 = planner decides); resident: schedule flags -- with BN given: bit 0 = weight-resident,
 * bit 1 = CTA-pair (cta_group::2, 256-row tiles); with BN == 0: 4 = pair forced, 8 = pair forbidden, else planner. */
TT_API int tt_linear_dev(const void* A, int lda, int M, int K, const void* W, int N, const float* bias, int act,
                  const void* residual, int res_f32, int ldr, void* out, int out_f32, int ldc, int BN, int resident,
                  void* stream);
/* Kernel test of the fused LayerNorm pair the PARSeq encoder runs (x += A W1^T + b1; y = act(Linear(LN(x)))).  The fp32
 * residual stream x is kept split: x_hi = bf16(x), x_lo = bf16(x - x_hi), both bf16 [M][D], updated in place (x_hi is
 * the second GEMM's A operand).  stats fp32 [M][8] scratch, W2f = W2 * gamma (bf16 [N2][D]), c0[n] = b2[n] + beta . W2[n],
 * c1[n] = sum_k W2f[n][k]; out bf16 [M][N2].  All device pointers. */
TT_API int tt_linear_ln_pair_dev(const void* A, int M, int K1, const void* W1, const float* b1, int D, void* x_hi, void* x_lo,
                          float* stats, const void* W2f, const float* c0, const float* c1, int N2, int act, float eps,
                          void* out, void* stream);
/* The LayerNorm-consumer GEMM alone (the second half of tt_linear_ln_pair_dev): out = LN(x) W^T + b from A = bf16(x)
 * [M][K], stats fp32 [M][parts][2] (1 <= parts <= 4 partial (sum x, sum x^2) pairs per row), Wf = W * gamma bf16 [N][K],
 * c0 / c1 fp32 [N] as above; out bf16 [M][N].  All device pointers. */
TT_API int tt_linear_ln_dev(const void* A, int M, int K, const void* Wf, const float* c0, const float* c1, int N, const float* stats,
                            int parts, float eps, void* out, void* stream);
/* Kernel test of the fused second half of a PARSeq-base encoder block (timm Block, reached by the reference through
 * TorchScript at tuatara.cpp:307):  x += att Wp^T + bp  (the attention output projection; skipped when att is NULL), then
 * x += fc2(GELU(fc1(LN2(x)))) -- one kernel, neither x1 nor the hidden activations leave the SM.  The residual stream is the
 * split pair of tt_linear_ln_pair_dev (bf16 [M][384] each, updated in place); stats fp32 [M][4]: with att == NULL two
 * partial (sum x, sum x^2) pairs per row on entry; on return the two partials of the new x.  att bf16 [M][384], Wp bf16
 * [384][384], bp fp32 [384]; W1f = fc1 * gamma bf16 [1536][384], c0 / c1 as above, W2 bf16 [384][1536], b2 fp32 [384].
 * All device pointers. */
TT_API int tt_enc_mlp_dev(void* x_hi, void* x_lo, float* stats, long long M, const void* att, const void* Wp, const float* bp,
                   const void* W1f, const float* c0, const float* c1, const void* W2, const float* b2, float eps, void* stream);
/* Kernel test of the fused first half of a PARSeq encoder block: qkv = LN1(x) Wqkv^T + b (LayerNorm applied to the
 * accumulators, as tt_linear_ln_pair_dev's second GEMM does) and the self attention of tt_attn_enc_dev (one-pass), in one
 * kernel -- qkv never leaves the SM.  x_hi bf16 [crops*128][D] (D = 384 or 192, heads = D / 64), stats fp32 [crops*128]
 * [parts][2] (1 <= parts <= 4 partial (sum x, sum x^2) pairs per row), Wf = Wqkv * gamma bf16 [3D][D], c0 / c1 fp32 [3D]
 * (16-byte aligned), att bf16 [crops*128][D].  All device pointers. */
TT_API int tt_enc_qkv_attn_dev(const void* x_hi, const float* stats, int parts, const void* Wf, const float* c0, const float* c1,
                               void* att, int crops, int D, int heads, float eps, void* stream);
/* NHWC bf16 stride-1 "same" convolution as implicit GEMM; src1 may be NULL (else channel concat).
 * weight bf16 [Cout][taps][C0+C1]; out bf16 [batch][H][W][Cout]. */
TT_API int tt_conv_dev(const void* src0, int C0, const void* src1, int C1, int batch, int H, int W, int taps, int dil,
                const void* weight, const float* bias, int Cout, int relu, void* out, int BN, int resident,
                void* stream);
/* Kernel tests of the PARSeq attention family: each calls the launcher the engine calls.  All pointers are device
 * pointers; bf16 buffers are passed as void*.
 * tt_attn_enc_dev: encoder self attention, T = 128 tokens, head dim 64 (D = 64 * heads): qkv bf16 [crops*128][3D]
 *   (q | k | v, head-major inside each) -> out bf16 [crops*128][D]; onepass != 0 reads the S row from TMEM once. */
TT_API int tt_attn_enc_dev(const void* qkv, void* out, int crops, int D, int heads, int onepass, void* stream);
/* out fp32 [L][L][n_tok][heads] = q_table fp32 [L][D] . K of kv_table bf16 [L][n_tok][2D] (K | V), per head / sqrt(32) */
TT_API int tt_dec_score_table_dev(const float* q_table, const void* kv_table, int L, int n_tok, int D, int heads, float* out,
                                  void* stream);
/* Decoder self attention of query positions [p0, p0+np): key j of crop c is row (j, tokens[c][j]) of kv_table
 * bf16 [L][n_tok][2D]; q_table fp32 [L][D]; tokens int32 [n_crops][L].  refine == 0: keys j <= p (np == 1 with a
 * score table sc_table fp32 [L][L][n_tok][heads] takes the AR-step kernel, which alone honours active / n_act: output row
 * = slot, crop = active[slot], slots < *n_act); refine != 0: j != p+1 and j before the first eos_id among tokens[c][1..].
 * out bf16 [n_crops*np][D] (crop-major, then position).  active / n_act may be NULL. */
TT_API int tt_dec_self_attn_dev(int n_crops, int D, int heads, int L, int p0, int np, int refine, const int32_t* active,
                                const int32_t* n_act, const float* q_table, const float* sc_table, const void* kv_table,
                                const int32_t* tokens, int eos_id, int n_tok, void* out, void* stream);
/* Decoder cross attention over the 128 memory rows of each crop, no mask: q bf16 [n_crops*np][D], mem_kv bf16
 * [n_crops][128][2D] (K | V) -> out bf16 [n_crops*np][D].  active / n_act (may be NULL) as above, honoured when the
 * per-position kernel runs (np == 1, or D == 192): q / out rows by slot, memory by crop. */
TT_API int tt_dec_cross_attn_dev(int n_crops, int D, int heads, int L, int p0, int np, const int32_t* active,
                                 const int32_t* n_act, const void* q, const void* mem_kv, void* out, void* stream);
/* Kernel test of the rotation choice (tt_ocr_pages_oriented): ids int32 / pmax fp32 [n_words * n_candidates][26], crop
 * w * n_candidates + r being candidate r (angle angles[r], host array) of word w.  Writes the winner's ids_out [n_words][26],
 * pmax_out [n_words][26] (nullable) and angle_out [n_words].  Device pointers except angles. */
TT_API int tt_orient_select_dev(const int32_t* ids, const float* pmax, int n_words, const int32_t* angles, int n_candidates,
                                int32_t* ids_out, float* pmax_out, int32_t* angle_out, void* stream);
/* Kernel test of the contrast re-read's choice: for i < n_listed, the second read ids2 int32 / pmax2 fp32 [n_listed][26]
 * replaces ids / pmax [.][26] of word list[i] in place when its conf is strictly greater.  Device pointers. */
TT_API int tt_contrast_select_dev(int32_t* ids, float* pmax, const int32_t* list, int n_listed, const int32_t* ids2,
                                  const float* pmax2, void* stream);
/* Kernel test of the lexicon refinement head: the walk of lex's trie over device logits fp32 [n][26][95], every crop from
 * the root.  Writes ids_out int32 [n][26] and pmax_out fp32 [n][26] (nullable), device pointers. */
TT_API int tt_lexicon_walk_dev(const tt_lexicon* lex, const float* logits, int n, int32_t* ids_out, float* pmax_out,
                               void* stream);
/* Batched device-side post-processing (bench): maps_dev [batch][H][W][2] fp32. Returns total rects. */
TT_API int tt_postprocess_dev(tt_engine* e, const float* maps_dev, int batch, int H, int W, int* n_rects_total,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TUATARA_C_H */
