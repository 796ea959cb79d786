// Drop-in replacement for the reference's public header (/root/reference/tuatara.h:1-15).
//
// Same names, same return type: `OutputItem {text, bbox}` and
// `std::vector<OutputItem> image_to_data(image, weights_dir, outputs_dir)`.  The reference's
// signature takes a cv::Mat, which forces OpenCV on every caller; here the real parameter type is
// the OpenCV-free `tuatara::ImageView`, and when <opencv2/core.hpp> is available an inline
// cv::Mat overload forwards to it, so reference callers (examples/resume.cpp:9-11) compile
// unchanged.  Header-only on top of the C ABI (tuatara_c.h): link with -ltuatara_b200.
//
// Behavioural contract kept from tuatara.cpp:314-512: synchronous; one item per detected box in
// CCL label order; empty weights_dir / outputs_dir print to stderr and return {} (:315-323);
// engine errors print to stderr and return {} (the reference's soft-failure convention, :337-347).
// Differences, all deliberate: models are loaded once per (weights_dir) and cached instead of on
// every call (:333, :423); the caller's pixels are not modified (:349 swaps them in place);
// zero detections return {} instead of crashing in torch::cat (:485); a box whose boundingRect
// leaves the image is clamped instead of throwing (:416).
#ifndef TUATARA_H
#define TUATARA_H

#include <cstdint>
#include <cstdlib>
#include <iostream>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "tuatara_c.h"

#if defined(__has_include)
#if __has_include(<opencv2/core.hpp>)
#include <opencv2/core.hpp>
#define TUATARA_HAVE_OPENCV 1
#endif
#endif

struct OutputItem {
  std::string text;
  std::vector<float> bbox;  // [min_x, min_y, max_x, max_y]
};

namespace tuatara {

struct ImageView {  // 8-bit, 3 channels, row-major (what cv::imread / np.uint8[H,W,3] hold)
  const uint8_t* data = nullptr;
  int rows = 0, cols = 0, channels = 3;
  size_t step = 0;  // bytes per row; 0 = cols * channels
};

// An OutputItem with its scores (image_to_data_scored), all on a 0..1 scale; definitions at tt_item_scores.
struct ScoredItem {
  std::string text;
  std::vector<float> bbox;               // [min_x, min_y, max_x, max_y]
  float confidence = -1.f;               // word confidence; -1 when the word was not recognised
  float detection_score = 0.f;           // the box's maximum normalised text score (>= text_threshold)
  std::vector<float> char_confidence;    // one probability per character of text
  int angle = 0;                         // image_to_data_oriented: the candidate read (0, 90, 180, 270 ccw)
};

// Character filter (tt_char_filter, INTEGRATION.md section 7): recognition only produces characters that are in `allow`
// (when not null) and not in `block` (when not null).  E.g. CharFilter{"0123456789"} for digits only.
struct CharFilter {
  const char* allow = nullptr;
  const char* block = nullptr;
};

// A caller's word list (tt_lexicon, INTEGRATION.md section 9): every word recognised under it is one of its words.
// Build it once and pass it to as many calls as needed; it is immutable.  Move-only.  A list that tt_lexicon_create
// rejects gives !ok() and error() says why; the entry points print that and return {} when given it.
class Lexicon {
 public:
  Lexicon() = default;
  explicit Lexicon(const std::vector<std::string>& words) {
    std::vector<const char*> p;
    for (const std::string& w : words) p.push_back(w.c_str());
    if (tt_lexicon_create(p.data(), static_cast<int>(p.size()), &h_) != 0) {
      h_ = nullptr;
      err_ = tt_last_error();
    }
  }
  ~Lexicon() { if (h_) tt_lexicon_destroy(h_); }
  Lexicon(Lexicon&& o) noexcept : h_(o.h_), err_(std::move(o.err_)) { o.h_ = nullptr; }
  Lexicon& operator=(Lexicon&& o) noexcept {
    if (this != &o) {
      if (h_) tt_lexicon_destroy(h_);
      h_ = o.h_;
      err_ = std::move(o.err_);
      o.h_ = nullptr;
    }
    return *this;
  }
  Lexicon(const Lexicon&) = delete;
  Lexicon& operator=(const Lexicon&) = delete;
  bool ok() const { return h_ != nullptr; }
  const std::string& error() const { return err_; }
  const tt_lexicon* get() const { return h_; }

 private:
  tt_lexicon* h_ = nullptr;
  std::string err_ = "empty lexicon";
};

// The contrast re-read (tt_ocr_pages_contrast, INTEGRATION.md section 10): a word read with a confidence below
// contrast_ths from a low-contrast crop is read again from a contrast-stretched crop, and the more confident read is kept.
// The defaults are EasyOCR's readtext defaults.
struct Contrast {
  float contrast_ths = 0.1f;
  float adjust_contrast = 0.5f;
};

namespace detail {
inline tt_engine* engine_for(const std::string& weights_dir) {
  static std::mutex mu;
  static std::map<std::string, tt_engine*> cache;  // process-wide, keyed by weights_dir (SURVEY 8b)
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(weights_dir);
  if (it != cache.end()) return it->second;
  tt_engine* e = nullptr;
  // devices: the TT_DEVICES environment variable when set ("0,2" / "all"), else every visible GPU -- a batch is cut
  // into detection units that all of them pull from one queue; a single page simply runs on the first
  std::vector<int> devs;
  if (std::getenv("TT_DEVICES") == nullptr)
    for (int i = 0; i < tt_device_count(); ++i) devs.push_back(i);
  if (tt_engine_create(weights_dir.c_str(), devs.empty() ? nullptr : devs.data(), static_cast<int>(devs.size()), nullptr, &e) != 0)
    return nullptr;
  cache[weights_dir] = e;
  return e;
}
}  // namespace detail

namespace detail {
// The one path of every entry point: the checks, the soft failures ({} after printing the reason), one
// tt_ocr_pages_contrast call and the walk over its result.  Each item's scores are fetched when `scores`, its angle when
// rotation_info is not empty.  filters: none (empty), one for every page, or one per page.  lexicons (tt_lexicon
// handles): likewise; a null entry is a page without lexicon.  contrast: off (contrast_ths 0) unless given.
inline std::vector<std::vector<ScoredItem>> ocr_pages(const std::vector<ImageView>& images, const std::string& weights_dir,
                                                      const std::string& outputs_dir, bool scores,
                                                      const std::vector<CharFilter>& filters,
                                                      const std::vector<int>& rotation_info = {},
                                                      const std::vector<const tt_lexicon*>& lexicons = {},
                                                      const Contrast& contrast = Contrast{0.f, 0.5f}) {
  std::vector<std::vector<ScoredItem>> out;
  if (weights_dir.empty()) { std::cerr << "Please provide a value for weights_dir" << std::endl; return out; }
  if (outputs_dir.empty()) { std::cerr << "Please provide a value for outputs_dir" << std::endl; return out; }
  std::vector<tt_image> pages(images.size());
  for (size_t i = 0; i < images.size(); ++i) {
    const ImageView& v = images[i];
    if (!v.data || v.rows <= 0 || v.cols <= 0) { std::cerr << "Error reading image from file"; return out; }
    pages[i] = tt_image{v.data, v.rows, v.cols, v.channels, v.step ? v.step : static_cast<size_t>(v.cols) * v.channels};
  }
  tt_engine* e = engine_for(weights_dir);
  if (!e) { std::cerr << "error loading the models: " << tt_last_error() << std::endl; return out; }
  std::vector<tt_char_filter> f;
  for (const CharFilter& cf : filters) f.push_back(tt_char_filter{cf.allow, cf.block});
  tt_ocr_options opt = {};
  opt.with_scores = scores ? 1 : 0;
  tt_result* r = nullptr;
  if (tt_ocr_pages_contrast(e, pages.data(), static_cast<int>(pages.size()), &opt, f.data(), static_cast<int>(f.size()),
                            rotation_info.data(), static_cast<int>(rotation_info.size()), lexicons.data(),
                            static_cast<int>(lexicons.size()), contrast.contrast_ths, contrast.adjust_contrast, &r) != 0) {
    std::cerr << "tuatara: " << tt_last_error() << std::endl;
    return out;
  }
  out.resize(r->n_pages);
  for (int p = 0; p < r->n_pages; ++p)
    for (int k = 0; k < r->pages[p].n_items; ++k) {
      const tt_item& it = r->pages[p].items[k];
      ScoredItem s;
      s.text = it.text;
      s.bbox.assign(it.bbox, it.bbox + 4);
      const float* cc = nullptr;
      int n = 0;
      if ((scores && tt_item_scores(r, p, k, &s.confidence, &s.detection_score, &cc, &n) != 0) ||
          (!rotation_info.empty() && tt_item_angle(r, p, k, &s.angle) != 0)) {
        std::cerr << "tuatara: " << tt_last_error() << std::endl;
        tt_result_free(r);
        return std::vector<std::vector<ScoredItem>>{};
      }
      if (n > 0) s.char_confidence.assign(cc, cc + n);
      out[p].push_back(std::move(s));
    }
  tt_result_free(r);
  return out;
}

// ocr_pages with Lexicon objects (null: a page without lexicon); one that is not ok() prints its error and gives {}.
inline std::vector<std::vector<ScoredItem>> ocr_pages_lex(const std::vector<ImageView>& images, const std::string& weights_dir,
                                                          const std::string& outputs_dir, bool scores,
                                                          const std::vector<int>& rotation_info,
                                                          const std::vector<const Lexicon*>& lexicons) {
  std::vector<const tt_lexicon*> h;
  for (const Lexicon* l : lexicons) {
    if (l && !l->ok()) { std::cerr << "tuatara: " << l->error() << std::endl; return {}; }
    h.push_back(l ? l->get() : nullptr);
  }
  return ocr_pages(images, weights_dir, outputs_dir, scores, {}, rotation_info, h);
}

inline std::vector<std::vector<OutputItem>> unscored(std::vector<std::vector<ScoredItem>> pages) {
  std::vector<std::vector<OutputItem>> out(pages.size());
  for (size_t p = 0; p < pages.size(); ++p)
    for (ScoredItem& s : pages[p]) out[p].push_back(OutputItem{std::move(s.text), std::move(s.bbox)});
  return out;
}
}  // namespace detail

// Additive batch API: many pages in one call, spread over the engine's GPUs (all visible ones, or TT_DEVICES).
inline std::vector<std::vector<OutputItem>> image_to_data_batch(const std::vector<ImageView>& images,
                                                                const std::string& weights_dir,
                                                                const std::string& outputs_dir) {
  return detail::unscored(detail::ocr_pages(images, weights_dir, outputs_dir, false, {}));
}

// image_to_data_batch with character filters: `filters` holds one filter for every page, or one per page.
inline std::vector<std::vector<OutputItem>> image_to_data_batch(const std::vector<ImageView>& images,
                                                                const std::string& weights_dir,
                                                                const std::string& outputs_dir,
                                                                const std::vector<CharFilter>& filters) {
  return detail::unscored(detail::ocr_pages(images, weights_dir, outputs_dir, false, filters));
}

// image_to_data_batch with scores: same items (text, bbox) and the same soft failures, plus each item's scores.
inline std::vector<std::vector<ScoredItem>> image_to_data_scored_batch(const std::vector<ImageView>& images,
                                                                       const std::string& weights_dir,
                                                                       const std::string& outputs_dir) {
  return detail::ocr_pages(images, weights_dir, outputs_dir, true, {});
}

// image_to_data_scored_batch with character filters (one for every page, or one per page); the scores are renormalised
// over each page's allowed characters (tt_item_scores).
inline std::vector<std::vector<ScoredItem>> image_to_data_scored_batch(const std::vector<ImageView>& images,
                                                                       const std::string& weights_dir,
                                                                       const std::string& outputs_dir,
                                                                       const std::vector<CharFilter>& filters) {
  return detail::ocr_pages(images, weights_dir, outputs_dir, true, filters);
}

inline std::vector<ScoredItem> image_to_data_scored(const ImageView& image, const std::string& weights_dir,
                                                    const std::string& outputs_dir) {
  std::vector<std::vector<ScoredItem>> pages = image_to_data_scored_batch({image}, weights_dir, outputs_dir);
  return pages.empty() ? std::vector<ScoredItem>{} : pages[0];
}

inline std::vector<ScoredItem> image_to_data_scored(const ImageView& image, const std::string& weights_dir,
                                                    const std::string& outputs_dir, const CharFilter& filter) {
  std::vector<std::vector<ScoredItem>> pages =
      image_to_data_scored_batch({image}, weights_dir, outputs_dir, std::vector<CharFilter>{filter});
  return pages.empty() ? std::vector<ScoredItem>{} : pages[0];
}

// Rotation candidates (tt_ocr_pages_oriented, INTEGRATION.md section 8): every word is also read turned by each angle of
// rotation_info (90, 180, 270 degrees counter-clockwise) and the reading with the highest confidence is kept;
// ScoredItem::angle says which.  filters: none (empty), one for every page, or one per page.  Same soft failures as
// image_to_data; an invalid angle prints the error and returns {}.
inline std::vector<std::vector<ScoredItem>> image_to_data_oriented_batch(const std::vector<ImageView>& images,
                                                                         const std::string& weights_dir,
                                                                         const std::string& outputs_dir,
                                                                         const std::vector<int>& rotation_info,
                                                                         const std::vector<CharFilter>& filters = {}) {
  return detail::ocr_pages(images, weights_dir, outputs_dir, true, filters, rotation_info);
}

inline std::vector<ScoredItem> image_to_data_oriented(const ImageView& image, const std::string& weights_dir,
                                                      const std::string& outputs_dir, const std::vector<int>& rotation_info,
                                                      const CharFilter& filter = CharFilter()) {
  const bool filtered = filter.allow != nullptr || filter.block != nullptr;
  std::vector<std::vector<ScoredItem>> pages = image_to_data_oriented_batch(
      {image}, weights_dir, outputs_dir, rotation_info, filtered ? std::vector<CharFilter>{filter} : std::vector<CharFilter>{});
  return pages.empty() ? std::vector<ScoredItem>{} : pages[0];
}

// Lexicons (tt_ocr_pages_lexicon, INTEGRATION.md section 9): every recognised word is one of the lexicon's words.  One
// lexicon for every page, or one pointer per page (nullptr: the page reads as without lexicon).  Same soft failures.
inline std::vector<std::vector<OutputItem>> image_to_data_batch(const std::vector<ImageView>& images,
                                                                const std::string& weights_dir,
                                                                const std::string& outputs_dir, const Lexicon& lexicon) {
  return detail::unscored(detail::ocr_pages_lex(images, weights_dir, outputs_dir, false, {}, {&lexicon}));
}

inline std::vector<std::vector<OutputItem>> image_to_data_batch(const std::vector<ImageView>& images,
                                                                const std::string& weights_dir,
                                                                const std::string& outputs_dir,
                                                                const std::vector<const Lexicon*>& lexicons) {
  return detail::unscored(detail::ocr_pages_lex(images, weights_dir, outputs_dir, false, {}, lexicons));
}

inline std::vector<std::vector<ScoredItem>> image_to_data_scored_batch(const std::vector<ImageView>& images,
                                                                       const std::string& weights_dir,
                                                                       const std::string& outputs_dir,
                                                                       const Lexicon& lexicon) {
  return detail::ocr_pages_lex(images, weights_dir, outputs_dir, true, {}, {&lexicon});
}

inline std::vector<std::vector<ScoredItem>> image_to_data_scored_batch(const std::vector<ImageView>& images,
                                                                       const std::string& weights_dir,
                                                                       const std::string& outputs_dir,
                                                                       const std::vector<const Lexicon*>& lexicons) {
  return detail::ocr_pages_lex(images, weights_dir, outputs_dir, true, {}, lexicons);
}

inline std::vector<ScoredItem> image_to_data_scored(const ImageView& image, const std::string& weights_dir,
                                                    const std::string& outputs_dir, const Lexicon& lexicon) {
  std::vector<std::vector<ScoredItem>> pages = image_to_data_scored_batch({image}, weights_dir, outputs_dir, lexicon);
  return pages.empty() ? std::vector<ScoredItem>{} : pages[0];
}

inline std::vector<std::vector<ScoredItem>> image_to_data_oriented_batch(const std::vector<ImageView>& images,
                                                                         const std::string& weights_dir,
                                                                         const std::string& outputs_dir,
                                                                         const std::vector<int>& rotation_info,
                                                                         const Lexicon& lexicon) {
  return detail::ocr_pages_lex(images, weights_dir, outputs_dir, true, rotation_info, {&lexicon});
}

inline std::vector<std::vector<ScoredItem>> image_to_data_oriented_batch(const std::vector<ImageView>& images,
                                                                         const std::string& weights_dir,
                                                                         const std::string& outputs_dir,
                                                                         const std::vector<int>& rotation_info,
                                                                         const std::vector<const Lexicon*>& lexicons) {
  return detail::ocr_pages_lex(images, weights_dir, outputs_dir, true, rotation_info, lexicons);
}

inline std::vector<ScoredItem> image_to_data_oriented(const ImageView& image, const std::string& weights_dir,
                                                      const std::string& outputs_dir, const std::vector<int>& rotation_info,
                                                      const Lexicon& lexicon) {
  std::vector<std::vector<ScoredItem>> pages =
      image_to_data_oriented_batch({image}, weights_dir, outputs_dir, rotation_info, lexicon);
  return pages.empty() ? std::vector<ScoredItem>{} : pages[0];
}

// The contrast re-read (tt_ocr_pages_contrast, INTEGRATION.md section 10) on every page; Contrast() is EasyOCR's
// defaults.  Same soft failures; an invalid value prints the error and returns {}.
inline std::vector<std::vector<OutputItem>> image_to_data_batch(const std::vector<ImageView>& images,
                                                                const std::string& weights_dir,
                                                                const std::string& outputs_dir, const Contrast& contrast) {
  return detail::unscored(detail::ocr_pages(images, weights_dir, outputs_dir, false, {}, {}, {}, contrast));
}

inline std::vector<std::vector<ScoredItem>> image_to_data_scored_batch(const std::vector<ImageView>& images,
                                                                       const std::string& weights_dir,
                                                                       const std::string& outputs_dir,
                                                                       const Contrast& contrast) {
  return detail::ocr_pages(images, weights_dir, outputs_dir, true, {}, {}, {}, contrast);
}

inline std::vector<ScoredItem> image_to_data_scored(const ImageView& image, const std::string& weights_dir,
                                                    const std::string& outputs_dir, const Contrast& contrast) {
  std::vector<std::vector<ScoredItem>> pages = image_to_data_scored_batch({image}, weights_dir, outputs_dir, contrast);
  return pages.empty() ? std::vector<ScoredItem>{} : pages[0];
}

inline std::vector<std::vector<ScoredItem>> image_to_data_oriented_batch(const std::vector<ImageView>& images,
                                                                         const std::string& weights_dir,
                                                                         const std::string& outputs_dir,
                                                                         const std::vector<int>& rotation_info,
                                                                         const Contrast& contrast) {
  return detail::ocr_pages(images, weights_dir, outputs_dir, true, {}, rotation_info, {}, contrast);
}

inline std::vector<ScoredItem> image_to_data_oriented(const ImageView& image, const std::string& weights_dir,
                                                      const std::string& outputs_dir, const std::vector<int>& rotation_info,
                                                      const Contrast& contrast) {
  std::vector<std::vector<ScoredItem>> pages =
      image_to_data_oriented_batch({image}, weights_dir, outputs_dir, rotation_info, contrast);
  return pages.empty() ? std::vector<ScoredItem>{} : pages[0];
}

}  // namespace tuatara

inline std::vector<OutputItem> image_to_data(const tuatara::ImageView& image, std::string weights_dir,
                                             std::string outputs_dir) {
  auto pages = tuatara::image_to_data_batch({image}, weights_dir, outputs_dir);
  return pages.empty() ? std::vector<OutputItem>{} : pages[0];
}

// image_to_data with a character filter: every character of every item's text obeys it.
inline std::vector<OutputItem> image_to_data(const tuatara::ImageView& image, std::string weights_dir,
                                             std::string outputs_dir, const tuatara::CharFilter& filter) {
  auto pages = tuatara::image_to_data_batch({image}, weights_dir, outputs_dir, std::vector<tuatara::CharFilter>{filter});
  return pages.empty() ? std::vector<OutputItem>{} : pages[0];
}

// image_to_data with a lexicon: every item's text is one of its words.
inline std::vector<OutputItem> image_to_data(const tuatara::ImageView& image, std::string weights_dir,
                                             std::string outputs_dir, const tuatara::Lexicon& lexicon) {
  auto pages = tuatara::image_to_data_batch({image}, weights_dir, outputs_dir, lexicon);
  return pages.empty() ? std::vector<OutputItem>{} : pages[0];
}

// image_to_data with the contrast re-read: a low-confidence word on a low-contrast crop is read again, stretched.
inline std::vector<OutputItem> image_to_data(const tuatara::ImageView& image, std::string weights_dir,
                                             std::string outputs_dir, const tuatara::Contrast& contrast) {
  auto pages = tuatara::image_to_data_batch({image}, weights_dir, outputs_dir, contrast);
  return pages.empty() ? std::vector<OutputItem>{} : pages[0];
}

#ifdef TUATARA_HAVE_OPENCV
// The reference's exact signature (tuatara.h:13).
inline std::vector<OutputItem> image_to_data(cv::Mat image, std::string weights_dir, std::string outputs_dir) {
  if (image.empty()) { std::cerr << "Error reading image from file"; return {}; }  // tuatara.cpp:344-347
  tuatara::ImageView v;
  v.data = image.data; v.rows = image.rows; v.cols = image.cols; v.channels = image.channels(); v.step = image.step;
  return image_to_data(v, weights_dir, outputs_dir);
}
#endif

#endif  // TUATARA_H
