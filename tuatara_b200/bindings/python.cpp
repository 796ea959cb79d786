// pytuatara: the reference's Python module (bindings/python.cpp:1-58) re-created on the B200 path.
// Same module name, function name, keyword names and return shape:
//   pytuatara.image_to_data(image, weights_dir, outputs_dir) -> list[dict(text=str, bbox=list[float])]
// The reference copies the buffer into a cv::Mat (buffer_to_mat, :12-28); here the numpy buffer is
// passed straight to the C ABI as an ImageView.
#include <memory>

#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "tuatara.h"

namespace py = pybind11;

using Image = py::array_t<unsigned char, py::array::c_style | py::array::forcecast>;

static tuatara::ImageView buffer_to_view(const Image& input) {
  py::buffer_info buf = input.request();
  if (buf.ndim != 3) throw std::runtime_error("Input array should have 3 dimensions");  // python.cpp:15-17
  tuatara::ImageView v;
  v.data = static_cast<const uint8_t*>(buf.ptr);
  v.rows = static_cast<int>(buf.shape[0]);
  v.cols = static_cast<int>(buf.shape[1]);
  v.channels = static_cast<int>(buf.shape[2]);
  v.step = static_cast<size_t>(buf.strides[0]);
  if (v.channels != 3) throw std::runtime_error("Input array should have 3 channels");
  return v;
}

// rotation_info keyword -> angles (None: no rotation candidates)
struct RotationArgs {
  bool given = false;
  std::vector<int> angles;
};

static RotationArgs rotation_args(const py::object& rotation_info) {
  RotationArgs ra;
  if (rotation_info.is_none()) return ra;
  if (py::isinstance<py::str>(rotation_info) || !py::isinstance<py::iterable>(rotation_info))
    throw py::type_error("rotation_info: expected an iterable of ints from {90, 180, 270}");
  ra.given = true;
  for (const py::handle& v : rotation_info) {
    if (!py::isinstance<py::int_>(v) || py::isinstance<py::bool_>(v)) throw py::type_error("rotation_info: expected ints");
    ra.angles.push_back(v.cast<int>());
  }
  return ra;
}

// allowlist / blocklist keywords -> character filters (tuatara::CharFilter).  Each is None, a str (every page) or, for
// the batch functions, a list with one str or None per page.  No filter at all when both are None.
struct FilterArgs {
  std::vector<std::unique_ptr<std::string>> keep;   // the strings the filters point into
  std::vector<tuatara::CharFilter> filters;          // empty: no filter
};

static const char* filter_str(const py::handle& v, FilterArgs* fa, const char* name) {
  if (v.is_none()) return nullptr;
  if (!py::isinstance<py::str>(v)) throw py::type_error(std::string(name) + ": expected str or None");
  fa->keep.emplace_back(new std::string(v.cast<std::string>()));
  return fa->keep.back()->c_str();
}

static FilterArgs filter_args(const py::object& allow, const py::object& block, size_t n_pages, bool batch) {
  FilterArgs fa;
  if (allow.is_none() && block.is_none()) return fa;
  const bool al = batch && py::isinstance<py::list>(allow), bl = batch && py::isinstance<py::list>(block);
  if (al && py::len(allow) != n_pages)
    throw py::value_error("allowlist: expected one entry per page (" + std::to_string(n_pages) + "), got " +
                          std::to_string(py::len(allow)));
  if (bl && py::len(block) != n_pages)
    throw py::value_error("blocklist: expected one entry per page (" + std::to_string(n_pages) + "), got " +
                          std::to_string(py::len(block)));
  const size_t n = (al || bl) ? n_pages : 1;
  for (size_t i = 0; i < n; ++i) {
    tuatara::CharFilter f;
    f.allow = filter_str(al ? py::handle(allow.cast<py::list>()[i]) : py::handle(allow), &fa, "allowlist");
    f.block = filter_str(bl ? py::handle(block.cast<py::list>()[i]) : py::handle(block), &fa, "blocklist");
    fa.filters.push_back(f);
  }
  return fa;
}

// lexicon keyword -> tt_lexicon handles (empty: no lexicon).  A tuatara_b200.Lexicon (its handle is borrowed) or an
// iterable of str is one lexicon for every page; for the batch functions a list with one entry per page, each None or one
// of those, is a lexicon per page (a list of str alone is always one word list).
struct LexiconArgs {
  std::vector<std::unique_ptr<tuatara::Lexicon>> keep;   // lexicons built here from word lists
  std::vector<const tt_lexicon*> handles;
};

static bool is_word_list(const py::handle& v) {
  if (py::isinstance<py::str>(v) || py::isinstance<py::bytes>(v) || !py::isinstance<py::iterable>(v)) return false;
  for (const py::handle& w : v)
    if (!py::isinstance<py::str>(w)) return false;
  return true;
}

static const tt_lexicon* lexicon_handle(const py::handle& v, LexiconArgs* la) {
  if (v.is_none()) return nullptr;
  if (py::hasattr(v, "_h") && py::hasattr(v, "info")) {   // tuatara_b200.Lexicon
    const py::object h = v.attr("_h").attr("value");
    if (h.is_none()) throw py::value_error("lexicon: the Lexicon was closed");
    return reinterpret_cast<const tt_lexicon*>(h.cast<uintptr_t>());
  }
  if (!is_word_list(v)) throw py::type_error("lexicon: expected a Lexicon, an iterable of str, or None");
  std::vector<std::string> words;
  for (const py::handle& w : v) words.push_back(w.cast<std::string>());
  la->keep.emplace_back(new tuatara::Lexicon(words));
  if (!la->keep.back()->ok()) throw py::value_error(la->keep.back()->error());
  return la->keep.back()->get();
}

static LexiconArgs lexicon_args(const py::object& lexicon, size_t n_pages, bool batch) {
  LexiconArgs la;
  if (lexicon.is_none()) return la;
  if (batch && py::isinstance<py::list>(lexicon) && !is_word_list(lexicon)) {
    if (py::len(lexicon) != n_pages)
      throw py::value_error("lexicon: expected one entry per page (" + std::to_string(n_pages) + "), got " +
                            std::to_string(py::len(lexicon)));
    for (const py::handle& v : lexicon) la.handles.push_back(lexicon_handle(v, &la));
    return la;
  }
  if (py::isinstance<py::str>(lexicon)) throw py::type_error("lexicon: expected a Lexicon or an iterable of str, not a str");
  la.handles.push_back(lexicon_handle(lexicon, &la));
  return la;
}

// One item as a dict: text and bbox; conf (None for a word that was not recognised, ScoredItem::confidence == -1),
// det_score and char_conf when scored; angle when rotation_info was given (0 for every word when it is empty).
static py::dict item_to_dict(const tuatara::ScoredItem& item, bool scored, bool angle) {  // python.cpp:36-41
  py::dict d;
  d["text"] = item.text;
  d["bbox"] = item.bbox;
  if (scored) {
    d["conf"] = item.confidence < 0.f ? py::object(py::none()) : py::object(py::float_(item.confidence));
    d["det_score"] = item.detection_score;
    d["char_conf"] = item.char_confidence;
  }
  if (angle) d["angle"] = item.angle;
  return d;
}

// The four functions' one path -> a list of pages of item dicts.  batch: allowlist / blocklist may hold one entry per page.
static py::list ocr_pages(const std::vector<tuatara::ImageView>& views, bool batch, const std::string& weights_dir,
                          const std::string& output_dir, const py::object& allowlist, const py::object& blocklist,
                          const py::object& rotation_info, const py::object& lexicon, float contrast_ths,
                          float adjust_contrast, bool scored) {
  const FilterArgs fa = filter_args(allowlist, blocklist, views.size(), batch);
  const RotationArgs ra = rotation_args(rotation_info);
  const LexiconArgs la = lexicon_args(lexicon, views.size(), batch);
  std::vector<std::vector<tuatara::ScoredItem>> pages;
  {
    py::gil_scoped_release release;
    pages = tuatara::detail::ocr_pages(views, weights_dir, output_dir, scored, fa.filters, ra.angles, la.handles,
                                       tuatara::Contrast{contrast_ths, adjust_contrast});
  }
  py::list result;
  for (const auto& page : pages) {
    py::list items;
    for (const auto& item : page) items.append(item_to_dict(item, scored, ra.given));
    result.append(items);
  }
  return result;
}

// image_to_data / image_to_data_scored: page 0, or [] after a soft failure
template <bool kScored>
static py::list image_wrapper(Image image_data, std::string weights_dir, std::string output_dir, py::object allowlist,
                              py::object blocklist, py::object rotation_info, py::object lexicon, float contrast_ths,
                              float adjust_contrast) {
  py::list pages = ocr_pages({buffer_to_view(image_data)}, false, weights_dir, output_dir, allowlist, blocklist,
                             rotation_info, lexicon, contrast_ths, adjust_contrast, kScored);
  return pages.empty() ? py::list() : py::list(pages[0]);
}

// images_to_data / images_to_data_scored
template <bool kScored>
static py::list images_wrapper(std::vector<Image> images, std::string weights_dir, std::string output_dir,
                               py::object allowlist, py::object blocklist, py::object rotation_info, py::object lexicon,
                               float contrast_ths, float adjust_contrast) {
  std::vector<tuatara::ImageView> views;
  for (auto& a : images) views.push_back(buffer_to_view(a));
  return ocr_pages(views, true, weights_dir, output_dir, allowlist, blocklist, rotation_info, lexicon, contrast_ths,
                   adjust_contrast, kScored);
}

PYBIND11_MODULE(pytuatara, m) {
  m.doc() = "Tuatara ocr";
  // allowlist / blocklist (keyword only): recognition only produces characters in allowlist and not in blocklist.
  // rotation_info (keyword only): angles from {90, 180, 270} at which each word is also read; items then carry "angle".
  // lexicon (keyword only): every recognised word is one of a word list (a tuatara_b200.Lexicon or an iterable of str).
  // contrast_ths / adjust_contrast (keyword only): a word read with a confidence below contrast_ths from a crop whose
  // contrast is below adjust_contrast is read again from a contrast-stretched crop (0 = off; EasyOCR uses 0.1 / 0.5).
  m.def("image_to_data", &image_wrapper<false>, py::arg("image"), py::arg("weights_dir"), py::arg("outputs_dir"), py::kw_only(),
        py::arg("allowlist") = py::none(), py::arg("blocklist") = py::none(), py::arg("rotation_info") = py::none(),
        py::arg("lexicon") = py::none(), py::arg("contrast_ths") = 0.0f, py::arg("adjust_contrast") = 0.5f,
        "Extract text and bounding boxes from an image");
  m.def("images_to_data", &images_wrapper<false>, py::arg("images"), py::arg("weights_dir"), py::arg("outputs_dir"), py::kw_only(),
        py::arg("allowlist") = py::none(), py::arg("blocklist") = py::none(), py::arg("rotation_info") = py::none(),
        py::arg("lexicon") = py::none(), py::arg("contrast_ths") = 0.0f, py::arg("adjust_contrast") = 0.5f,
        "Batch variant: list of images -> list of per-page results");
  m.def("image_to_data_scored", &image_wrapper<true>, py::arg("image"), py::arg("weights_dir"), py::arg("outputs_dir"),
        py::kw_only(), py::arg("allowlist") = py::none(), py::arg("blocklist") = py::none(), py::arg("rotation_info") = py::none(),
        py::arg("lexicon") = py::none(), py::arg("contrast_ths") = 0.0f, py::arg("adjust_contrast") = 0.5f,
        "image_to_data whose items also carry conf (word confidence 0..1, None when not recognised), det_score and char_conf");
  m.def("images_to_data_scored", &images_wrapper<true>, py::arg("images"), py::arg("weights_dir"), py::arg("outputs_dir"),
        py::kw_only(), py::arg("allowlist") = py::none(), py::arg("blocklist") = py::none(), py::arg("rotation_info") = py::none(),
        py::arg("lexicon") = py::none(), py::arg("contrast_ths") = 0.0f, py::arg("adjust_contrast") = 0.5f,
        "Batch variant of image_to_data_scored");
}
