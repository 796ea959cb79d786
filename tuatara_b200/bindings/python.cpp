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

static tuatara::ImageView buffer_to_view(const py::array_t<unsigned char, py::array::c_style | py::array::forcecast>& input) {
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

static py::dict output_item_to_dict(const OutputItem& item) {  // python.cpp:36-41
  py::dict d;
  d["text"] = item.text;
  d["bbox"] = item.bbox;
  return d;
}

// conf is None for a word that was not recognised (ScoredItem::confidence == -1)
static py::dict scored_item_to_dict(const tuatara::ScoredItem& item) {
  py::dict d;
  d["text"] = item.text;
  d["bbox"] = item.bbox;
  d["conf"] = item.confidence < 0.f ? py::object(py::none()) : py::object(py::float_(item.confidence));
  d["det_score"] = item.detection_score;
  d["char_conf"] = item.char_confidence;
  return d;
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

// the items of an oriented call; as_scored: with conf / det_score / char_conf, else text / bbox only.  An empty
// rotation_info reads every word upright: angle 0.
static py::dict oriented_item_to_dict(const tuatara::ScoredItem& item, bool as_scored) {
  py::dict d = as_scored ? scored_item_to_dict(item) : output_item_to_dict(OutputItem{item.text, item.bbox});
  d["angle"] = item.angle;
  return d;
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

static py::list oriented_pages(const std::vector<tuatara::ImageView>& views, const std::string& weights_dir,
                               const std::string& output_dir, const FilterArgs& fa, const RotationArgs& ra, bool as_scored) {
  std::vector<std::vector<tuatara::ScoredItem>> pages;
  {
    py::gil_scoped_release release;
    pages = tuatara::image_to_data_oriented_batch(views, weights_dir, output_dir, ra.angles, fa.filters);
  }
  py::list result;
  for (const auto& page : pages) {
    py::list items;
    for (const auto& item : page) items.append(oriented_item_to_dict(item, as_scored));
    result.append(items);
  }
  return result;
}

static py::list image_to_data_wrapper(py::array_t<unsigned char, py::array::c_style | py::array::forcecast> image_data,
                                      std::string weights_dir, std::string output_dir, py::object allowlist,
                                      py::object blocklist, py::object rotation_info) {
  const tuatara::ImageView img = buffer_to_view(image_data);
  const FilterArgs fa = filter_args(allowlist, blocklist, 1, false);
  const RotationArgs ra = rotation_args(rotation_info);
  if (ra.given) {
    py::list pages = oriented_pages({img}, weights_dir, output_dir, fa, ra, false);
    return pages.empty() ? py::list() : py::list(pages[0]);
  }
  std::vector<OutputItem> items;
  {
    py::gil_scoped_release release;
    items = fa.filters.empty() ? image_to_data(img, weights_dir, output_dir)
                               : image_to_data(img, weights_dir, output_dir, fa.filters[0]);
  }
  py::list result;
  for (const auto& item : items) result.append(output_item_to_dict(item));
  return result;
}

static py::list images_to_data_wrapper(std::vector<py::array_t<unsigned char, py::array::c_style | py::array::forcecast>> images,
                                       std::string weights_dir, std::string output_dir, py::object allowlist,
                                       py::object blocklist, py::object rotation_info) {
  std::vector<tuatara::ImageView> views;
  for (auto& a : images) views.push_back(buffer_to_view(a));
  const FilterArgs fa = filter_args(allowlist, blocklist, views.size(), true);
  const RotationArgs ra = rotation_args(rotation_info);
  if (ra.given) return oriented_pages(views, weights_dir, output_dir, fa, ra, false);
  std::vector<std::vector<OutputItem>> pages;
  {
    py::gil_scoped_release release;
    pages = fa.filters.empty() ? tuatara::image_to_data_batch(views, weights_dir, output_dir)
                               : tuatara::image_to_data_batch(views, weights_dir, output_dir, fa.filters);
  }
  py::list result;
  for (const auto& page : pages) {
    py::list items;
    for (const auto& item : page) items.append(output_item_to_dict(item));
    result.append(items);
  }
  return result;
}

static py::list image_to_data_scored_wrapper(py::array_t<unsigned char, py::array::c_style | py::array::forcecast> image_data,
                                             std::string weights_dir, std::string output_dir, py::object allowlist,
                                             py::object blocklist, py::object rotation_info) {
  const tuatara::ImageView img = buffer_to_view(image_data);
  const FilterArgs fa = filter_args(allowlist, blocklist, 1, false);
  const RotationArgs ra = rotation_args(rotation_info);
  if (ra.given) {
    py::list pages = oriented_pages({img}, weights_dir, output_dir, fa, ra, true);
    return pages.empty() ? py::list() : py::list(pages[0]);
  }
  std::vector<tuatara::ScoredItem> items;
  {
    py::gil_scoped_release release;
    items = fa.filters.empty() ? tuatara::image_to_data_scored(img, weights_dir, output_dir)
                               : tuatara::image_to_data_scored(img, weights_dir, output_dir, fa.filters[0]);
  }
  py::list result;
  for (const auto& item : items) result.append(scored_item_to_dict(item));
  return result;
}

static py::list images_to_data_scored_wrapper(std::vector<py::array_t<unsigned char, py::array::c_style | py::array::forcecast>> images,
                                              std::string weights_dir, std::string output_dir, py::object allowlist,
                                              py::object blocklist, py::object rotation_info) {
  std::vector<tuatara::ImageView> views;
  for (auto& a : images) views.push_back(buffer_to_view(a));
  const FilterArgs fa = filter_args(allowlist, blocklist, views.size(), true);
  const RotationArgs ra = rotation_args(rotation_info);
  if (ra.given) return oriented_pages(views, weights_dir, output_dir, fa, ra, true);
  std::vector<std::vector<tuatara::ScoredItem>> pages;
  {
    py::gil_scoped_release release;
    pages = fa.filters.empty() ? tuatara::image_to_data_scored_batch(views, weights_dir, output_dir)
                               : tuatara::image_to_data_scored_batch(views, weights_dir, output_dir, fa.filters);
  }
  py::list result;
  for (const auto& page : pages) {
    py::list items;
    for (const auto& item : page) items.append(scored_item_to_dict(item));
    result.append(items);
  }
  return result;
}

PYBIND11_MODULE(pytuatara, m) {
  m.doc() = "Tuatara ocr";
  // allowlist / blocklist (keyword only): recognition only produces characters in allowlist and not in blocklist.
  // rotation_info (keyword only): angles from {90, 180, 270} at which each word is also read; items then carry "angle".
  m.def("image_to_data", &image_to_data_wrapper, py::arg("image"), py::arg("weights_dir"), py::arg("outputs_dir"), py::kw_only(),
        py::arg("allowlist") = py::none(), py::arg("blocklist") = py::none(), py::arg("rotation_info") = py::none(),
        "Extract text and bounding boxes from an image");
  m.def("images_to_data", &images_to_data_wrapper, py::arg("images"), py::arg("weights_dir"), py::arg("outputs_dir"), py::kw_only(),
        py::arg("allowlist") = py::none(), py::arg("blocklist") = py::none(), py::arg("rotation_info") = py::none(),
        "Batch variant: list of images -> list of per-page results");
  m.def("image_to_data_scored", &image_to_data_scored_wrapper, py::arg("image"), py::arg("weights_dir"), py::arg("outputs_dir"),
        py::kw_only(), py::arg("allowlist") = py::none(), py::arg("blocklist") = py::none(), py::arg("rotation_info") = py::none(),
        "image_to_data whose items also carry conf (word confidence 0..1, None when not recognised), det_score and char_conf");
  m.def("images_to_data_scored", &images_to_data_scored_wrapper, py::arg("images"), py::arg("weights_dir"), py::arg("outputs_dir"),
        py::kw_only(), py::arg("allowlist") = py::none(), py::arg("blocklist") = py::none(), py::arg("rotation_info") = py::none(),
        "Batch variant of image_to_data_scored");
}
