#include "detect.h"

#include <algorithm>

namespace tt {

bool collect_boxes(const uint8_t* block, int comp_cap, int row_cap, int H, int W, const tt_config& cfg,
                   std::vector<DetBox>* out) {
  const PostHeader* h = reinterpret_cast<const PostHeader*>(block);
  if (h->overflow || h->n_comp > comp_cap || h->n_rows > row_cap) return false;
  const PostComp* comps = reinterpret_cast<const PostComp*>(block + sizeof(PostHeader));
  const PostRow* rows = reinterpret_cast<const PostRow*>(block + sizeof(PostHeader) + sizeof(PostComp) * comp_cap);
  std::vector<Pt2i> scratch;
  for (int j = 0; j < h->n_comp; ++j) {  // k = j + 1 in cv label numbering, tuatara.cpp:146
    const PostComp& c = comps[j];
    CompIn ci{c.left, c.top, c.right, c.bottom, c.area, c.max_text};
    RotatedRect rr;
    if (!component_rect(ci, reinterpret_cast<const int*>(rows + c.row_off), W, H, cfg.min_area, cfg.text_threshold,
                        &rr, &scratch))
      continue;
    out->push_back(DetBox{j + 1, rr, c.max_text});
  }
  return true;
}

void resize_plan(int rows, int cols, float canvas_size, float mag_ratio, int* th, int* tw, int* h32, int* w32,
                 float* ratio_out) {
  const int m = std::max(rows, cols);
  float target_size = mag_ratio * static_cast<float>(m);  // tuatara.cpp:211
  if (target_size > canvas_size) target_size = canvas_size;  // :213-215
  const float ratio = target_size / static_cast<float>(m);  // :217
  const int target_h = static_cast<int>(static_cast<float>(rows) * ratio);  // :219
  const int target_w = static_cast<int>(static_cast<float>(cols) * ratio);  // :220
  *th = target_h;
  *tw = target_w;
  *h32 = target_h % 32 != 0 ? target_h + (32 - target_h % 32) : target_h;  // :225
  *w32 = target_w % 32 != 0 ? target_w + (32 - target_w % 32) : target_w;  // :226
  *ratio_out = ratio;
}

}  // namespace tt
