// Host half of get_detected_boxes (tuatara.cpp:146-201): turns the GPU's per-component stats and
// row extents (postprocess.cuh) into RotatedRects, in CCL label order.
#pragma once
#include <vector>

#include "geometry.h"
#include "postprocess.cuh"
#include "tuatara_c.h"

namespace tt {

struct DetBox {
  int label;        // cv label of the component (1-based)
  RotatedRect rect; // in score-map coordinates
  float score;      // the component's maximum normalised text score (>= text_threshold, tuatara.cpp:151-154)
};

// `block` = one page's result block copied from PostWorkspace::result (header | comps | rows).
// Returns false if the block overflowed its capacities (caller re-runs with larger ones).
bool collect_boxes(const uint8_t* block, int comp_cap, int row_cap, int H, int W, const tt_config& cfg,
                   std::vector<DetBox>* out);

// tuatara.cpp:211-226 in fp32.
void resize_plan(int rows, int cols, float canvas_size, float mag_ratio, int* th, int* tw, int* h32, int* w32,
                 float* ratio);

}  // namespace tt
