// Bit-exact restatements of cv::resize(INTER_LINEAR, 8UC3) as used by the reference:
//   page:  resize_aspect_ratio (tuatara.cpp:206-234) + channel swap (:349) + zero pad to x32
//   crops: image(boundingRect) -> cv::resize(128x32) -> channel swap back (tuatara.cpp:416,440-441)
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tt {

// src: device u8 HWC (row pitch `src_step` bytes) exactly as the caller passed it.
// dst: device u8 [H32][W32][3], channels swapped (c2,c1,c0), resized region [0,th)x[0,tw), rest 0.
cudaError_t page_resize_pad(const uint8_t* src, int src_h, int src_w, size_t src_step, uint8_t* dst, int th, int tw,
                            int h32, int w32, cudaStream_t s);

// u8 [B][H][W][3] -> bf16 [B][H][W][32]: the 3x3 neighbourhood (zero padded) of every pixel, k = tap*3 + c,
// k 27..31 zero -- conv1_1 as a K=32 GEMM.  Values are the raw integers 0..255 (exact in bf16);
// the /255 of tuatara.cpp:370 is folded into conv1_1's weights.
cudaError_t page_im2col(const uint8_t* img, int batch, int H, int W, __nv_bfloat16* out, cudaStream_t s);

struct CropBox {
  int page;        // index into the page table
  int x, y, w, h;  // source rectangle, already clamped to the image; w or h == 0 -> black crop
};
struct PageRef {
  const uint8_t* data;
  int rows, cols;
  size_t step;
};

// One launch for all boxes of all pages.  out_u8 (optional): [N][32][128][3] in the caller's channel
// order (what PARSeq is fed before /255).  out_patches (optional): bf16 [N*128][96], row = crop*128 +
// (y/4)*16 + x/8, k = c*32 + (y%4)*8 + x%8 -- the patch-embed GEMM's A operand, raw integers 0..255.
cudaError_t crop_resize(const PageRef* pages_dev, const CropBox* boxes_dev, int n_boxes, uint8_t* out_u8,
                        __nv_bfloat16* out_patches, cudaStream_t s);

// Rotation candidates (tt_ocr_pages_oriented): crop b is box b / R (boxes_dev holds n_crops / R boxes) turned rot_dev[b]
// quarter turns counter-clockwise (0..3) before the resize, cv::resize(cv::rotate(roi, code), (128, 32)) bit for bit.
// Outputs as crop_resize; rot_dev[b] == 0 gives crop_resize's bytes.
cudaError_t crop_resize_rot(const PageRef* pages_dev, const CropBox* boxes_dev, const uint8_t* rot_dev, int R, int n_crops,
                            uint8_t* out_u8, __nv_bfloat16* out_patches, cudaStream_t s);

// Opt-in rectified crops (tt_config.rectify; the TODO at tuatara.cpp:411-415): every crop is the 128 x 32 perspective
// warp of its box's quadrilateral, sampled the way cv::warpPerspective(INTER_LINEAR, BORDER_REPLICATE) samples it
// (source coordinates in double, rounded to 1/32 pixel, 15-bit fixed-point bilinear weights).
struct WarpBox {
  int page;        // index into the page table; < 0 -> black crop
  int pad_;
  double m[9];     // output pixel (x, y, 1) -> source (X, Y, W), the inverted cv::getPerspectiveTransform matrix
};
cudaError_t crop_warp(const PageRef* pages_dev, const WarpBox* boxes_dev, int n_boxes, uint8_t* out_u8,
                      __nv_bfloat16* out_patches, cudaStream_t s);

}  // namespace tt
