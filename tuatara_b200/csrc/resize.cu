// cv::resize INTER_LINEAR for 8-bit images, restated bit-exactly (OpenCV 4.x resize.cpp:
// ResizeLinear + HResizeLinear<uchar,int,short,2048> + VResizeLinear<uchar,int,short,FixedPtCast<..,22>>).
//
// Per axis:  f = (float)((d + 0.5) * scale - 0.5) in double, s = floor(f), f -= s.
//   horizontal: s < 0 -> s = 0, f = 0;  s >= W-1 -> s = W-1, f = 0
//   vertical:   f kept, both row indices clamped to [0, H-1]
//   coefficients: c1 = rint(f * 2048), c0 = rint((1.f - f) * 2048)   (int16)
//   horizontal pass: S = I[s] * c0 + I[s+1] * c1                      (int32)
//   vertical pass:   out = (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2
// scale = 1.0 / ((double)dst / src).  The exact-2x INTER_AREA shortcut OpenCV takes gives the same
// integers as this rule, and equal sizes reduce to a copy.
#include "resize.cuh"

#include "common.h"

namespace tt {

namespace {

struct AxisCoef { int s; int c0, c1; };

__device__ __forceinline__ AxisCoef axis_coef(int d, double scale, int src_len, bool horizontal) {
  const double m = __dmul_rn(static_cast<double>(d) + 0.5, scale);
  float f = static_cast<float>(__dadd_rn(m, -0.5));
  int s = __float2int_rd(f);
  f = __fsub_rn(f, static_cast<float>(s));
  if (horizontal) {
    if (s < 0) { s = 0; f = 0.f; }
    if (s >= src_len - 1) { s = src_len - 1; f = 0.f; }
  }
  AxisCoef a;
  a.s = s;
  a.c0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f));
  a.c1 = __float2int_rn(__fmul_rn(f, 2048.f));
  return a;
}

__device__ __forceinline__ int vblend(int S0, int S1, int b0, int b1) {
  return (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2;
}

__global__ void k_page_resize(const uint8_t* __restrict__ src, int sh, int sw, size_t step, uint8_t* __restrict__ dst,
                              int th, int tw, int h32, int w32, double scale_x, double scale_y) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= w32) return;
  uint8_t* o = dst + (static_cast<size_t>(y) * w32 + x) * 3;
  if (y >= th || x >= tw) { o[0] = 0; o[1] = 0; o[2] = 0; return; }
  const AxisCoef ax = axis_coef(x, scale_x, sw, true);
  const AxisCoef ay = axis_coef(y, scale_y, sh, false);
  const int y0 = min(max(ay.s, 0), sh - 1), y1 = min(max(ay.s + 1, 0), sh - 1);
  const int x1 = min(ax.s + 1, sw - 1);
  const uint8_t* r0 = src + y0 * step;
  const uint8_t* r1 = src + y1 * step;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int S0 = r0[ax.s * 3 + c] * ax.c0 + r0[x1 * 3 + c] * ax.c1;
    const int S1 = r1[ax.s * 3 + c] * ax.c0 + r1[x1 * 3 + c] * ax.c1;
    o[2 - c] = static_cast<uint8_t>(vblend(S0, S1, ay.c0, ay.c1));  // channel swap, tuatara.cpp:349
  }
}

__global__ void k_im2col(const uint8_t* __restrict__ img, int H, int W, __nv_bfloat16* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y, n = blockIdx.z;
  if (x >= W) return;
  const uint8_t* base = img + static_cast<size_t>(n) * H * W * 3;
  __align__(16) __nv_bfloat16 v[32];
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const int yy = y + t / 3 - 1, xx = x + t % 3 - 1;
    const bool in = yy >= 0 && yy < H && xx >= 0 && xx < W;
    const uint8_t* p = base + (static_cast<size_t>(yy) * W + xx) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) v[t * 3 + c] = __float2bfloat16(in ? static_cast<float>(p[c]) : 0.f);
  }
#pragma unroll
  for (int k = 27; k < 32; ++k) v[k] = __float2bfloat16(0.f);
  uint4* o = reinterpret_cast<uint4*>(out + ((static_cast<size_t>(n) * H + y) * W + x) * 32);
  const uint4* vv = reinterpret_cast<const uint4*>(v);
#pragma unroll
  for (int i = 0; i < 4; ++i) o[i] = vv[i];
}

// grid (32 output rows, n_boxes), 128 threads = one output pixel each.  The two source rows an
// output row blends are staged in shared memory with coalesced loads when they fit.
constexpr int kCropStage = 12 * 1024;  // bytes per staged source row

__global__ void __launch_bounds__(128) k_crop(const PageRef* __restrict__ pages, const CropBox* __restrict__ boxes,
                                              uint8_t* __restrict__ out_u8, __nv_bfloat16* __restrict__ out_patch) {
  __shared__ uint8_t rows[2][kCropStage];
  const int dy = blockIdx.x, b = blockIdx.y, dx = threadIdx.x;
  const CropBox box = boxes[b];
  int val[3] = {0, 0, 0};
  if (box.w > 0 && box.h > 0) {
    const PageRef pg = pages[box.page];
    const double scale_x = 1.0 / (128.0 / static_cast<double>(box.w));
    const double scale_y = 1.0 / (32.0 / static_cast<double>(box.h));
    const AxisCoef ay = axis_coef(dy, scale_y, box.h, false);
    const int y0 = min(max(ay.s, 0), box.h - 1), y1 = min(max(ay.s + 1, 0), box.h - 1);
    const uint8_t* g0 = pg.data + static_cast<size_t>(box.y + y0) * pg.step + static_cast<size_t>(box.x) * 3;
    const uint8_t* g1 = pg.data + static_cast<size_t>(box.y + y1) * pg.step + static_cast<size_t>(box.x) * 3;
    const int nbytes = box.w * 3;
    const bool staged = nbytes <= kCropStage;
    if (staged) {
      for (int i = threadIdx.x; i < nbytes; i += blockDim.x) { rows[0][i] = g0[i]; rows[1][i] = g1[i]; }
      __syncthreads();
    }
    const uint8_t* r0 = staged ? rows[0] : g0;
    const uint8_t* r1 = staged ? rows[1] : g1;
    const AxisCoef ax = axis_coef(dx, scale_x, box.w, true);
    const int x1 = min(ax.s + 1, box.w - 1);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int S0 = r0[ax.s * 3 + c] * ax.c0 + r0[x1 * 3 + c] * ax.c1;
      const int S1 = r1[ax.s * 3 + c] * ax.c0 + r1[x1 * 3 + c] * ax.c1;
      val[c] = vblend(S0, S1, ay.c0, ay.c1);
    }
  }
  if (out_u8 != nullptr) {
    uint8_t* o = out_u8 + ((static_cast<size_t>(b) * 32 + dy) * 128 + dx) * 3;
    o[0] = static_cast<uint8_t>(val[0]); o[1] = static_cast<uint8_t>(val[1]); o[2] = static_cast<uint8_t>(val[2]);
  }
  if (out_patch != nullptr) {
    const size_t row = static_cast<size_t>(b) * 128 + (dy >> 2) * 16 + (dx >> 3);
    __nv_bfloat16* o = out_patch + row * 96 + (dy & 3) * 8 + (dx & 7);
#pragma unroll
    for (int c = 0; c < 3; ++c) o[c * 32] = __float2bfloat16(static_cast<float>(val[c]));
  }
}

// Rotation candidates (INTEGRATION.md section 8): crop b is box b / R turned rot[b] quarter turns counter-clockwise
// before the resize, cv::resize(cv::rotate(roi, code), (128, 32)).  The turned ROI T is rw x rh = w x h (0, 180) or
// h x w (90, 270) and gets k_crop's coefficients for that size.  T's pixel (ty, tx) is the source pixel
//   0: (ty, tx)   90: (tx, w-1-ty)   180: (h-1-ty, w-1-tx)   270: (h-1-tx, ty)
// so each output row blends two "lines" of the source (rows for 0 / 180, columns for 90 / 270), and pixel k of a line
// sits at line + k * stride (stride 3, -3, step or -step bytes).  Both lines are staged in shared memory in T's order:
// coalesced for rows, one source row per three threads for columns.  grid (32, n_crops), 128 threads, as k_crop.
__global__ void __launch_bounds__(128) k_crop_rot(const PageRef* __restrict__ pages, const CropBox* __restrict__ boxes,
                                                  const uint8_t* __restrict__ rot, int R, uint8_t* __restrict__ out_u8,
                                                  __nv_bfloat16* __restrict__ out_patch) {
  __shared__ uint8_t rows[2][kCropStage];
  const int dy = blockIdx.x, b = blockIdx.y, dx = threadIdx.x;
  const CropBox box = boxes[b / R];
  const int q = rot[b] & 3;
  int val[3] = {0, 0, 0};
  if (box.w > 0 && box.h > 0) {
    const PageRef pg = pages[box.page];
    const bool turned = q & 1;
    const int rw = turned ? box.h : box.w, rh = turned ? box.w : box.h;
    const double scale_x = 1.0 / (128.0 / static_cast<double>(rw));
    const double scale_y = 1.0 / (32.0 / static_cast<double>(rh));
    const AxisCoef ay = axis_coef(dy, scale_y, rh, false);
    const int ty[2] = {min(max(ay.s, 0), rh - 1), min(max(ay.s + 1, 0), rh - 1)};
    const long long step = static_cast<long long>(pg.step);
    const uint8_t* org = pg.data + static_cast<long long>(box.y) * step + static_cast<long long>(box.x) * 3;
    const long long stride = q == 0 ? 3 : q == 1 ? step : q == 2 ? -3 : -step;
    const uint8_t* line[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int t = ty[j];
      line[j] = org + (q == 0 ? t * step
                     : q == 1 ? static_cast<long long>(box.w - 1 - t) * 3
                     : q == 2 ? (box.h - 1 - t) * step + static_cast<long long>(box.w - 1) * 3
                              : static_cast<long long>(t) * 3 + (box.h - 1) * step);
    }
    const int nbytes = rw * 3;
    const bool staged = nbytes <= kCropStage;
    if (staged) {
      for (int i = threadIdx.x; i < nbytes; i += blockDim.x) {
        const long long off = (i / 3) * stride + i % 3;
        rows[0][i] = line[0][off];
        rows[1][i] = line[1][off];
      }
      __syncthreads();
    }
    const AxisCoef ax = axis_coef(dx, scale_x, rw, true);
    const int x1 = min(ax.s + 1, rw - 1);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      int v[2][2];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        v[j][0] = staged ? rows[j][ax.s * 3 + c] : line[j][ax.s * stride + c];
        v[j][1] = staged ? rows[j][x1 * 3 + c] : line[j][x1 * stride + c];
      }
      const int S0 = v[0][0] * ax.c0 + v[0][1] * ax.c1;
      const int S1 = v[1][0] * ax.c0 + v[1][1] * ax.c1;
      val[c] = vblend(S0, S1, ay.c0, ay.c1);
    }
  }
  if (out_u8 != nullptr) {
    uint8_t* o = out_u8 + ((static_cast<size_t>(b) * 32 + dy) * 128 + dx) * 3;
    o[0] = static_cast<uint8_t>(val[0]); o[1] = static_cast<uint8_t>(val[1]); o[2] = static_cast<uint8_t>(val[2]);
  }
  if (out_patch != nullptr) {
    const size_t row = static_cast<size_t>(b) * 128 + (dy >> 2) * 16 + (dx >> 3);
    __nv_bfloat16* o = out_patch + row * 96 + (dy & 3) * 8 + (dx & 7);
#pragma unroll
    for (int c = 0; c < 3; ++c) o[c * 32] = __float2bfloat16(static_cast<float>(val[c]));
  }
}

// grid (32, n), 128 threads: one output row of one crop per block, as k_crop.  Arithmetic follows
// cv::warpPerspective's block loop (64 x 16 blocks for a 128 x 32 destination): X0 = M0*x + M1*y + M2 at the block
// origin, then (X0 + M0*x1) * (32 / W) per pixel, no fused multiply-add (the CPU code has none either).
__global__ void __launch_bounds__(128) k_crop_warp(const PageRef* __restrict__ pages, const WarpBox* __restrict__ boxes,
                                                   uint8_t* __restrict__ out_u8, __nv_bfloat16* __restrict__ out_patch) {
  const int dy = blockIdx.x, b = blockIdx.y, dx = threadIdx.x;
  const WarpBox box = boxes[b];
  int val[3] = {0, 0, 0};
  if (box.page >= 0) {
    const PageRef pg = pages[box.page];
    const double xb = static_cast<double>(dx & ~63), x1 = static_cast<double>(dx & 63), yy = static_cast<double>(dy);
    const double X0 = __dadd_rn(__dadd_rn(__dmul_rn(box.m[0], xb), __dmul_rn(box.m[1], yy)), box.m[2]);
    const double Y0 = __dadd_rn(__dadd_rn(__dmul_rn(box.m[3], xb), __dmul_rn(box.m[4], yy)), box.m[5]);
    const double W0 = __dadd_rn(__dadd_rn(__dmul_rn(box.m[6], xb), __dmul_rn(box.m[7], yy)), box.m[8]);
    double W = __dadd_rn(W0, __dmul_rn(box.m[6], x1));
    W = W != 0.0 ? __ddiv_rn(32.0, W) : 0.0;
    const double fX = fmax(-2147483648.0, fmin(2147483647.0, __dmul_rn(__dadd_rn(X0, __dmul_rn(box.m[0], x1)), W)));
    const double fY = fmax(-2147483648.0, fmin(2147483647.0, __dmul_rn(__dadd_rn(Y0, __dmul_rn(box.m[3], x1)), W)));
    const int X = __double2int_rn(fX), Y = __double2int_rn(fY);   // saturate_cast<int>: round half to even
    // remap stores the integer parts as shorts (saturate_cast<short>)
    const int sx = max(-32768, min(32767, X >> 5)), sy = max(-32768, min(32767, Y >> 5));
    const int fx = X & 31, fy = Y & 31;
    const int w00 = (32 - fx) * (32 - fy) * 32, w01 = fx * (32 - fy) * 32, w10 = (32 - fx) * fy * 32, w11 = fx * fy * 32;
    const int xa = min(max(sx, 0), pg.cols - 1), xc = min(max(sx + 1, 0), pg.cols - 1);
    const int ya = min(max(sy, 0), pg.rows - 1), yc = min(max(sy + 1, 0), pg.rows - 1);
    const uint8_t* r0 = pg.data + static_cast<size_t>(ya) * pg.step;
    const uint8_t* r1 = pg.data + static_cast<size_t>(yc) * pg.step;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int v = r0[xa * 3 + c] * w00 + r0[xc * 3 + c] * w01 + r1[xa * 3 + c] * w10 + r1[xc * 3 + c] * w11;
      val[c] = (v + (1 << 14)) >> 15;
    }
  }
  if (out_u8 != nullptr) {
    uint8_t* o = out_u8 + ((static_cast<size_t>(b) * 32 + dy) * 128 + dx) * 3;
    o[0] = static_cast<uint8_t>(val[0]); o[1] = static_cast<uint8_t>(val[1]); o[2] = static_cast<uint8_t>(val[2]);
  }
  if (out_patch != nullptr) {
    const size_t row = static_cast<size_t>(b) * 128 + (dy >> 2) * 16 + (dx >> 3);
    __nv_bfloat16* o = out_patch + row * 96 + (dy & 3) * 8 + (dx & 7);
#pragma unroll
    for (int c = 0; c < 3; ++c) o[c * 32] = __float2bfloat16(static_cast<float>(val[c]));
  }
}

}  // namespace

cudaError_t page_resize_pad(const uint8_t* src, int src_h, int src_w, size_t src_step, uint8_t* dst, int th, int tw,
                            int h32, int w32, cudaStream_t s) {
  const double scale_x = 1.0 / (static_cast<double>(tw) / src_w);
  const double scale_y = 1.0 / (static_cast<double>(th) / src_h);
  k_page_resize<<<dim3((w32 + 127) / 128, h32), 128, 0, s>>>(src, src_h, src_w, src_step, dst, th, tw, h32, w32,
                                                             scale_x, scale_y);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t page_im2col(const uint8_t* img, int batch, int H, int W, __nv_bfloat16* out, cudaStream_t s) {
  k_im2col<<<dim3((W + 127) / 128, H, batch), 128, 0, s>>>(img, H, W, out);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t crop_resize(const PageRef* pages_dev, const CropBox* boxes_dev, int n_boxes, uint8_t* out_u8,
                        __nv_bfloat16* out_patches, cudaStream_t s) {
  if (n_boxes <= 0) return cudaSuccess;
  k_crop<<<dim3(32, n_boxes), 128, 0, s>>>(pages_dev, boxes_dev, out_u8, out_patches);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t crop_resize_rot(const PageRef* pages_dev, const CropBox* boxes_dev, const uint8_t* rot_dev, int R, int n_crops,
                            uint8_t* out_u8, __nv_bfloat16* out_patches, cudaStream_t s) {
  if (n_crops <= 0) return cudaSuccess;
  k_crop_rot<<<dim3(32, n_crops), 128, 0, s>>>(pages_dev, boxes_dev, rot_dev, R, out_u8, out_patches);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

cudaError_t crop_warp(const PageRef* pages_dev, const WarpBox* boxes_dev, int n_boxes, uint8_t* out_u8,
                      __nv_bfloat16* out_patches, cudaStream_t s) {
  if (n_boxes <= 0) return cudaSuccess;
  k_crop_warp<<<dim3(32, n_boxes), 128, 0, s>>>(pages_dev, boxes_dev, out_u8, out_patches);
  TT_LAUNCH_CHECK();
  return cudaSuccess;
}

}  // namespace tt
