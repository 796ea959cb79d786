// The contrast re-read (INTEGRATION.md section 10): a word whose first read is below contrast_ths and whose 128 x 32
// crop has low contrast is read again from a contrast-stretched crop, and the more confident read is kept.  Every step
// runs on the device; the host only reads how many words are re-read.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "orient.cuh"

namespace tt {

// Per word w of n_words (one block each).  ids / p [n_words][L]: the first read (the winner with rotation candidates);
// ids == nullptr considers every word (tt_contrast_adjust).  A word is considered when its conf (word_conf) is below
// contrast_ths.  Its crop is crop w * R + r of patches (bf16 patch rows, crop_resize's layout), r being the candidate of
// angle[w] in set (r = 0 when angle is null).  grey = cv2 BGR2GRAY of the crop's channels in stored order; low / high are
// np.percentile(grey, 10 / 90); contrast = (high - low) / max(10, high + low), all in double.  flag[w] = 1 iff the word is
// considered and contrast < adjust_contrast, else 0; then lr[w] = (low, 200 / max(10, high - low)).
cudaError_t contrast_stats(const int* ids, const float* p, int n_words, int L, float contrast_ths, float adjust_contrast,
                           const __nv_bfloat16* patches, int R, const int* angle, const OrientSet& set, int* flag,
                           double2* lr, cudaStream_t s);

// Order-preserving compaction: list = the words w with flag[w] != 0 in increasing order, *count = their number.
cudaError_t contrast_compact(const int* flag, int n_words, int* list, int* count, cudaStream_t s);

// For listed word i (w = list[i], crop as in contrast_stats): every channel value v of its crop becomes
// uint8(clip((v - low + 25) * ratio, 0, 255)) in double (EasyOCR's adjust_contrast_grey), via a 256-entry table.
// out_patches (nullable): crop i of a contiguous patch batch [n_listed * 128][96].  out_u8 (nullable): word w of
// [n_words][32][128][3] (crop_resize's u8 layout).  mask / root (nullable): the crop's class mask [4] or lexicon root,
// gathered to mask_out [n_listed][4] / root_out [n_listed] for the second forward.
cudaError_t contrast_apply(const int* list, int n_listed, const __nv_bfloat16* patches, int R, const int* angle,
                           const OrientSet& set, const double2* lr, __nv_bfloat16* out_patches, uint8_t* out_u8,
                           const uint32_t* mask, uint32_t* mask_out, const int* root, int* root_out, cudaStream_t s);

// One thread per listed word: the second read ids2 / p2 [n_listed][L] replaces word list[i]'s ids / p [.][L] in place
// when its conf is strictly greater (ties and NaN keep the first read).
cudaError_t contrast_select(int* ids, float* p, int L, const int* list, int n_listed, const int* ids2, const float* p2,
                            cudaStream_t s);

}  // namespace tt
