// Bounding-box weak labels at one pixel: the arithmetic of
//   code/input_pipelines/open_images/input_subset_bboxes_v2.py:74-98 (_generate_rla: box rasterisation, overlapping
//   boxes add counts, per-pixel normalisation to a multinomial, void where no box)
// shared by the rasteriser (weak_labels.cu) and the training gather (preproc.cu), so that the two agree by
// construction.  Bit-exact with the numpy original: box corners are int(coord * size) evaluated in double as numpy does
// for float32 * int32, the slice [min : max + 1] is clipped to the image, counts are small integers and the
// normalisation is one IEEE float32 division per channel.
#pragma once

#include "common.cuh"

namespace wlseg {

constexpr int kWeakC = 15;            // 14 Open Images classes + void (input_subset_bboxes_v2.py:38-53)
constexpr int kMaxBoxesSmem = 1024;   // boxes of one image held in shared memory

struct BoxI { int x0, x1, y0, y1, cid; };

// Integer corners at H x W of the box (xmin, xmax, ymin, ymax normalised) of class `cid`; false when it covers no
// pixel: python's rla[y0 : y1 + 1, x0 : x1 + 1] for non-negative corners is clipped to the image and empty when
// min > max.
__device__ __forceinline__ bool box_corners(float xmin, float xmax, float ymin, float ymax, int cid, int H, int W,
                                            BoxI& bx) {
  bx.x0 = (int)((double)xmin * (double)W);
  bx.x1 = (int)((double)xmax * (double)W);
  bx.y0 = (int)((double)ymin * (double)H);
  bx.y1 = (int)((double)ymax * (double)H);
  bx.cid = cid;
  if (bx.x0 < 0) bx.x0 = 0;
  if (bx.y0 < 0) bx.y0 = 0;
  if (bx.x1 > W - 1) bx.x1 = W - 1;
  if (bx.y1 > H - 1) bx.y1 = H - 1;
  return bx.x0 <= bx.x1 && bx.y0 <= bx.y1;
}

// The 15-way multinomial of pixel (y, x) under `nb` boxes (shared memory): counts per class, divided by their sum, or
// void = 1 where no box covers the pixel.
__device__ __forceinline__ void box_multinomial(const BoxI* boxes, int nb, int y, int x, float (&v)[kWeakC]) {
#pragma unroll
  for (int c = 0; c < kWeakC; ++c) v[c] = 0.f;
  for (int b = 0; b < nb; ++b) {
    const BoxI bx = boxes[b];
    const bool in = (x >= bx.x0) & (x <= bx.x1) & (y >= bx.y0) & (y <= bx.y1);
#pragma unroll
    for (int c = 0; c < kWeakC; ++c) v[c] += (in && bx.cid == c) ? 1.f : 0.f;   // small integers: order-free
  }
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < kWeakC; ++c) s += v[c];
  if (s > 0.5f) {
#pragma unroll
    for (int c = 0; c < kWeakC; ++c) v[c] = __fdiv_rn(v[c], s);
  } else {
#pragma unroll
    for (int c = 0; c < kWeakC; ++c) v[c] = (c == kWeakC - 1) ? 1.f : 0.f;
  }
}

}  // namespace wlseg
