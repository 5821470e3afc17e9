// Device-side generation of the dense weak-label tensors the loss consumes, from the compact form the
// Open Images side stores (SURVEY.md 8f-2): replaces the host-side numpy of
//   code/input_pipelines/open_images/input_subset_bboxes_v2.py:74-98   (_generate_rla: box rasterisation,
//       overlapping boxes add counts, per-pixel normalisation to a multinomial, void where no box)
//   code/input_pipelines/open_images/input_subset_image_labels.py:73-107 (uniform over the image's
//       classes, tiled over the image)
// The box arithmetic (bit-exact with the numpy original) is weak_boxes.cuh, shared with the training gather.
//
// Bandwidth kernel: writes 60 B per pixel, reads the <= a few hundred boxes of the image from shared
// memory.  One thread per pixel; a CTA's 256 x 15 floats are one contiguous span of the output and leave
// through a shared-memory transpose as fully coalesced stores.
#include "weak_boxes.cuh"

namespace wlseg {

constexpr int kRastThreads = 256;

__global__ void __launch_bounds__(kRastThreads)
rasterize_bbox_kernel(const float* __restrict__ coords, const int32_t* __restrict__ cids, int max_boxes, int H, int W,
                      float* __restrict__ out) {
  __shared__ BoxI boxes[kMaxBoxesSmem];
  __shared__ int nbox;
  __shared__ float stage[kRastThreads * kWeakC];
  const int n = blockIdx.y;
  if (threadIdx.x == 0) nbox = 0;
  __syncthreads();
  // integer corners of the boxes of this image (entries with cid outside [0, 14] are skipped, as the
  // reference skips label ids that are not in mid2cid)
  for (int b = threadIdx.x; b < max_boxes; b += kRastThreads) {
    const int cid = cids[(int64_t)n * max_boxes + b];
    if (cid < 0 || cid >= kWeakC) continue;
    const float* c = coords + ((int64_t)n * max_boxes + b) * 4;   // xmin, xmax, ymin, ymax (normalised)
    BoxI bx;
    if (!box_corners(c[0], c[1], c[2], c[3], cid, H, W, bx)) continue;
    const int slot = atomicAdd(&nbox, 1);
    if (slot < kMaxBoxesSmem) boxes[slot] = bx;
  }
  __syncthreads();
  const int nb = nbox < kMaxBoxesSmem ? nbox : kMaxBoxesSmem;
  const int64_t npix = (int64_t)H * W;
  for (int64_t p0 = (int64_t)blockIdx.x * kRastThreads; p0 < npix; p0 += (int64_t)gridDim.x * kRastThreads) {
    const int64_t p = p0 + threadIdx.x;
    float v[kWeakC];
    if (p < npix) box_multinomial(boxes, nb, (int)(p / W), (int)(p % W), v);
    // transpose through shared memory: the block's 256 x 15 floats are one contiguous span of the output
    __syncthreads();
#pragma unroll
    for (int c = 0; c < kWeakC; ++c) stage[threadIdx.x * kWeakC + c] = v[c];
    __syncthreads();
    const int64_t valid = (npix - p0 < kRastThreads ? npix - p0 : kRastThreads) * kWeakC;
    float* dst = out + ((int64_t)n * npix + p0) * kWeakC;
    for (int i = threadIdx.x; i < valid; i += kRastThreads) dst[i] = stage[i];
  }
}

__global__ void __launch_bounds__(256)
tile_image_labels_kernel(const float* __restrict__ vec, int64_t npix, float* __restrict__ out) {
  // out[n, p, c] = vec[n, c]
  const int n = blockIdx.y;
  __shared__ float v[kWeakC];
  if (threadIdx.x < kWeakC) v[threadIdx.x] = vec[n * kWeakC + threadIdx.x];
  __syncthreads();
  const int64_t total = npix * kWeakC;
  float* dst = out + (int64_t)n * total;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = v[(int)(i % kWeakC)];
}

}  // namespace wlseg

using namespace wlseg;

extern "C" int wlseg_rasterize_bbox_labels(const float* coords, const int32_t* cids, int32_t N, int32_t max_boxes,
                                           int32_t H, int32_t W, float* out, wlseg_stream_t stream) {
  WLSEG_CHECK_ARG(N >= 0 && max_boxes >= 0 && H > 0 && W > 0, "rasterize_bbox_labels: bad shape");
  WLSEG_CHECK_ARG(max_boxes <= kMaxBoxesSmem, "rasterize_bbox_labels: more than %d boxes per image", kMaxBoxesSmem);
  WLSEG_CHECK_ARG(N <= 65535, "rasterize_bbox_labels: N too large");
  if (N == 0) return 0;
  WLSEG_CHECK_ARG(out && (max_boxes == 0 || (coords && cids)), "rasterize_bbox_labels: null pointer");
  const int64_t npix = (int64_t)H * W;
  int gx = (int)ceil_div(npix, kRastThreads);
  const int cap = (kNumSMs * 8 + N - 1) / N;
  if (gx > cap) gx = cap;
  dim3 grid(gx, N);
  rasterize_bbox_kernel<<<grid, kRastThreads, 0, (cudaStream_t)stream>>>(coords, cids, max_boxes, H, W, out);
  WLSEG_LAUNCH_CHECK();
  return 0;
}

extern "C" int wlseg_tile_image_labels(const float* vec, int32_t N, int32_t H, int32_t W, float* out,
                                       wlseg_stream_t stream) {
  WLSEG_CHECK_ARG(N >= 0 && H > 0 && W > 0 && N <= 65535, "tile_image_labels: bad shape");
  if (N == 0) return 0;
  WLSEG_CHECK_ARG(vec && out, "tile_image_labels: null pointer");
  const int64_t npix = (int64_t)H * W;
  int gx = (int)ceil_div(npix * kWeakC, 256 * 8);
  const int cap = (kNumSMs * 8 + N - 1) / N;
  if (gx > cap) gx = cap;
  if (gx < 1) gx = 1;
  dim3 grid(gx, N);
  tile_image_labels_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(vec, npix, out);
  WLSEG_LAUNCH_CHECK();
  return 0;
}
