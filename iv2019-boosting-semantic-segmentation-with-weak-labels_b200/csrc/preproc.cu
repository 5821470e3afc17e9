// Input-side resize + crop of the training pipelines, code/input_pipelines/utils.py:181-247
// `resize_images_and_labels` over code/utils/utils.py:540-605 `resize_images_or_labels`:
//   images  tf.image.resize_images(BILINEAR),          align_corners=False  (TF-1.12 legacy mapping src = dst * in/out)
//   labels  tf.image.resize_images(NEAREST_NEIGHBOR),  align_corners=False  (src = min(floor(dst * in/out), in - 1))
//   --preserve_aspect_ratio: both are resized so that the target size fits tightly (mode 'max') and the SAME random
//   window of the target size is cut out of them.
// One pass: the crop window is read straight out of the source - the resized full-size tensor never exists.
// Bandwidth kernel, one thread per output element (consecutive threads = consecutive addresses).
#include "weak_boxes.cuh"

namespace wlseg {

// kind 0: fp32 bilinear, 1: fp32 nearest (dense 15-way weak labels), 2: int32 nearest (class-id labels)
template <int kKind, typename T>
__global__ void __launch_bounds__(256)
resize_crop_kernel(const T* __restrict__ x, T* __restrict__ y, int N, int H, int W, int C, int oy, int ox, int TH, int TW,
                   float sy, float sx) {
  const int64_t total = (int64_t)N * TH * TW * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    int64_t t = i / C;
    const int X = (int)(t % TW); t /= TW;
    const int Y = (int)(t % TH);
    const int n = (int)(t / TH);
    const float fy = (float)(Y + oy) * sy, fx = (float)(X + ox) * sx;
    const T* base = x + (int64_t)n * H * W * C + c;
    if (kKind == 0) {
      const int yl = min((int)floorf(fy), H - 1), xl = min((int)floorf(fx), W - 1);
      const int yh = min(yl + 1, H - 1), xh = min(xl + 1, W - 1);
      const float ly = fy - floorf(fy), lx = fx - floorf(fx);
      const float tl = (float)__ldg(base + ((int64_t)yl * W + xl) * C), tr = (float)__ldg(base + ((int64_t)yl * W + xh) * C);
      const float bl = (float)__ldg(base + ((int64_t)yh * W + xl) * C), br = (float)__ldg(base + ((int64_t)yh * W + xh) * C);
      const float top = tl + (tr - tl) * lx;
      const float bot = bl + (br - bl) * lx;
      y[i] = (T)(top + (bot - top) * ly);
    } else {
      const int yi = min((int)floorf(fy), H - 1), xi = min((int)floorf(fx), W - 1);
      y[i] = __ldg(base + ((int64_t)yi * W + xi) * C);
    }
  }
}

// [TF-1.12] CalculateResizeScale without align_corners: in / static_cast<float>(out)
__device__ __forceinline__ float legacy_scale(int in, int out) { return __fdiv_rn((float)in, (float)out); }

// Image part of the input contract (SURVEY.md 3.5) at one output pixel: an RGB image packed HWC at H x W, resized with
// the scales sy = legacy_scale(H, RH), sx = legacy_scale(W, RW) and sampled at (Ys, Xs) of the resized grid (the crop
// window's offset is already added).
//   u8 -> float * (float)(1/255) (tf.image.convert_image_dtype multiplies), TF-1.12 legacy bilinear (align_corners=False,
//   x first, then y), (v - 0.5) / 0.5.  Every operation is rounded on its own (__f*_rn keep the compiler from
//   contracting the lerps into FMAs): the host pipeline of wlseg/image_input.py and oracle/preprocess.py round that way,
//   and the contract is bit equality with them.
// -> the nearest source pixel (yl, xl) = min(floor(.), in - 1), which is also where legacy nearest reads labels.
struct SrcPixel { int y, x; };

__device__ __forceinline__ SrcPixel contract_image_pixel(const uint8_t* __restrict__ img, int H, int W, float sy, float sx,
                                                     int Ys, int Xs, float* __restrict__ pro) {
  const float inv255 = 1.0f / 255.0f;
  const float fy = __fmul_rn((float)Ys, sy), fx = __fmul_rn((float)Xs, sx);
  const float fly = floorf(fy), flx = floorf(fx);
  const int yl = min((int)fly, H - 1), xl = min((int)flx, W - 1);
  const int yh = min(yl + 1, H - 1), xh = min(xl + 1, W - 1);
  const float ly = __fsub_rn(fy, fly), lx = __fsub_rn(fx, flx);
  const uint8_t* ptl = img + ((int64_t)yl * W + xl) * 3;
  const uint8_t* ptr = img + ((int64_t)yl * W + xh) * 3;
  const uint8_t* pbl = img + ((int64_t)yh * W + xl) * 3;
  const uint8_t* pbr = img + ((int64_t)yh * W + xh) * 3;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float tl = __fmul_rn((float)__ldg(ptl + c), inv255), tr = __fmul_rn((float)__ldg(ptr + c), inv255);
    const float bl = __fmul_rn((float)__ldg(pbl + c), inv255), br = __fmul_rn((float)__ldg(pbr + c), inv255);
    const float top = __fadd_rn(tl, __fmul_rn(__fsub_rn(tr, tl), lx));
    const float bot = __fadd_rn(bl, __fmul_rn(__fsub_rn(br, bl), lx));
    const float v = __fadd_rn(top, __fmul_rn(__fsub_rn(bot, top), ly));
    pro[c] = __fmul_rn(__fsub_rn(v, 0.5f), 2.0f);   // / 0.5 is exact as * 2
  }
  return SrcPixel{yl, xl};
}

// Per-pixel input contract of output pixel (Y, X) from one raw example: the image part above resized straight to the
// target size, and the label-id map with legacy nearest, then lut[id] from shared memory; an id >= n_lids writes
// void_id and returns false.  Shared by the evaluation and training kernels, so that their bit equality with the host
// pipeline lives in one place.
__device__ __forceinline__ bool input_contract_pixel(const uint8_t* __restrict__ img, const uint8_t* __restrict__ lids,
                                                     int H, int W, int Y, int X, int TH, int TW,
                                                     const int32_t* s_lut, int n_lids, int void_id,
                                                     float* __restrict__ pro, int32_t* __restrict__ lab) {
  const SrcPixel src = contract_image_pixel(img, H, W, legacy_scale(H, TH), legacy_scale(W, TW), Y, X, pro);
  const int id = __ldg(lids + (int64_t)src.y * W + src.x);   // nearest: the same min(floor(.), in - 1)
  const bool ok = id < n_lids;
  *lab = ok ? s_lut[id] : void_id;
  return ok;
}

// Evaluation input contract from raw bytes, one thread per output pixel.  Example n is an RGB image packed HWC at its
// own size sizes[n] = (H, W) in row n of `images` (cap_img bytes per row) and its label-id map in row n of `lids`
// (cap_lab bytes per row).  A row whose size does not fit its buffers writes nothing and counts once; an out-of-range
// label id counts once per output pixel.
__global__ void __launch_bounds__(256)
eval_inputs_kernel(const uint8_t* __restrict__ images, int64_t cap_img, const uint8_t* __restrict__ lids, int64_t cap_lab,
                   const int32_t* __restrict__ sizes, int N, const int32_t* __restrict__ lut, int n_lids, int void_id,
                   int TH, int TW, float* __restrict__ pro, int32_t* __restrict__ lab,
                   unsigned long long* __restrict__ invalid) {
  __shared__ int32_t s_lut[256];
  for (int i = threadIdx.x; i < n_lids; i += blockDim.x) s_lut[i] = lut[i];
  __syncthreads();
  unsigned bad = 0;
  const int64_t total = (int64_t)N * TH * TW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int X = (int)(i % TW);
    const int64_t t = i / TW;
    const int Y = (int)(t % TH);
    const int n = (int)(t / TH);
    const int H = __ldg(sizes + 2 * n), W = __ldg(sizes + 2 * n + 1);
    if (H <= 0 || W <= 0 || (int64_t)H * W * 3 > cap_img || (int64_t)H * W > cap_lab) {
      bad += (X == 0 && Y == 0);
      continue;
    }
    bad += !input_contract_pixel(images + (int64_t)n * cap_img, lids + (int64_t)n * cap_lab, H, W, Y, X, TH, TW, s_lut,
                                 n_lids, void_id, pro + i * 3, lab + i);
  }
  // one atomic per warp: every lane leaves the grid-stride loop before this point
  const unsigned warp_bad = __reduce_add_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && warp_bad) atomicAdd(invalid, (unsigned long long)warp_bad);
}

// Training input contract (per-pixel part of the batch) gathered from a device-resident arena of raw examples, one
// thread per output pixel.  Output example n is arena example e = index[n]: its RGB image (H x W x 3 bytes, HWC) starts
// at byte offsets[e] and its label-id map (H x W bytes) follows it; sizes[e] = (H, W).  An index outside
// [0, n_examples) or a non-positive size writes nothing for that example and counts once; an out-of-range label id
// counts once per output pixel.
__global__ void __launch_bounds__(256)
train_inputs_kernel(const uint8_t* __restrict__ arena, const int64_t* __restrict__ offsets,
                    const int32_t* __restrict__ sizes, int n_examples, const int32_t* __restrict__ index, int N,
                    const int32_t* __restrict__ lut, int n_lids, int void_id, int TH, int TW, float* __restrict__ pro,
                    int32_t* __restrict__ lab, unsigned long long* __restrict__ invalid) {
  __shared__ int32_t s_lut[256];
  for (int i = threadIdx.x; i < n_lids; i += blockDim.x) s_lut[i] = lut[i];
  __syncthreads();
  unsigned bad = 0;
  const int64_t total = (int64_t)N * TH * TW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int X = (int)(i % TW);
    const int64_t t = i / TW;
    const int Y = (int)(t % TH);
    const int n = (int)(t / TH);
    const int e = __ldg(index + n);
    if (e < 0 || e >= n_examples) {
      bad += (X == 0 && Y == 0);
      continue;
    }
    const int H = __ldg(sizes + 2 * e), W = __ldg(sizes + 2 * e + 1);
    if (H <= 0 || W <= 0) {
      bad += (X == 0 && Y == 0);
      continue;
    }
    const uint8_t* img = arena + __ldg(offsets + e);
    bad += !input_contract_pixel(img, img + (int64_t)H * W * 3, H, W, Y, X, TH, TW, s_lut, n_lids, void_id, pro + i * 3,
                                 lab + i);
  }
  const unsigned warp_bad = __reduce_add_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && warp_bad) atomicAdd(invalid, (unsigned long long)warp_bad);
}

// Weak part of the training batch (bounding-box or image-level examples, SURVEY.md 3.5) gathered from a
// device-resident arena, one thread per output pixel and one row of CTAs (blockIdx.y) per output example.  Output
// example n is arena example e = index[n]: an RGB image (H x W x 3 bytes, HWC) at byte offsets[e], resized (aspect
// preserved) to resized[e] = (RH, RW) and cropped to TH x TW at crops[n] = (oy, ox).  Its label is, for the bbox part,
// _generate_rla of the boxes [box_start[e], box_start[e + 1]) rasterised at H x W, read with legacy nearest at the
// source pixel the image's bilinear lower corner uses; for the image-level part, vectors[e] at every pixel.  An index
// outside [0, n_examples), a crop outside [0, RH - TH] x [0, RW - TW], a non-positive size or more than kMaxBoxesSmem
// boxes writes nothing for that example and counts once.
constexpr int kWeakThreads = 256;

__global__ void __launch_bounds__(kWeakThreads)
weak_train_inputs_kernel(const uint8_t* __restrict__ arena, const int64_t* __restrict__ offsets,
                         const int32_t* __restrict__ sizes, const int32_t* __restrict__ resized, int n_examples,
                         const int32_t* __restrict__ box_start, const float4* __restrict__ box_coords,
                         const int32_t* __restrict__ box_cids, const float* __restrict__ vectors,
                         const int32_t* __restrict__ index, const int32_t* __restrict__ crops, int TH, int TW,
                         float* __restrict__ pro, float* __restrict__ lab, unsigned long long* __restrict__ invalid) {
  __shared__ BoxI boxes[kMaxBoxesSmem];
  __shared__ float s_vec[kWeakC];
  __shared__ float s_scale[2];
  __shared__ int nbox;
  __shared__ float stage[kWeakThreads * kWeakC];
  const int n = blockIdx.y;
  const int e = __ldg(index + n);
  // every thread of the CTA reaches the same verdict, so an invalid example leaves as a whole
  bool ok = e >= 0 && e < n_examples;
  int H = 0, W = 0, RH = 0, RW = 0, oy = 0, ox = 0, b0 = 0, b1 = 0;
  if (ok) {
    H = __ldg(sizes + 2 * e), W = __ldg(sizes + 2 * e + 1);
    RH = __ldg(resized + 2 * e), RW = __ldg(resized + 2 * e + 1);
    oy = __ldg(crops + 2 * n), ox = __ldg(crops + 2 * n + 1);
    ok = H > 0 && W > 0 && oy >= 0 && ox >= 0 && oy <= RH - TH && ox <= RW - TW;
    if (box_start != nullptr) {
      b0 = __ldg(box_start + e), b1 = __ldg(box_start + e + 1);
      ok = ok && b0 >= 0 && b1 >= b0 && b1 - b0 <= kMaxBoxesSmem;
    }
  }
  if (!ok) {
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(invalid, 1ull);
    return;
  }
  // the two scale divisions in different warps: one thread computing both keeps the first result across the second's
  // slow-path call in local memory
  if (threadIdx.x == 0) {
    nbox = 0;
    s_scale[0] = legacy_scale(H, RH);
  }
  if (threadIdx.x == 32) s_scale[1] = legacy_scale(W, RW);
  if (vectors != nullptr && threadIdx.x < kWeakC) s_vec[threadIdx.x] = __ldg(vectors + (int64_t)e * kWeakC + threadIdx.x);
  __syncthreads();
  // integer corners at H x W of the example's boxes (cids outside [0, 14] are skipped, as the reference skips mids that
  // are not in mid2cid); slots come in any order, the counts they add are order-free
  for (int b = b0 + threadIdx.x; b < b1; b += kWeakThreads) {
    const int cid = __ldg(box_cids + b);
    if (cid < 0 || cid >= kWeakC) continue;
    const float4 c = __ldg(box_coords + b);
    BoxI bx;
    if (box_corners(c.x, c.y, c.z, c.w, cid, H, W, bx)) boxes[atomicAdd(&nbox, 1)] = bx;   // b1 - b0 <= kMaxBoxesSmem
  }
  __syncthreads();
  const uint8_t* img = arena + __ldg(offsets + e);
  const int64_t npix = (int64_t)TH * TW;
  float* pro_n = pro + (int64_t)n * npix * 3;
  float* lab_n = lab + (int64_t)n * npix * kWeakC;
  for (int64_t p0 = (int64_t)blockIdx.x * kWeakThreads; p0 < npix; p0 += (int64_t)gridDim.x * kWeakThreads) {
    const int64_t p = p0 + threadIdx.x;
    float v[kWeakC];
    if (p < npix) {
      const int Y = (int)p / TW, X = (int)p - Y * TW;   // TH * TW < 2^31 (checked at launch)
      // the scales are read from shared memory per pixel: held in registers across the slow-path calls of the box
      // divisions, one of them spills to local memory
      const float sy = *(volatile float*)&s_scale[0], sx = *(volatile float*)&s_scale[1];
      const SrcPixel src = contract_image_pixel(img, H, W, sy, sx, Y + oy, X + ox, pro_n + p * 3);
      if (vectors != nullptr) {
#pragma unroll
        for (int c = 0; c < kWeakC; ++c) v[c] = s_vec[c];
      } else {
        box_multinomial(boxes, nbox, src.y, src.x, v);
      }
    }
    // transpose through shared memory: the CTA's 256 x 15 floats are one contiguous span of the output
    __syncthreads();
#pragma unroll
    for (int c = 0; c < kWeakC; ++c) stage[threadIdx.x * kWeakC + c] = v[c];
    __syncthreads();
    const int64_t valid = (npix - p0 < kWeakThreads ? npix - p0 : kWeakThreads) * kWeakC;
    float* dst = lab_n + p0 * kWeakC;
    for (int i = threadIdx.x; i < valid; i += kWeakThreads) dst[i] = stage[i];
  }
}

}  // namespace wlseg

using namespace wlseg;

extern "C" int wlseg_resize_crop(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, int32_t RH,
                                 int32_t RW, int32_t oy, int32_t ox, int32_t TH, int32_t TW, int32_t kind,
                                 wlseg_stream_t stream) {
  WLSEG_CHECK_ARG(N >= 0 && H > 0 && W > 0 && C > 0 && RH > 0 && RW > 0 && TH > 0 && TW > 0, "resize_crop: bad geometry");
  WLSEG_CHECK_ARG(oy >= 0 && ox >= 0 && oy + TH <= RH && ox + TW <= RW, "resize_crop: the crop window [%d+%d, %d+%d] leaves the resized tensor %d x %d",
                  oy, TH, ox, TW, RH, RW);
  WLSEG_CHECK_ARG(kind >= 0 && kind <= 2, "resize_crop: kind must be 0 (fp32 bilinear), 1 (fp32 nearest) or 2 (int32 nearest)");
  if (N == 0) return 0;
  WLSEG_CHECK_ARG(x && y, "resize_crop: null pointer");
  // [TF-1.12] CalculateResizeScale without align_corners: in / static_cast<float>(out)
  const float sy = (float)H / (float)RH, sx = (float)W / (float)RW;
  const int grid = bw_grid((int64_t)N * TH * TW * C, 256, 8);
  cudaStream_t s = (cudaStream_t)stream;
  if (kind == 0) resize_crop_kernel<0, float><<<grid, 256, 0, s>>>((const float*)x, (float*)y, N, H, W, C, oy, ox, TH, TW, sy, sx);
  else if (kind == 1) resize_crop_kernel<1, float><<<grid, 256, 0, s>>>((const float*)x, (float*)y, N, H, W, C, oy, ox, TH, TW, sy, sx);
  else resize_crop_kernel<2, int32_t><<<grid, 256, 0, s>>>((const int32_t*)x, (int32_t*)y, N, H, W, C, oy, ox, TH, TW, sy, sx);
  WLSEG_LAUNCH_CHECK();
  return 0;
}

extern "C" int wlseg_eval_inputs(const uint8_t* images, int64_t cap_img, const uint8_t* lids, int64_t cap_lab,
                                 const int32_t* sizes, int32_t N, const int32_t* lut, int32_t n_lids, int32_t void_id,
                                 int32_t TH, int32_t TW, float* proimages, int32_t* prolabels, int64_t* invalid,
                                 wlseg_stream_t stream) {
  WLSEG_CHECK_ARG(N >= 0 && TH > 0 && TW > 0 && cap_img > 0 && cap_lab > 0, "eval_inputs: bad geometry");
  WLSEG_CHECK_ARG(n_lids >= 1 && n_lids <= 256, "eval_inputs: the label-id table has %d entries, 1..256 supported", n_lids);
  if (N == 0) return 0;
  WLSEG_CHECK_ARG(images && lids && sizes && lut && proimages && prolabels && invalid, "eval_inputs: null pointer");
  const int grid = bw_grid((int64_t)N * TH * TW, 256, 8);
  eval_inputs_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(images, cap_img, lids, cap_lab, sizes, N, lut, n_lids, void_id,
                                                             TH, TW, proimages, prolabels, (unsigned long long*)invalid);
  WLSEG_LAUNCH_CHECK();
  return 0;
}

extern "C" int wlseg_train_inputs(const uint8_t* arena, const int64_t* offsets, const int32_t* sizes, int32_t n_examples,
                                  const int32_t* index, int32_t N, const int32_t* lut, int32_t n_lids, int32_t void_id,
                                  int32_t TH, int32_t TW, float* proimages, int32_t* prolabels, int64_t* invalid,
                                  wlseg_stream_t stream) {
  WLSEG_CHECK_ARG(N >= 0 && n_examples >= 0 && TH > 0 && TW > 0, "train_inputs: bad geometry");
  WLSEG_CHECK_ARG(n_lids >= 1 && n_lids <= 256, "train_inputs: the label-id table has %d entries, 1..256 supported", n_lids);
  if (N == 0) return 0;
  WLSEG_CHECK_ARG(index && lut && proimages && prolabels && invalid, "train_inputs: null pointer");
  WLSEG_CHECK_ARG(n_examples == 0 || (arena && offsets && sizes), "train_inputs: null arena");
  const int grid = bw_grid((int64_t)N * TH * TW, 256, 8);
  train_inputs_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(arena, offsets, sizes, n_examples, index, N, lut, n_lids,
                                                              void_id, TH, TW, proimages, prolabels,
                                                              (unsigned long long*)invalid);
  WLSEG_LAUNCH_CHECK();
  return 0;
}

extern "C" int wlseg_weak_train_inputs(const uint8_t* arena, const int64_t* offsets, const int32_t* sizes,
                                       const int32_t* resized, int32_t n_examples, const int32_t* box_start,
                                       const float* box_coords, const int32_t* box_cids, const float* vectors,
                                       const int32_t* index, const int32_t* crops, int32_t N, int32_t TH, int32_t TW,
                                       float* proimages, float* labels, int64_t* invalid, wlseg_stream_t stream) {
  WLSEG_CHECK_ARG(N >= 0 && N <= 65535 && n_examples >= 0 && TH > 0 && TW > 0 && (int64_t)TH * TW < (1ll << 31),
                  "weak_train_inputs: bad geometry");
  WLSEG_CHECK_ARG((box_start != nullptr) != (vectors != nullptr),
                  "weak_train_inputs: give either the box table (bounding-box part) or the vectors (image-level part)");
  if (N == 0) return 0;
  WLSEG_CHECK_ARG(index && crops && proimages && labels && invalid, "weak_train_inputs: null pointer");
  WLSEG_CHECK_ARG(n_examples == 0 || (arena && offsets && sizes && resized), "weak_train_inputs: null arena");
  WLSEG_CHECK_ARG(box_start == nullptr || (box_coords && box_cids), "weak_train_inputs: null box table");
  WLSEG_CHECK_ARG(((uintptr_t)box_coords & 15) == 0, "weak_train_inputs: box_coords must be 16-byte aligned");
  const int64_t npix = (int64_t)TH * TW;
  int gx = (int)ceil_div(npix, kWeakThreads);
  const int cap = (kNumSMs * 8 + N - 1) / N;
  if (gx > cap) gx = cap;
  weak_train_inputs_kernel<<<dim3(gx, N), kWeakThreads, 0, (cudaStream_t)stream>>>(
      arena, offsets, sizes, resized, n_examples, box_start, (const float4*)box_coords, box_cids, vectors, index, crops,
      TH, TW, proimages, labels, (unsigned long long*)invalid);
  WLSEG_LAUNCH_CHECK();
  return 0;
}
