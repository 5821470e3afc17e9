/*
 * wlseg.h -- C ABI of libwlseg.so, the B200 (sm_100a) implementation of the
 * segmentation hot path of pmeletis/IV2019-boosting-semantic-segmentation-with-weak-labels.
 *
 * The reference has no FFI layer: every device op it runs is a TensorFlow-1.12 op reached
 * from its Python model / loss / estimator code.  Each entry point below therefore cites the
 * reference call site (relative to /root/reference/code/) whose TF op(s) it replaces; the
 * Python host (wlseg/ops.py) binds them with ctypes exactly as INTEGRATION.md shows.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless named `h_*`;
 *     the library never allocates or frees user memory and keeps no reference to it
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing blocks
 *   - activations are NHWC, convolution kernels are KRSC ([Cout][kh][kw][Cin])
 *   - dtype: WLSEG_F32 or WLSEG_BF16 storage; all arithmetic accumulates in fp32
 *   - return 0 on success, <0 invalid argument / unsupported configuration,
 *     >0 a cudaError_t; wlseg_last_error() returns a thread-local description
 *   - there is NO CPU fallback: unsupported configurations return an error
 */
#ifndef WLSEG_H_
#define WLSEG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WLSEG_VERSION 100 /* 0.1.0 */

typedef void* wlseg_stream_t;

enum { WLSEG_F32 = 0, WLSEG_BF16 = 1 };
enum { WLSEG_ALGO_AUTO = 0, WLSEG_ALGO_DIRECT = 1, WLSEG_ALGO_TCGEN05 = 2 };

int wlseg_version(void);
const char* wlseg_last_error(void);

/* ------------------------------------------------------------------------------------------
 * Convolution (replaces slim.conv2d / resnet_utils.conv2d_same:
 *   models/resnet50_extended_feature_extractor.py:25-30,39-43,
 *   models/resnet50_extended_model_hierarchical.py:60-64,80)
 * y[n,p,q,k] = epi( sum_{r,s,c} x[n, p*stride - pad_top + r*dilation,
 *                                   q*stride - pad_left + s*dilation, c] * w[k,r,s,c] )
 * epi(v) = relu?( v*scale[k] + shift[k] + residual[n, p*res_stride, q*res_stride, k] )
 * (scale/shift/residual optional; they carry the folded inference batch-norm,
 *  resnet50_extended_model_hierarchical.py:298-312, and the bottleneck shortcut add).
 * bn_sum/bn_sqsum (optional, double[K]) receive sum / sum of squares of the RAW fp32
 * accumulators per output channel (training-mode batch-norm statistics); they are
 * accumulated into, the caller zeroes them.
 * ------------------------------------------------------------------------------------------ */
typedef struct wlseg_conv_params {
  int32_t N, H, W, C;       /* input NHWC, C = input channels */
  int32_t K, R, S;          /* output channels, kernel height / width */
  int32_t P, Q;             /* output height / width */
  int32_t stride, dilation;
  int32_t pad_top, pad_left; /* zero padding before; padding after is implied by P, Q */
  int32_t x_pitch;          /* elements between consecutive input pixels  (>= C) */
  int32_t y_pitch;          /* elements between consecutive output pixels (>= K) */
  int32_t res_pitch;        /* elements between consecutive residual pixels */
  int32_t res_stride;       /* residual is read at (p*res_stride, q*res_stride) */
  int32_t res_H, res_W;     /* spatial size of the residual tensor */
  int32_t relu;
  int32_t dtype;            /* WLSEG_F32 | WLSEG_BF16: x, w, residual (and y) storage */
  int32_t y_dtype;          /* storage of y; WLSEG_F32 lets a bf16 layer emit fp32 (logits) */
  int32_t algo;             /* WLSEG_ALGO_* */
  int32_t accumulate;       /* wgrad only: 0 = dw is overwritten, 1 = dw += (the caller zeroed it) */
  int32_t reverse;          /* fprop (tcgen05): output tiles are produced from the END of the tensor to its start.
                             * Same result; a consumer that starts where its producer ended finds its first
                             * ~L2-size of input still on chip (layers alternate directions in inference). */
} wlseg_conv_params;

/* 1 if the tcgen05 implicit-GEMM kernel covers this configuration, else 0. */
int wlseg_conv2d_tcgen05_supported(const wlseg_conv_params* p);

int wlseg_conv2d_fprop(const wlseg_conv_params* p, const void* x, const void* w, void* y,
                       const float* scale, const float* shift, const void* residual,
                       double* bn_sum, double* bn_sqsum, wlseg_stream_t stream);

/* y = (conv(x, w) + residual) * mask, bf16, tcgen05 only: the data gradient of a layer whose INPUT tensor is the
 * output of a ReLU (+ residual) unit leaves the dgrad epilogue already multiplied by that ReLU's derivative.
 * out_mask: one bit per output element, [N*P*Q][K / 8] bytes, bit (c & 7) of byte c >> 3 (wlseg_bn_apply_mask writes
 * it in the forward pass).  The batch-norm backward of the unit then runs without reading its activation and without
 * writing a separate residual gradient (it IS this tensor): 3 of its 8 tensor passes disappear
 * (models/resnet50_extended_model_hierarchical.py:298-312 backward, slim bottleneck shortcut add). */
int wlseg_conv2d_fprop_masked(const wlseg_conv_params* p, const void* x, const void* w, void* y,
                              const void* residual, const uint8_t* out_mask, wlseg_stream_t stream);

/* Training-mode batch-norm finalisation carried by the convolution that produces the statistics
 * (wlseg_conv2d_fprop_bn): what wlseg_bn_finalize computes, run by the last CTA of the convolution grid to commit
 * its partial sums.  `counter`: one zero-initialised device word, left at zero (shared by all layers of a stream). */
typedef struct wlseg_bn_finalize_args {
  int64_t count;             /* pixels the statistics are taken over: N * P * Q */
  float eps, decay;
  float moving_var_factor;   /* < 0: Bessel-corrected moving variance (slim.batch_norm); >= 0: var * factor */
  int32_t reserved;
  const float* gamma;
  const float* beta;
  float* moving_mean;        /* may both be NULL */
  float* moving_var;
  float* scale;              /* out: gamma * invstd */
  float* shift;              /* out: beta - mean * scale */
  float* saved_mean;         /* out */
  float* saved_invstd;       /* out */
  uint32_t* counter;
} wlseg_bn_finalize_args;

/* y = conv(x, w) (raw, bf16), bn_sum / bn_sqsum += per-channel sums of the stored y, and - by the last CTA - the
 * layer's scale / shift / saved mean / inverse std and moving statistics: wlseg_conv2d_fprop(..., bn_sum, bn_sqsum)
 * followed by wlseg_bn_finalize in ONE launch (slim.conv2d + training-mode FusedBatchNorm statistics,
 * models/resnet50_extended_model_hierarchical.py:298-312).  tcgen05 only, K % 64 == 0. */
int wlseg_conv2d_fprop_bn(const wlseg_conv_params* p, const void* x, const void* w, void* y, double* bn_sum,
                          double* bn_sqsum, const wlseg_bn_finalize_args* fin, wlseg_stream_t stream);

/* y = conv(x, w) * relu'(bn(z)), bf16, tcgen05 only, fused with the batch-norm backward REDUCTION of the layer that
 * produced z: the data gradient of a tensor a = relu(z * scale + shift) leaves the dgrad epilogue already multiplied
 * by the ReLU derivative (sign of the exact fp32 value the forward pass rounded), and the epilogue accumulates
 *   dgamma[c] += sum y * (z - mean[c]) * invstd[c],   dbeta[c] += sum y     (over the STORED bf16 y, fp64 atomics,
 * one per channel and CTA) - what wlseg_bn_bwd_reduce would compute in a separate pass over y and z
 * (FusedBatchNormGrad behind models/resnet50_extended_model_hierarchical.py:298-312; the ReLU is slim.conv2d's
 * activation_fn).  z has y's shape; the res_* fields of the parameters describe it (res_stride 1, res_H = P,
 * res_W = Q, res_pitch).  K % 64 == 0; y, z, scale, shift 16-byte aligned.  wlseg_bn_bwd_apply then runs with
 * relu = 0 on (y, z). */
int wlseg_conv2d_fprop_bnbwd(const wlseg_conv_params* p, const void* x, const void* w, void* y, const void* z,
                             const float* scale, const float* shift, const float* mean, const float* invstd,
                             double* dgamma, double* dbeta, wlseg_stream_t stream);

/* dx = conv_transpose(dy, w): gradient wrt the input (TF Conv2DBackpropInput, reached through
 * create_train_op, estimator/define_estimator_hierarchical.py:120-129).  dx is fully written. */
int wlseg_conv2d_dgrad(const wlseg_conv_params* p, const void* dy, const void* w, void* dx,
                       wlseg_stream_t stream);

/* dw[k,r,s,c] = sum_{n,p,q} dy[n,p,q,k] * x[...]  (TF Conv2DBackpropFilter); dw is fp32 KRSC,
 * fully written (beta = 0) unless p->accumulate is set (then added to: one memset of the whole
 * gradient arena per step replaces one per layer). */
int wlseg_conv2d_wgrad(const wlseg_conv_params* p, const void* x, const void* dy, float* dw,
                       wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Batch norm, training mode (replaces tf.contrib.layers.batch_norm / FusedBatchNorm(+Grad),
 * models/resnet50_extended_model_hierarchical.py:298-312,325).
 * ------------------------------------------------------------------------------------------ */
/* per-channel sum / sum of squares of z (count x C, pitch elements per row) into double[C]
 * (accumulated into; the caller zeroes). */
int wlseg_bn_stats(const void* z, int64_t count, int32_t C, int32_t pitch, int32_t dtype,
                   double* sum, double* sqsum, wlseg_stream_t stream);

/* mean = sum/count, var = sqsum/count - mean^2 (biased); scale = gamma*rsqrt(var+eps),
 * shift = beta - mean*scale; moving stats updated in place with `decay` and the unbiased
 * variance (skipped if moving_mean is NULL); saved_mean / saved_invstd for the backward.
 * moving_var_factor < 0: the moving variance takes var * count / (count - 1) (tf.contrib.layers
 * .batch_norm, fused); >= 0: it takes var * moving_var_factor.  --cross_replica_norm passes the
 * all-reduced sums with count = replicas * n_local and the factor (n_local - 1) / n_local, the
 * "Bessel removal" of utils/cross_replica_batch_normalization.py:452-459. */
int wlseg_bn_finalize(const double* sum, const double* sqsum, int64_t count, int32_t C,
                      const float* gamma, const float* beta, float eps, float decay,
                      float moving_var_factor, float* moving_mean, float* moving_var, float* scale,
                      float* shift, float* saved_mean, float* saved_invstd, wlseg_stream_t stream);

/* wlseg_bn_finalize + wlseg_bn_apply in one launch (C % 8 == 0, C <= 2048): every thread derives scale / shift of
 * its 8 channels from the sums; CTA 0 publishes them (+ saved mean / invstd, moving statistics).  relu_mask (may be
 * NULL): as wlseg_bn_apply_mask. */
int wlseg_bn_finalize_apply(const double* sum, const double* sqsum, int64_t count, int32_t C,
                            const float* gamma, const float* beta, float eps, float decay,
                            float* moving_mean, float* moving_var, float* scale, float* shift,
                            float* saved_mean, float* saved_invstd, const void* z, const void* residual,
                            void* y, uint8_t* relu_mask, int32_t relu, int32_t dtype, wlseg_stream_t stream);

/* y = relu?( z*scale[c] + shift[c] + residual ), elementwise over count x C. */
int wlseg_bn_apply(const void* z, const float* scale, const float* shift, const void* residual,
                   void* y, int64_t count, int32_t C, int32_t relu, int32_t dtype,
                   wlseg_stream_t stream);

/* wlseg_bn_apply with ReLU that also records relu_mask[row][c >> 3] bit (c & 7) = (y > 0)
 * (C % 32 == 0, C <= 2048); see wlseg_conv2d_fprop_masked. */
int wlseg_bn_apply_mask(const void* z, const float* scale, const float* shift, const void* residual,
                        void* y, uint8_t* relu_mask, int64_t count, int32_t C, int32_t dtype,
                        wlseg_stream_t stream);

/* Backward of y = relu?(bn(z) + residual).  Pass 1 (reduce): with g = dy * (y > 0 if relu),
 * dbeta[c] += sum g, dgamma[c] += sum g * (z - mean)*invstd  (double[C], caller zeroes).
 * Pass 2 (apply): dz = gamma*invstd*(g - dbeta/count - zhat*dgamma/count); if dres != NULL the
 * masked gradient g is also written there (gradient of the residual input).
 * `y` may be NULL for a ReLU layer WITHOUT a residual input: the mask is then the sign of
 * fmaf(z, scale[c], shift[c]) - the fp32 value the forward pass rounded to y - and y is not read.
 * `pitch` = elements between consecutive rows of dy / y / z / dz / dres (all share it): a channel
 * slice [c0, c0 + C) of a wider tensor is processed by passing pointers offset by c0 and the full
 * width as pitch; the host mirror runs reduce + apply slice by slice so that the second pass reads
 * its three inputs from L2 instead of HBM.
 * `stat_count` (apply) = number of pixels dgamma / dbeta were summed over: equal to `count` (the
 * rows of THIS tensor) except under --cross_replica_norm, where the sums are all-reduced over the
 * replicas and stat_count = replicas * count. */
int wlseg_bn_bwd_reduce(const void* dy, const void* y, const void* z, const float* mean,
                        const float* invstd, const float* scale, const float* shift, int64_t count,
                        int32_t C, int32_t pitch, int32_t relu, int32_t dtype, double* dgamma,
                        double* dbeta, wlseg_stream_t stream);
int wlseg_bn_bwd_apply(const void* dy, const void* y, const void* z, const float* mean,
                       const float* invstd, const float* gamma, const float* scale, const float* shift,
                       const double* dgamma, const double* dbeta, int64_t count, int64_t stat_count,
                       int32_t C, int32_t pitch, int32_t relu, int32_t dtype, void* dz, void* dres,
                       wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Max pool, TF 'SAME' padding (replaces slim.max_pool2d: resnet pool1 3x3 s2 and the 1x1 s2
 * shortcut subsample; arg scope models/resnet50_extended_model_hierarchical.py:351-353).
 * Backward routes the gradient to the first maximum of each window in row-major scan order.
 * `argmax` (optional, uint8 [N,P,Q,C]) receives / supplies the winning window position r*k+s of
 * every output element; with it the backward is a pure gather over dy (no re-read of x).  Without
 * it (NULL) the backward recomputes the winners from x.
 * ------------------------------------------------------------------------------------------ */
int wlseg_maxpool_same_fwd(const void* x, void* y, uint8_t* argmax, int32_t N, int32_t H, int32_t W,
                           int32_t C, int32_t ksize, int32_t stride, int32_t dtype,
                           wlseg_stream_t stream);
int wlseg_maxpool_same_bwd(const void* x, const uint8_t* argmax, const void* dy, void* dx, int32_t N,
                           int32_t H, int32_t W, int32_t C, int32_t ksize, int32_t stride,
                           int32_t dtype, wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Group normalisation, `--norm_layer group` (tf.contrib.layers.group_norm, groups = 32 / 1 for the logits layers,
 * models/resnet50_extended_model_hierarchical.py:75-77,314-333).  Statistics are per (sample, group) over
 * H*W*(C/groups) values, biased variance, no moving statistics.  The per-sample passes over the activations are
 * the batch-norm entry points above called on one sample's H*W rows (wlseg_bn_stats, wlseg_bn_apply,
 * wlseg_bn_bwd_reduce); these three turn their per-(sample, channel) results into the per-(sample, channel)
 * affine forms.  All arrays indexed [n * C + c].
 *   gn_finalize:     sum / sqsum (double) -> scale, shift (y = z * scale + shift), mean, invstd
 *   gn_bwd_finalize: dgamma_nc = sum g * xhat, dbeta_nc = sum g (double, from wlseg_bn_bwd_reduce with the mean /
 *                    invstd rows of gn_finalize) -> cA, c1, c0 with dz = cA * g + c1 * z + c0, and
 *                    dgamma[c] += sum_n dgamma_nc, dbeta[c] += sum_n dbeta_nc (double, accumulated into)
 *   gn_bwd_apply:    dz (and dres = masked g) for the whole batch [N, hw, C]; ReLU mask from y, or from
 *                    sign(fmaf(z, scale, shift)) when y is NULL
 * ------------------------------------------------------------------------------------------ */
int wlseg_gn_finalize(const double* sum, const double* sqsum, int32_t N, int32_t C, int32_t groups, int64_t hw,
                      const float* gamma, const float* beta, float eps, float* scale, float* shift, float* mean,
                      float* invstd, wlseg_stream_t stream);
int wlseg_gn_bwd_finalize(const double* dgamma_nc, const double* dbeta_nc, int32_t N, int32_t C, int32_t groups,
                          int64_t hw, const float* gamma, const float* mean, const float* invstd, float* cA,
                          float* c1, float* c0, double* dgamma, double* dbeta, wlseg_stream_t stream);
int wlseg_gn_bwd_apply(const void* dy, const void* y, const void* z, const float* cA, const float* c1,
                       const float* c0, const float* scale, const float* shift, int32_t N, int64_t hw, int32_t C,
                       int32_t relu, int32_t dtype, void* dz, void* dres, wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Pyramid (PSP) module pieces, `--psp_module` (models/resnet50_extended_model_hierarchical.py:186-207):
 * slim.layers.avg_pool2d VALID (:191-200), tf.image.resize_images(bilinear, align_corners=True) of
 * the pooled branches back to the feature size (:193-202), and their gradients.  NHWC, C % 8 == 0.
 *   avgpool fwd: y[N, P, Q, C], P = (H - kh) / sh + 1 (windows that do not fit are dropped).
 *   avgpool bwd (kernel == stride): dx (+)= dy[h / kh, w / kw] / (kh * kw); accumulate != 0 adds to dx.
 *   resize fwd writes y with pixel pitch y_pitch (a channel slice of the 5 * C concatenation);
 *   resize bwd reads dy with pixel pitch dy_pitch and fully writes dx[N, h, w, C].
 * ------------------------------------------------------------------------------------------ */
int wlseg_avgpool_valid_fwd(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, int32_t kh,
                            int32_t kw, int32_t sh, int32_t sw, int32_t dtype, wlseg_stream_t stream);
int wlseg_avgpool_valid_bwd(const void* dy, void* dx, int32_t N, int32_t H, int32_t W, int32_t C, int32_t kh,
                            int32_t kw, int32_t accumulate, int32_t dtype, wlseg_stream_t stream);
int wlseg_resize_bilinear_fwd(const void* x, void* y, int32_t N, int32_t h, int32_t w, int32_t C, int32_t H,
                              int32_t W, int32_t y_pitch, int32_t dtype, wlseg_stream_t stream);
int wlseg_resize_bilinear_bwd(const void* dy, void* dx, int32_t N, int32_t h, int32_t w, int32_t C, int32_t H,
                              int32_t W, int32_t dy_pitch, int32_t dtype, wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Weak labels from their compact form (SURVEY.md 8f-2; the reference builds them on the host:
 * input_pipelines/open_images/input_subset_bboxes_v2.py:74-98 `_generate_rla`,
 * input_pipelines/open_images/input_subset_image_labels.py:73-107).  Bit-exact with the numpy code.
 *   coords float32 [N, max_boxes, 4] = (xmin, xmax, ymin, ymax) normalised to [0, 1];
 *   cids   int32   [N, max_boxes]    = class id 0..13, anything else = padding / unknown label (skipped);
 *   out    float32 [N, H, W, 15]: per pixel the box counts per class divided by their sum, or
 *   void (channel 14) = 1 where no box covers the pixel.
 * wlseg_tile_image_labels: out[n, :, :, :] = vec[n, :] (the image-level multinomial, tiled).
 * ------------------------------------------------------------------------------------------ */
int wlseg_rasterize_bbox_labels(const float* coords, const int32_t* cids, int32_t N, int32_t max_boxes,
                                int32_t H, int32_t W, float* out, wlseg_stream_t stream);
int wlseg_tile_image_labels(const float* vec, int32_t N, int32_t H, int32_t W, float* out,
                            wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Hierarchical head, forward (replaces _create_upsampler + softmax x3 + argmax x3 + gather /
 * where composition, models/resnet50_extended_model_hierarchical.py:84-117,143-184).
 * logits: fp32 [N, h, w, logits_pitch] low-resolution logits of the three heads, concatenated
 * along channels (the first C1+Cv+Ch of every logits_pitch-wide pixel are used).  Bilinear upsampling to (H, W) with align_corners=True is done on the fly.
 * Outputs (each optional, NULL to skip): decisions int32 [N,H,W] in common class ids;
 * l1/l2v/l2h decisions int32 [N,H,W]; l1/l2v/l2h probabilities fp32 [N,H,W,C*];
 * full-resolution logits fp32 [N,H,W,C1+Cv+Ch].
 * ------------------------------------------------------------------------------------------ */
typedef struct wlseg_hierarchy {
  int32_t C1, Cv, Ch;           /* head widths (14/7/3 cityscapes, 53/12/5 vistas) */
  int32_t cid_l1_vehicle, cid_l1_human;
  int32_t l1_to_common[64];     /* l1 cid -> common cid */
  int32_t veh_to_common[16];
  int32_t hum_to_common[8];
  /* loss side (estimator/define_losses_hierarchical.py:38-93) */
  int32_t num_classes;          /* strong label ids in [0, num_classes) */
  int32_t pp_to_l1[80], pp_to_veh[80], pp_to_hum[80];
  int32_t bb_to_veh[15], bb_to_hum[15];
} wlseg_hierarchy;

int wlseg_head_fwd(const wlseg_hierarchy* hier, const float* logits, int32_t logits_pitch,
                   int32_t N, int32_t h, int32_t w, int32_t H, int32_t W, int32_t* decisions, int32_t* l1_decisions,
                   int32_t* l2v_decisions, int32_t* l2h_decisions, float* l1_probs,
                   float* l2v_probs, float* l2h_probs, float* fullres_logits,
                   wlseg_stream_t stream);

/* Evaluation step tail in ONE launch: x8 bilinear upsample + three arg-maxima + hierarchical composition
 * (models/resnet50_extended_model_hierarchical.py:84-117) fused with the streaming confusion matrix
 * (estimator/define_estimator_hierarchical.py:185-194) and the decisions part of _map_predictions_to_new_cids (:511-514,
 * `lut`).  cm[label, lut[decision]] += 1 for every pixel, bit-exact (integer); out-of-range pairs are skipped and counted
 * in *invalid (may be NULL).  decisions (int32 [N,H,W]) is optional: NULL = the decisions never touch HBM.
 * labels NULL = decisions only.  Decisions are bit-identical to wlseg_head_fwd's.  Hierarchies other than 14/7/3 and
 * 53/12/5, or an upsampling factor below 2, fall back to wlseg_head_fwd + wlseg_confmat_accumulate and need the
 * decisions buffer. */
int wlseg_head_confmat(const wlseg_hierarchy* hier, const float* logits, int32_t logits_pitch, int32_t N, int32_t h,
                       int32_t w, int32_t H, int32_t W, const int32_t* labels, int32_t num_classes, const int32_t* lut,
                       int32_t lut_size, int64_t* cm, int64_t* invalid, int32_t* decisions, wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Prediction post-processing (estimator/define_estimator_hierarchical.py:530-571 `_resize_predictions`,
 * :573-630 `_replace_voids`), used by the EVAL branch when labels and network differ in size and by the
 * PREDICT branch for --height_system / --width_system or the raw image size (:219-232).
 *   probabilities fp32 [N, h, w, C] -> [N, H, W, C]: tf.image.resize_images bilinear, align_corners=True
 *   decisions int32 [N, h, w] -> [N, H, W]: NEAREST_NEIGHBOR, align_corners=True, in = min(roundf(out * scale), in - 1)
 *   replace_voids: decisions (in place, n_pixels of them) equal to void_cid are recomposed from the three
 *   probability maps with every head restricted to its non-void classes (its last channel is void): the
 *   reference's "runner-up of top_k(probs, 2) where the decision is void", applied per head.  The reference
 *   itself stops at the key-set assert of :589-592 on this model.
 * ------------------------------------------------------------------------------------------ */
int wlseg_resize_probabilities(const float* x, float* y, int32_t N, int32_t h, int32_t w, int32_t C, int32_t H,
                               int32_t W, wlseg_stream_t stream);
int wlseg_resize_decisions(const int32_t* x, int32_t* y, int32_t N, int32_t h, int32_t w, int32_t H, int32_t W,
                           wlseg_stream_t stream);
int wlseg_replace_voids(const wlseg_hierarchy* hier, const float* l1_probs, const float* l2v_probs,
                        const float* l2h_probs, int32_t* decisions, int64_t n_pixels, int32_t void_cid,
                        wlseg_stream_t stream);

/* wlseg_loss_fwd_bwd with the weak labels in their COMPACT form (SURVEY.md 8f-2): the bbox images carry
 * (class, box) lists - coords float32 [n_bbox, max_boxes, 4] = (xmin, xmax, ymin, ymax) normalised, cids int32
 * [n_bbox, max_boxes], anything outside [0, 14] = padding - and the image-level images one 15-way vector each
 * (float32 [n_image, 15]).  The kernel evaluates `_generate_rla` (input_subset_bboxes_v2.py:74-98) and the
 * image-level tiling (input_subset_image_labels.py:73-107) per pixel in registers instead of reading 60 B per
 * pixel of dense labels; results are identical to rasterising first.  14/7/3 hierarchy at >= 2x upsampling
 * (the column-walking kernel); other configurations return an error: rasterise and call wlseg_loss_fwd_bwd. */
int wlseg_loss_fwd_bwd_lists(const wlseg_hierarchy* hier, const float* logits, int32_t logits_pitch,
                             int32_t n_strong, int32_t n_bbox, int32_t n_image, int32_t h, int32_t w,
                             int32_t H, int32_t W, const int32_t* strong_labels, const float* box_coords,
                             const int32_t* box_cids, int32_t max_boxes, const float* image_vectors,
                             double* sums, double* counts, float* dlogits, wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Hierarchical strong + weak masked cross-entropy, forward and backward fused with the
 * bilinear upsample and its transpose (replaces estimator/define_losses_hierarchical.py:97-203
 * and ResizeBilinearGrad).  Batch order: n_strong images with per-pixel labels int32 [.,H,W],
 * then n_bbox images with fp32 [.,H,W,15] labels, then n_image images with fp32 [.,H,W,15].
 * sums: double[3] += sum(ce*w) for (l1, l2_vehicle, l2_human); counts: double[3] += count(w!=0)
 * (caller zeroes).  dlogits: fp32 [N,h,w,logits_pitch], accumulated into (caller zeroes), holds the
 * UNNORMALISED gradient sum_pixels w*(softmax - target) transposed through the upsample;
 * wlseg_loss_finalize scales it by coef/count per head and produces the six scalar losses.
 * ------------------------------------------------------------------------------------------ */
int wlseg_loss_fwd_bwd(const wlseg_hierarchy* hier, const float* logits, int32_t logits_pitch,
                       int32_t n_strong, int32_t n_bbox, int32_t n_image, int32_t h, int32_t w, int32_t H, int32_t W,
                       const int32_t* strong_labels, const float* bbox_labels,
                       const float* image_labels, double* sums, double* counts, float* dlogits,
                       wlseg_stream_t stream);
/* losses: float[4] = {l1, l2_vehicle, l2_human, segmentation = l1 + l2_coef*(l2v + l2h)};
 * dlogits scaled in place by grad_scale * coef_head / count_head (0 where count is 0). */
int wlseg_loss_finalize(const wlseg_hierarchy* hier, const double* sums, const double* counts,
                        float l2_coef, float grad_scale, float* dlogits, int32_t logits_pitch,
                        int64_t n_lowres_pixels, float* losses, wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Confusion matrix (replaces metrics_impl._streaming_confusion_matrix,
 * estimator/define_estimator_hierarchical.py:185-194, and tf.confusion_matrix in
 * estimator/define_metrics.py:10-12): cm[label*C + decision] += 1 for n pixels, int64,
 * accumulated into.  `lut` (optional, int32[lut_size]) remaps decisions first
 * (_map_predictions_to_new_cids, define_estimator_hierarchical.py:511-514).  Pairs outside
 * [0, C) are skipped and counted in *invalid (optional, int64).
 * ------------------------------------------------------------------------------------------ */
int wlseg_confmat_accumulate(const int32_t* labels, const int32_t* decisions, int64_t n,
                             int32_t num_classes, const int32_t* lut, int32_t lut_size,
                             int64_t* cm, int64_t* invalid, wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Optimizer (replaces tf.train.MomentumOptimizer + slim.l2_regularizer gradient,
 * estimator/define_optimizer.py:17-22, models/resnet50_extended_model_hierarchical.py:336):
 *   g' = g*grad_scale + wd*w (wd only for the first n_decay elements: conv kernels)
 *   acc = momentum*acc + g' ; w -= lr*acc   (nesterov: w -= lr*(g' + momentum*acc))
 * over flat fp32 buffers of n elements; w_bf16 (optional) receives the rounded copy;
 * reg_loss (optional, double) += wd/2 * sum_{i<n_decay} w_i^2 (pre-update weights).
 * lr is read from device memory (`lr_dev`, float[1]) so the step is CUDA-graph replayable.
 * ------------------------------------------------------------------------------------------ */
int wlseg_sgdm_step(float* w, const float* g, float* acc, void* w_bf16, int64_t n, int64_t n_decay,
                    const float* lr_dev, float momentum, int32_t nesterov, float wd,
                    float grad_scale, double* reg_loss, wlseg_stream_t stream);

/* Shadow variables of tf.train.ExponentialMovingAverage(decay, num_updates=global_step)
 * (estimator/define_estimator_hierarchical.py:96-111): biased <- biased - (1-decay)*(biased - w);
 * shadow = biased * inv_correction.  For tf.Variables TF initialises the shadow with the variable
 * and applies no zero-debiasing: pass biased == shadow and inv_correction = 1; a zero-debiased
 * average (plain tensors) passes a zero-initialised `biased` and 1/(1-decay^t). */
int wlseg_ema_update(float* biased, float* shadow, const float* w, int64_t n, float decay,
                     float inv_correction, wlseg_stream_t stream);

/* dst += src (n elements, n % 8 == 0): gradient fan-in of the residual connections
 * (tf.add_n of the gradients reaching one tensor in the reference's backward graph). */
int wlseg_add_inplace(void* dst, const void* src, int64_t n, int32_t dtype, wlseg_stream_t stream);

/* Layout / dtype helpers used by the host mirror (no reference counterpart: TF keeps HWIO
 * fp32 kernels; we keep KRSC bf16 operand copies). */
int wlseg_cast_f32_to_bf16(const float* src, void* dst, int64_t n, wlseg_stream_t stream);
int wlseg_cast_bf16_to_f32(const void* src, float* dst, int64_t n, wlseg_stream_t stream);
/* dst[k,r,s,c] (optionally rotated 180 degrees in r,s and with k<->c swapped: the kernel a
 * stride-1 dgrad runs as an fprop) from src KRSC. */
int wlseg_weights_transpose_flip(const void* src, void* dst, int32_t K, int32_t R, int32_t S,
                                 int32_t C, int32_t dtype, wlseg_stream_t stream);
/* The same for every layer of the network in one launch: `table` is int32[n_layers][6] on the
 * device, rows {src_off, dst_off, K, R, S, C} (element offsets into the two arenas). */
int wlseg_weights_transpose_flip_batched(const void* src_arena, void* dst_arena, const int32_t* table,
                                         int32_t n_layers, int32_t dtype, wlseg_stream_t stream);
/* dst[N,Hu,Wu,C] = src[N,P,Q,C] with stride-1 zeros inserted between the pixels (dst fully written).
 * The input gradient of a strided convolution (TF Conv2DBackpropInput) is a stride-1 convolution
 * over this tensor, which runs on the tensor cores. */
int wlseg_zero_insert(const void* src, void* dst, int32_t N, int32_t P, int32_t Q, int32_t C, int32_t stride,
                      int32_t Hu, int32_t Wu, int32_t dtype, wlseg_stream_t stream);
/* Packs a 3-channel NHWC image (fp32 or bf16) for the ResNet root convolution
 * (7x7 stride 2, models/resnet50_extended_feature_extractor.py:25-30) into the bf16 tensor
 * out[N, ceil(H/2), ceil(W/2), 64] = space-to-depth(2) with the 4 horizontal taps unrolled into
 * channels, so that conv1 runs on the tensor cores as an R=4, S=1, C=64 convolution
 * (csrc/transform.cu gives the exact index map). */
int wlseg_conv1_pack(const void* img, int32_t dtype, int32_t N, int32_t H, int32_t W, void* out,
                     wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Input-side resize + random crop, input_pipelines/utils.py:181-247 `resize_images_and_labels`
 * (over utils/utils.py:540-605): x [N,H,W,C] is resized to RH x RW with tf.image.resize_images,
 * align_corners=False (kind 0: fp32 BILINEAR for images; 1: fp32 NEAREST_NEIGHBOR for dense weak
 * labels; 2: int32 NEAREST_NEIGHBOR for class-id labels, C = 1) and the window [oy, oy+TH) x
 * [ox, ox+TW) of the result is written to y [N,TH,TW,C].  Without --preserve_aspect_ratio
 * RH x RW = TH x TW and the offsets are 0.
 * ------------------------------------------------------------------------------------------ */
int wlseg_resize_crop(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, int32_t RH,
                      int32_t RW, int32_t oy, int32_t ox, int32_t TH, int32_t TW, int32_t kind,
                      wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Evaluation inputs from raw bytes (the EVAL contract of SURVEY.md 3.5 as the reference's
 * evaluation pipeline produces it, with the arithmetic of _predict_preprocess,
 * input_pipelines/dataset_agnostic/dataset_agnostic_predict_input.py:109-119), for a batch whose
 * examples each have their own size:
 *   images    uint8 [N, cap_img]: row n holds an RGB image packed HWC, H_n x W_n x 3 bytes
 *   lids      uint8 [N, cap_lab]: row n holds its label-id map, H_n x W_n bytes
 *   sizes     int32 [N, 2] = (H_n, W_n)
 *   lut       int32 [n_lids], n_lids <= 256: label id -> class id (_replacevoids(lids2cids))
 *   proimages fp32  [N, TH, TW, 3] = (bilinear(u8 * (float)(1/255)) - 0.5) / 0.5, TF-1.12 legacy
 *             bilinear (align_corners=False), every operation rounded separately (bit-equal to
 *             wlseg/image_input.py)
 *   prolabels int32 [N, TH, TW] = lut[nearest(lids)], legacy nearest (align_corners=False)
 *   *invalid  int64, accumulated into (the caller zeroes): + 1 per label id >= n_lids (that pixel
 *             gets void_id) and + 1 per example whose size does not fit cap_img / cap_lab (its
 *             outputs are not written).
 * ------------------------------------------------------------------------------------------ */
int wlseg_eval_inputs(const uint8_t* images, int64_t cap_img, const uint8_t* lids, int64_t cap_lab,
                      const int32_t* sizes, int32_t N, const int32_t* lut, int32_t n_lids, int32_t void_id,
                      int32_t TH, int32_t TW, float* proimages, int32_t* prolabels, int64_t* invalid,
                      wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Training inputs (the per-pixel part of the TRAIN contract of SURVEY.md 3.5) gathered from a
 * device-resident arena of raw examples.  train.py does not preserve the aspect ratio of per-pixel
 * examples, so a training example is exactly the per-pixel arithmetic of wlseg_eval_inputs (one
 * shared device function):
 *   arena      uint8, ragged: example e starts at byte offsets[e] (int64: arenas exceed 4 GiB) with
 *              its RGB image packed HWC (H_e x W_e x 3 bytes), then its label-id map (H_e x W_e)
 *   sizes      int32 [n_examples, 2] = (H_e, W_e)
 *   index      int32 [N], device memory: output example n is arena example index[n]
 *   lut, void_id, TH, TW, proimages, prolabels: as wlseg_eval_inputs
 *   *invalid   int64, accumulated into (the caller zeroes): + 1 per label id >= n_lids (that pixel
 *              gets void_id) and + 1 per index outside [0, n_examples) or example of non-positive
 *              size (its outputs are not written).
 * ------------------------------------------------------------------------------------------ */
int wlseg_train_inputs(const uint8_t* arena, const int64_t* offsets, const int32_t* sizes, int32_t n_examples,
                       const int32_t* index, int32_t N, const int32_t* lut, int32_t n_lids, int32_t void_id,
                       int32_t TH, int32_t TW, float* proimages, int32_t* prolabels, int64_t* invalid,
                       wlseg_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Training inputs of one weak part of the batch (the bounding-box or the image-level examples
 * of the TRAIN contract of SURVEY.md 3.5) gathered from a device-resident arena of RGB images.
 * train.py preserves the aspect ratio of weak examples: example e (H x W) is resized to
 * resized[e] = (RH, RW) = wlseg.preprocess.resized_size(H, W, (TH, TW), True) and cropped to
 * TH x TW at the per-output offset crops[n] = (oy, ox).
 *   arena      uint8: example e is H_e x W_e x 3 bytes (RGB, HWC) at byte offsets[e] (int64)
 *   sizes, resized  int32 [n_examples, 2]
 *   box_start  int32 [n_examples + 1] or NULL: boxes [box_start[e], box_start[e + 1]) of example e
 *              in box_coords (fp32 [boxes, 4] = xmin, xmax, ymin, ymax normalised, 16-byte
 *              aligned) and box_cids (int32 [boxes], weak class id; ids outside 0..14 are skipped)
 *   vectors    fp32 [n_examples, 15] or NULL: one image-level multinomial per example.  Exactly one
 *              of box_start and vectors is given.
 *   index      int32 [N], crops int32 [N, 2]: output example n is arena example index[n] cut at
 *              crops[n]; N <= 65535
 *   proimages  fp32 [N, TH, TW, 3]: the image arithmetic of wlseg_train_inputs at the resized size
 *              (u8 / 255, legacy bilinear, [-1, 1)), sampled at (Y + oy, X + ox)
 *   labels     fp32 [N, TH, TW, 15]: bbox part = _generate_rla at H x W, then legacy nearest to
 *              RH x RW, then the crop (bit-equal to wlseg_rasterize_bbox_labels + wlseg_resize_crop);
 *              image-level part = vectors[index[n]] at every pixel
 *   *invalid   int64, accumulated into (the caller zeroes): + 1 per output example whose index is
 *              outside [0, n_examples), whose crop is outside [0, RH - TH] x [0, RW - TW], whose
 *              size is not positive or that has more than 1024 boxes (its outputs are not written).
 * ------------------------------------------------------------------------------------------ */
int wlseg_weak_train_inputs(const uint8_t* arena, const int64_t* offsets, const int32_t* sizes,
                            const int32_t* resized, int32_t n_examples, const int32_t* box_start,
                            const float* box_coords, const int32_t* box_cids, const float* vectors,
                            const int32_t* index, const int32_t* crops, int32_t N, int32_t TH, int32_t TW,
                            float* proimages, float* labels, int64_t* invalid, wlseg_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* WLSEG_H_ */
