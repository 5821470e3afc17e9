"""ctypes binding of libwlseg.so (include/wlseg.h) for torch CUDA tensors.

PyTorch is plumbing here: it owns device memory and streams; every device op of the hot path is
a call into the hand-written sm_100a library.  There is NO CPU / eager fallback: if the library
is missing or a call fails, `WlsegError` is raised.
"""

import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libwlseg.so')

F32, BF16 = 0, 1
ALGO_AUTO, ALGO_DIRECT, ALGO_TCGEN05 = 0, 1, 2

_c_int = ctypes.c_int32
_c_i64 = ctypes.c_int64
_c_f = ctypes.c_float
_vp = ctypes.c_void_p


class WlsegError(RuntimeError):
  pass


class ConvParams(ctypes.Structure):
  _fields_ = [(n, _c_int) for n in (
      'N', 'H', 'W', 'C', 'K', 'R', 'S', 'P', 'Q', 'stride', 'dilation', 'pad_top', 'pad_left',
      'x_pitch', 'y_pitch', 'res_pitch', 'res_stride', 'res_H', 'res_W', 'relu', 'dtype', 'y_dtype', 'algo',
      'accumulate', 'reverse')]


class BnFinalizeArgs(ctypes.Structure):
  _fields_ = [('count', ctypes.c_int64), ('eps', ctypes.c_float), ('decay', ctypes.c_float),
              ('moving_var_factor', ctypes.c_float), ('reserved', ctypes.c_int32),
              ('gamma', ctypes.c_void_p), ('beta', ctypes.c_void_p), ('moving_mean', ctypes.c_void_p),
              ('moving_var', ctypes.c_void_p), ('scale', ctypes.c_void_p), ('shift', ctypes.c_void_p),
              ('saved_mean', ctypes.c_void_p), ('saved_invstd', ctypes.c_void_p), ('counter', ctypes.c_void_p)]


class Hierarchy(ctypes.Structure):
  _fields_ = [('C1', _c_int), ('Cv', _c_int), ('Ch', _c_int),
              ('cid_l1_vehicle', _c_int), ('cid_l1_human', _c_int),
              ('l1_to_common', _c_int * 64), ('veh_to_common', _c_int * 16), ('hum_to_common', _c_int * 8),
              ('num_classes', _c_int),
              ('pp_to_l1', _c_int * 80), ('pp_to_veh', _c_int * 80), ('pp_to_hum', _c_int * 80),
              ('bb_to_veh', _c_int * 15), ('bb_to_hum', _c_int * 15)]


_SIGNATURES = {
    'wlseg_version': (ctypes.c_int, []),
    'wlseg_last_error': (ctypes.c_char_p, []),
    'wlseg_conv2d_tcgen05_supported': (ctypes.c_int, [ctypes.POINTER(ConvParams)]),
    'wlseg_conv2d_fprop': (ctypes.c_int, [ctypes.POINTER(ConvParams), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'wlseg_conv2d_dgrad': (ctypes.c_int, [ctypes.POINTER(ConvParams), _vp, _vp, _vp, _vp]),
    'wlseg_conv2d_wgrad': (ctypes.c_int, [ctypes.POINTER(ConvParams), _vp, _vp, _vp, _vp]),
    'wlseg_bn_stats': (ctypes.c_int, [_vp, _c_i64, _c_int, _c_int, _c_int, _vp, _vp, _vp]),
    'wlseg_bn_finalize': (ctypes.c_int, [_vp, _vp, _c_i64, _c_int, _vp, _vp, _c_f, _c_f, _c_f, _vp, _vp, _vp, _vp, _vp,
                                         _vp, _vp]),
    'wlseg_bn_finalize_apply': (ctypes.c_int, [_vp, _vp, _c_i64, _c_int, _vp, _vp, _c_f, _c_f, _vp, _vp, _vp, _vp, _vp,
                                               _vp, _vp, _vp, _vp, _vp, _c_int, _c_int, _vp]),
    'wlseg_bn_apply': (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _c_i64, _c_int, _c_int, _c_int, _vp]),
    'wlseg_bn_apply_mask': (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_int, _c_int, _vp]),
    'wlseg_conv2d_fprop_masked': (ctypes.c_int, [ctypes.POINTER(ConvParams), _vp, _vp, _vp, _vp, _vp, _vp]),
    'wlseg_conv2d_fprop_bnbwd': (ctypes.c_int, [ctypes.POINTER(ConvParams)] + [_vp] * 11),
    'wlseg_conv2d_fprop_bn': (ctypes.c_int, [ctypes.POINTER(ConvParams), _vp, _vp, _vp, _vp, _vp,
                                             ctypes.POINTER(BnFinalizeArgs), _vp]),
    'wlseg_bn_bwd_reduce': (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_int, _c_int, _c_int, _c_int,
                                           _vp, _vp, _vp]),
    'wlseg_bn_bwd_apply': (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_int, _c_int,
                                          _c_int, _c_int, _vp, _vp, _vp]),
    'wlseg_maxpool_same_fwd': (ctypes.c_int, [_vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                              _vp]),
    'wlseg_maxpool_same_bwd': (ctypes.c_int, [_vp, _vp, _vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                              _c_int, _vp]),
    'wlseg_gn_finalize': (ctypes.c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_i64, _vp, _vp, _c_f, _vp, _vp, _vp, _vp, _vp]),
    'wlseg_gn_bwd_finalize': (ctypes.c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_i64] + [_vp] * 9),
    'wlseg_gn_bwd_apply': (ctypes.c_int, [_vp] * 8 + [_c_int, _c_i64, _c_int, _c_int, _c_int, _vp, _vp, _vp]),
    'wlseg_avgpool_valid_fwd': (ctypes.c_int, [_vp, _vp] + [_c_int] * 9 + [_vp]),
    'wlseg_avgpool_valid_bwd': (ctypes.c_int, [_vp, _vp] + [_c_int] * 8 + [_vp]),
    'wlseg_resize_bilinear_fwd': (ctypes.c_int, [_vp, _vp] + [_c_int] * 8 + [_vp]),
    'wlseg_resize_bilinear_bwd': (ctypes.c_int, [_vp, _vp] + [_c_int] * 8 + [_vp]),
    'wlseg_rasterize_bbox_labels': (ctypes.c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp]),
    'wlseg_tile_image_labels': (ctypes.c_int, [_vp, _c_int, _c_int, _c_int, _vp, _vp]),
    'wlseg_head_fwd': (ctypes.c_int, [ctypes.POINTER(Hierarchy), _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                      _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'wlseg_resize_probabilities': (ctypes.c_int, [_vp, _vp] + [_c_int] * 6 + [_vp]),
    'wlseg_resize_decisions': (ctypes.c_int, [_vp, _vp] + [_c_int] * 5 + [_vp]),
    'wlseg_replace_voids': (ctypes.c_int, [ctypes.POINTER(Hierarchy), _vp, _vp, _vp, _vp, _c_i64, _c_int, _vp]),
    'wlseg_loss_fwd_bwd': (ctypes.c_int, [ctypes.POINTER(Hierarchy), _vp, _c_int, _c_int, _c_int, _c_int, _c_int,
                                          _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'wlseg_loss_fwd_bwd_lists': (ctypes.c_int, [ctypes.POINTER(Hierarchy), _vp, _c_int, _c_int, _c_int, _c_int, _c_int,
                                                _c_int, _c_int, _c_int, _vp, _vp, _vp, _c_int, _vp, _vp, _vp, _vp, _vp]),
    'wlseg_loss_finalize': (ctypes.c_int, [ctypes.POINTER(Hierarchy), _vp, _vp, _c_f, _c_f, _vp, _c_int, _c_i64, _vp,
                                           _vp]),
    'wlseg_confmat_accumulate': (ctypes.c_int, [_vp, _vp, _c_i64, _c_int, _vp, _c_int, _vp, _vp, _vp]),
    'wlseg_head_confmat': (ctypes.c_int, [ctypes.POINTER(Hierarchy), _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                          _vp, _c_int, _vp, _c_int, _vp, _vp, _vp, _vp]),
    'wlseg_sgdm_step': (ctypes.c_int, [_vp, _vp, _vp, _vp, _c_i64, _c_i64, _vp, _c_f, _c_int, _c_f, _c_f, _vp, _vp]),
    'wlseg_ema_update': (ctypes.c_int, [_vp, _vp, _vp, _c_i64, _c_f, _c_f, _vp]),
    'wlseg_add_inplace': (ctypes.c_int, [_vp, _vp, _c_i64, _c_int, _vp]),
    'wlseg_cast_f32_to_bf16': (ctypes.c_int, [_vp, _vp, _c_i64, _vp]),
    'wlseg_cast_bf16_to_f32': (ctypes.c_int, [_vp, _vp, _c_i64, _vp]),
    'wlseg_weights_transpose_flip': (ctypes.c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _vp]),
    'wlseg_weights_transpose_flip_batched': (ctypes.c_int, [_vp, _vp, _vp, _c_int, _c_int, _vp]),
    'wlseg_zero_insert': (ctypes.c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _vp]),
    'wlseg_conv1_pack': (ctypes.c_int, [_vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp]),
    'wlseg_resize_crop': (ctypes.c_int, [_vp, _vp] + [_c_int] * 11 + [_vp]),
    'wlseg_eval_inputs': (ctypes.c_int, [_vp, _c_i64, _vp, _c_i64, _vp, _c_int, _vp, _c_int, _c_int, _c_int, _c_int, _vp,
                                         _vp, _vp, _vp]),
    'wlseg_train_inputs': (ctypes.c_int, [_vp, _vp, _vp, _c_int, _vp, _c_int, _vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp,
                                          _vp, _vp]),
    'wlseg_weak_train_inputs': (ctypes.c_int, [_vp, _vp, _vp, _vp, _c_int, _vp, _vp, _vp, _vp, _vp, _vp, _c_int, _c_int,
                                               _c_int, _vp, _vp, _vp, _vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None
launches = 0  # number of library kernels enqueued (bench.py's gpu_launches claim)


def lib():
  """Load libwlseg.so; fails loudly when it has not been built (no fallback path exists)."""
  global _lib
  if _lib is None:
    if not os.path.exists(LIB_PATH):
      raise WlsegError(
          f'{LIB_PATH} is missing: build it with `python __graft_entry__.py` (or wlseg build.py). '
          'wlseg has no CPU or eager fallback.')
    L = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
      fn = getattr(L, name)
      fn.restype = res
      fn.argtypes = args
    _lib = L
  return _lib


def _check(rc, what):
  if rc != 0:
    msg = lib().wlseg_last_error().decode('utf-8', 'replace')
    raise WlsegError(f'{what} failed (rc={rc}): {msg}')


def _ptr(t):
  if t is None:
    return None
  assert t.is_cuda, 'wlseg ops take CUDA tensors only'
  return t.data_ptr()


def _stream():
  return torch.cuda.current_stream().cuda_stream


def dtype_code(dt):
  if dt == torch.bfloat16:
    return BF16
  if dt == torch.float32:
    return F32
  raise WlsegError(f'unsupported dtype {dt}')


def _count(n=1):
  global launches
  launches += n


# ------------------------------------------------------------------------------------ convolution
def conv_params(x_shape, w_shape, stride=1, dilation=1, pad=(0, 0), out_hw=None, x_pitch=None, y_pitch=None,
                relu=False, dtype=BF16, y_dtype=None, algo=ALGO_AUTO, res=None, res_stride=1, accumulate=False,
                reverse=False):
  N, H, W, C = x_shape
  K, R, S, Cw = w_shape
  assert Cw == C, f'filter channels {Cw} != input channels {C}'
  p = ConvParams()
  p.N, p.H, p.W, p.C = N, H, W, C
  p.K, p.R, p.S = K, R, S
  p.stride, p.dilation = stride, dilation
  p.pad_top, p.pad_left = pad
  if out_hw is None:
    raise WlsegError('conv_params: out_hw required')
  p.P, p.Q = out_hw
  p.x_pitch = x_pitch if x_pitch is not None else C
  p.y_pitch = y_pitch if y_pitch is not None else K
  if res is not None:
    p.res_H, p.res_W, p.res_pitch = res.shape[1], res.shape[2], res.stride(2)
    p.res_stride = res_stride
  else:
    p.res_H = p.res_W = p.res_pitch = 0
    p.res_stride = 1
  p.relu = int(relu)
  p.dtype = dtype
  p.y_dtype = dtype if y_dtype is None else y_dtype
  p.algo = algo
  p.accumulate = int(accumulate)
  p.reverse = int(reverse)
  return p


def conv2d_fprop(p, x, w, y, scale=None, shift=None, residual=None, bn_sum=None, bn_sqsum=None):
  _check(lib().wlseg_conv2d_fprop(ctypes.byref(p), _ptr(x), _ptr(w), _ptr(y), _ptr(scale), _ptr(shift),
                                  _ptr(residual), _ptr(bn_sum), _ptr(bn_sqsum), _stream()), 'wlseg_conv2d_fprop')
  _count()
  return y


def conv2d_fprop_masked(p, x, w, y, residual, out_mask):
  """y = (conv(x, w) + residual) * mask: a data gradient leaving through the ReLU of the tensor it belongs to."""
  _count()
  _check(lib().wlseg_conv2d_fprop_masked(ctypes.byref(p), _ptr(x), _ptr(w), _ptr(y), _ptr(residual), _ptr(out_mask),
                                         _stream()), 'wlseg_conv2d_fprop_masked')


def pdl_enabled():
  """Mirror of pdl_enabled() in csrc/abi.cu (programmatic dependent launches, opt-in)."""
  return os.environ.get('WLSEG_PDL') is not None


def conv2d_fprop_bn(p, x, w, y, bn_sum, bn_sqsum, count, gamma, beta, eps, decay, moving_mean, moving_var, scale, shift,
                    saved_mean, saved_invstd, counter, moving_var_factor=-1.0):
  """conv2d_fprop with fused statistics + bn_finalize in one launch (the last CTA finalises); counter: one zeroed
  int32 device word shared by the layers of a stream."""
  fin = BnFinalizeArgs(count, eps, decay, moving_var_factor, 0, _ptr(gamma), _ptr(beta), _ptr(moving_mean),
                       _ptr(moving_var), _ptr(scale), _ptr(shift), _ptr(saved_mean), _ptr(saved_invstd), _ptr(counter))
  _count()
  _check(lib().wlseg_conv2d_fprop_bn(ctypes.byref(p), _ptr(x), _ptr(w), _ptr(y), _ptr(bn_sum), _ptr(bn_sqsum),
                                     ctypes.byref(fin), _stream()), 'wlseg_conv2d_fprop_bn')
  return y


def conv2d_fprop_bnbwd(p, x, w, y, z, scale, shift, mean, invstd, dgamma, dbeta):
  """y = conv(x, w) * relu'(z * scale + shift), with the BN backward sums of (y, z) accumulated into dgamma / dbeta
  by the epilogue (the res_* fields of p describe z)."""
  _count()
  _check(lib().wlseg_conv2d_fprop_bnbwd(ctypes.byref(p), _ptr(x), _ptr(w), _ptr(y), _ptr(z), _ptr(scale), _ptr(shift),
                                        _ptr(mean), _ptr(invstd), _ptr(dgamma), _ptr(dbeta), _stream()),
         'wlseg_conv2d_fprop_bnbwd')


def conv2d_dgrad(p, dy, w, dx):
  _check(lib().wlseg_conv2d_dgrad(ctypes.byref(p), _ptr(dy), _ptr(w), _ptr(dx), _stream()), 'wlseg_conv2d_dgrad')
  _count()
  return dx


def conv2d_wgrad(p, x, dy, dw):
  _check(lib().wlseg_conv2d_wgrad(ctypes.byref(p), _ptr(x), _ptr(dy), _ptr(dw), _stream()), 'wlseg_conv2d_wgrad')
  _count()
  return dw


def conv2d_tcgen05_supported(p):
  return bool(lib().wlseg_conv2d_tcgen05_supported(ctypes.byref(p)))


def conv1_pack(img, out):
  N, H, W, C = img.shape
  assert C == 3
  _check(lib().wlseg_conv1_pack(_ptr(img), dtype_code(img.dtype), N, H, W, _ptr(out), _stream()), 'wlseg_conv1_pack')
  _count()
  return out


def weights_transpose_flip(src, dst):
  K, R, S, C = src.shape
  _check(lib().wlseg_weights_transpose_flip(_ptr(src), _ptr(dst), K, R, S, C, dtype_code(src.dtype), _stream()),
         'wlseg_weights_transpose_flip')
  _count()
  return dst


def weights_transpose_flip_batched(src_arena, dst_arena, table):
  """table: int32 [L, 6] device tensor of {src_off, dst_off, K, R, S, C} rows."""
  assert table.dtype == torch.int32 and table.is_contiguous() and src_arena.dtype == dst_arena.dtype
  _check(lib().wlseg_weights_transpose_flip_batched(_ptr(src_arena), _ptr(dst_arena), _ptr(table), table.shape[0],
                                                    dtype_code(src_arena.dtype), _stream()),
         'wlseg_weights_transpose_flip_batched')
  _count()
  return dst_arena


def zero_insert(src, dst, stride):
  N, P, Q, C = src.shape
  _, Hu, Wu, _ = dst.shape
  assert src.is_contiguous() and dst.is_contiguous() and dst.shape[3] == C and src.dtype == dst.dtype
  _check(lib().wlseg_zero_insert(_ptr(src), _ptr(dst), N, P, Q, C, stride, Hu, Wu, dtype_code(src.dtype), _stream()),
         'wlseg_zero_insert')
  _count()
  return dst


def cast_f32_to_bf16(src, dst):
  _check(lib().wlseg_cast_f32_to_bf16(_ptr(src), _ptr(dst), src.numel(), _stream()), 'wlseg_cast_f32_to_bf16')
  _count()
  return dst


def cast_bf16_to_f32(src, dst):
  _check(lib().wlseg_cast_bf16_to_f32(_ptr(src), _ptr(dst), src.numel(), _stream()), 'wlseg_cast_bf16_to_f32')
  _count()
  return dst


# ------------------------------------------------------------------------------------ batch norm
def bn_stats(z, count, C, pitch, sum_, sqsum):
  _check(lib().wlseg_bn_stats(_ptr(z), count, C, pitch, dtype_code(z.dtype), _ptr(sum_), _ptr(sqsum), _stream()),
         'wlseg_bn_stats')
  _count()


def bn_finalize(sum_, sqsum, count, C, gamma, beta, eps, decay, moving_mean, moving_var, scale, shift, saved_mean,
                saved_invstd, moving_var_factor=-1.0):
  """moving_var_factor < 0: unbiased moving variance (default); >= 0: var * factor (--cross_replica_norm)."""
  _check(lib().wlseg_bn_finalize(_ptr(sum_), _ptr(sqsum), count, C, _ptr(gamma), _ptr(beta), eps, decay,
                                 moving_var_factor, _ptr(moving_mean), _ptr(moving_var), _ptr(scale), _ptr(shift),
                                 _ptr(saved_mean), _ptr(saved_invstd), _stream()), 'wlseg_bn_finalize')
  _count()


def bn_finalize_apply(sum_, sqsum, count, C, gamma, beta, eps, decay, moving_mean, moving_var, scale, shift, saved_mean,
                      saved_invstd, z, residual, y, relu, mask=None):
  _check(lib().wlseg_bn_finalize_apply(_ptr(sum_), _ptr(sqsum), count, C, _ptr(gamma), _ptr(beta), eps, decay,
                                       _ptr(moving_mean), _ptr(moving_var), _ptr(scale), _ptr(shift), _ptr(saved_mean),
                                       _ptr(saved_invstd), _ptr(z), _ptr(residual), _ptr(y), _ptr(mask), int(relu),
                                       dtype_code(z.dtype), _stream()), 'wlseg_bn_finalize_apply')
  _count()
  return y


def bn_apply(z, scale, shift, residual, y, count, C, relu, mask=None):
  """mask: uint8 [count, C / 8], receives the ReLU bit mask (y > 0) - see conv2d_fprop_masked."""
  if mask is not None:
    assert relu and mask.dtype == torch.uint8 and mask.numel() == count * (C // 8)
    _count()
    _check(lib().wlseg_bn_apply_mask(_ptr(z), _ptr(scale), _ptr(shift), _ptr(residual), _ptr(y), _ptr(mask), count, C,
                                     dtype_code(z.dtype), _stream()), 'wlseg_bn_apply_mask')
    return
  _check(lib().wlseg_bn_apply(_ptr(z), _ptr(scale), _ptr(shift), _ptr(residual), _ptr(y), count, C, int(relu),
                              dtype_code(z.dtype), _stream()), 'wlseg_bn_apply')
  _count()
  return y


def bn_bwd_reduce(dy, y, z, mean, invstd, count, C, relu, dgamma, dbeta, scale=None, shift=None, pitch=None):
  """y=None on a ReLU layer: mask from sign(fmaf(z, scale, shift)).  Channel slices: pass views and pitch."""
  _check(lib().wlseg_bn_bwd_reduce(_ptr(dy), _ptr(y), _ptr(z), _ptr(mean), _ptr(invstd), _ptr(scale), _ptr(shift),
                                   count, C, C if pitch is None else pitch, int(relu), dtype_code(z.dtype),
                                   _ptr(dgamma), _ptr(dbeta), _stream()), 'wlseg_bn_bwd_reduce')
  _count()


def bn_bwd_apply(dy, y, z, mean, invstd, gamma, dgamma, dbeta, count, C, relu, dz, dres=None, scale=None, shift=None,
                 pitch=None, stat_count=None):
  """stat_count: pixels dgamma / dbeta were summed over (replicas * count under --cross_replica_norm)."""
  _check(lib().wlseg_bn_bwd_apply(_ptr(dy), _ptr(y), _ptr(z), _ptr(mean), _ptr(invstd), _ptr(gamma), _ptr(scale),
                                  _ptr(shift), _ptr(dgamma), _ptr(dbeta), count, count if stat_count is None else stat_count,
                                  C, C if pitch is None else pitch,
                                  int(relu), dtype_code(z.dtype), _ptr(dz), _ptr(dres), _stream()),
         'wlseg_bn_bwd_apply')
  _count()
  return dz


# ------------------------------------------------------------------------------------ group norm
def gn_finalize(sum_nc, sqsum_nc, N, C, groups, hw, gamma, beta, eps, scale, shift, mean, invstd):
  _check(lib().wlseg_gn_finalize(_ptr(sum_nc), _ptr(sqsum_nc), N, C, groups, hw, _ptr(gamma), _ptr(beta), eps, _ptr(scale),
                                 _ptr(shift), _ptr(mean), _ptr(invstd), _stream()), 'wlseg_gn_finalize')
  _count()


def gn_bwd_finalize(dgamma_nc, dbeta_nc, N, C, groups, hw, gamma, mean, invstd, cA, c1, c0, dgamma, dbeta):
  _check(lib().wlseg_gn_bwd_finalize(_ptr(dgamma_nc), _ptr(dbeta_nc), N, C, groups, hw, _ptr(gamma), _ptr(mean),
                                     _ptr(invstd), _ptr(cA), _ptr(c1), _ptr(c0), _ptr(dgamma), _ptr(dbeta), _stream()),
         'wlseg_gn_bwd_finalize')
  _count()


def gn_bwd_apply(dy, y, z, cA, c1, c0, scale, shift, N, hw, C, relu, dz, dres=None):
  assert dy.is_contiguous() and z.is_contiguous() and dz.is_contiguous()
  _check(lib().wlseg_gn_bwd_apply(_ptr(dy), _ptr(y), _ptr(z), _ptr(cA), _ptr(c1), _ptr(c0), _ptr(scale), _ptr(shift), N, hw,
                                  C, int(relu), dtype_code(z.dtype), _ptr(dz), _ptr(dres), _stream()), 'wlseg_gn_bwd_apply')
  _count()
  return dz


# ------------------------------------------------------------------------------------ pooling
def maxpool_same_fwd(x, y, ksize, stride, argmax=None):
  """argmax: optional uint8 tensor shaped like y receiving each output's winning window position."""
  N, H, W, C = x.shape
  _check(lib().wlseg_maxpool_same_fwd(_ptr(x), _ptr(y), _ptr(argmax), N, H, W, C, ksize, stride,
                                      dtype_code(x.dtype), _stream()), 'wlseg_maxpool_same_fwd')
  _count()
  return y


def maxpool_same_bwd(x, dy, dx, ksize, stride, argmax=None):
  N, H, W, C = dx.shape
  _check(lib().wlseg_maxpool_same_bwd(_ptr(x), _ptr(argmax), _ptr(dy), _ptr(dx), N, H, W, C, ksize, stride,
                                      dtype_code(dx.dtype), _stream()), 'wlseg_maxpool_same_bwd')
  _count()
  return dx


# ------------------------------------------------------------------------------------ pyramid (PSP) module
def avgpool_valid_fwd(x, y, kh, kw):
  """VALID average pooling with stride == kernel (the PSP bins); y: [N, H // kh, W // kw, C]."""
  N, H, W, C = x.shape
  assert x.is_contiguous() and y.is_contiguous() and tuple(y.shape) == (N, (H - kh) // kh + 1, (W - kw) // kw + 1, C)
  _check(lib().wlseg_avgpool_valid_fwd(_ptr(x), _ptr(y), N, H, W, C, kh, kw, kh, kw, dtype_code(x.dtype), _stream()),
         'wlseg_avgpool_valid_fwd')
  _count()
  return y


def avgpool_valid_bwd(dy, dx, kh, kw, accumulate=False):
  N, H, W, C = dx.shape
  assert dy.is_contiguous() and dx.is_contiguous()
  _check(lib().wlseg_avgpool_valid_bwd(_ptr(dy), _ptr(dx), N, H, W, C, kh, kw, int(accumulate), dtype_code(dx.dtype),
                                       _stream()), 'wlseg_avgpool_valid_bwd')
  _count()
  return dx


def resize_bilinear_fwd(x, y):
  """x [N, h, w, C] dense -> y [N, H, W, C], possibly a channel slice of a wider tensor (pixel pitch)."""
  N, h, w, C = x.shape
  _, H, W, _ = y.shape
  assert x.is_contiguous() and y.shape[3] == C and y.stride(3) == 1
  _check(lib().wlseg_resize_bilinear_fwd(_ptr(x), _ptr(y), N, h, w, C, H, W, y.stride(2), dtype_code(x.dtype), _stream()),
         'wlseg_resize_bilinear_fwd')
  _count()
  return y


def resize_bilinear_bwd(dy, dx):
  N, h, w, C = dx.shape
  _, H, W, _ = dy.shape
  assert dx.is_contiguous() and dy.shape[3] == C and dy.stride(3) == 1
  _check(lib().wlseg_resize_bilinear_bwd(_ptr(dy), _ptr(dx), N, h, w, C, H, W, dy.stride(2), dtype_code(dx.dtype), _stream()),
         'wlseg_resize_bilinear_bwd')
  _count()
  return dx


# ------------------------------------------------------------------------------------ weak labels
def rasterize_bbox_labels(coords, cids, H, W, out=None):
  """coords fp32 [N, B, 4] (xmin, xmax, ymin, ymax, normalised), cids int32 [N, B] (-1 = padding) ->
  fp32 [N, H, W, 15] per-pixel multinomial (input_subset_bboxes_v2.py:74-98)."""
  N, B = cids.shape
  assert coords.dtype == torch.float32 and cids.dtype == torch.int32 and coords.is_contiguous() and cids.is_contiguous()
  assert tuple(coords.shape) == (N, B, 4)
  if out is None:
    out = torch.empty((N, H, W, 15), dtype=torch.float32, device=cids.device)
  _check(lib().wlseg_rasterize_bbox_labels(_ptr(coords), _ptr(cids), N, B, H, W, _ptr(out), _stream()),
         'wlseg_rasterize_bbox_labels')
  _count()
  return out


def tile_image_labels(vec, H, W, out=None):
  """vec fp32 [N, 15] -> fp32 [N, H, W, 15] (input_subset_image_labels.py:73-107)."""
  N = vec.shape[0]
  assert vec.dtype == torch.float32 and vec.is_contiguous() and vec.shape[1] == 15
  if out is None:
    out = torch.empty((N, H, W, 15), dtype=torch.float32, device=vec.device)
  _check(lib().wlseg_tile_image_labels(_ptr(vec), N, H, W, _ptr(out), _stream()), 'wlseg_tile_image_labels')
  _count()
  return out


# ------------------------------------------------------------------------------------ head / loss / metrics
def head_fwd(hier, logits, H, W, decisions=None, l1_decisions=None, l2v_decisions=None, l2h_decisions=None,
             l1_probs=None, l2v_probs=None, l2h_probs=None, fullres_logits=None):
  N, h, w, pitch = logits.shape
  assert logits.dtype == torch.float32 and logits.is_contiguous()
  _check(lib().wlseg_head_fwd(ctypes.byref(hier), _ptr(logits), pitch, N, h, w, H, W, _ptr(decisions),
                              _ptr(l1_decisions), _ptr(l2v_decisions), _ptr(l2h_decisions), _ptr(l1_probs),
                              _ptr(l2v_probs), _ptr(l2h_probs), _ptr(fullres_logits), _stream()), 'wlseg_head_fwd')
  _count()


def resize_probabilities(probs, H, W):
  """`_resize_predictions` for a probability map (define_estimator_hierarchical.py:552-558): bilinear,
  align_corners=True.  fp32 [N, h, w, C] -> [N, H, W, C]; the same tensor when the size is unchanged."""
  N, h, w, C = probs.shape
  if (h, w) == (H, W):
    return probs
  assert probs.dtype == torch.float32 and probs.is_contiguous()
  out = torch.empty((N, H, W, C), dtype=torch.float32, device=probs.device)
  _check(lib().wlseg_resize_probabilities(_ptr(probs), _ptr(out), N, h, w, C, H, W, _stream()),
         'wlseg_resize_probabilities')
  _count()
  return out


def resize_decisions(decs, H, W):
  """`_resize_predictions` for decisions (define_estimator_hierarchical.py:559-563): NEAREST_NEIGHBOR,
  align_corners=True.  int32 [N, h, w] -> [N, H, W]."""
  N, h, w = decs.shape
  if (h, w) == (H, W):
    return decs
  assert decs.dtype == torch.int32 and decs.is_contiguous()
  out = torch.empty((N, H, W), dtype=torch.int32, device=decs.device)
  _check(lib().wlseg_resize_decisions(_ptr(decs), _ptr(out), N, h, w, H, W, _stream()), 'wlseg_resize_decisions')
  _count()
  return out


def replace_voids(hier, l1_probs, l2v_probs, l2h_probs, decisions, void_cid):
  """`_replace_voids` (define_estimator_hierarchical.py:573-630) for the hierarchical classifier, in place."""
  n = decisions.numel()
  for t, c in ((l1_probs, hier.C1), (l2v_probs, hier.Cv), (l2h_probs, hier.Ch)):
    assert t.dtype == torch.float32 and t.is_contiguous() and t.numel() == n * c
  assert decisions.dtype == torch.int32 and decisions.is_contiguous()
  _check(lib().wlseg_replace_voids(ctypes.byref(hier), _ptr(l1_probs), _ptr(l2v_probs), _ptr(l2h_probs), _ptr(decisions),
                                   n, int(void_cid), _stream()), 'wlseg_replace_voids')
  _count()
  return decisions


def loss_fwd_bwd(hier, logits, H, W, strong_labels, bbox_labels, image_labels, sums, counts, dlogits):
  B, h, w, pitch = logits.shape
  ns = 0 if strong_labels is None else strong_labels.shape[0]
  nb = 0 if bbox_labels is None else bbox_labels.shape[0]
  ni = 0 if image_labels is None else image_labels.shape[0]
  assert ns + nb + ni == B, 'labels do not cover the batch'
  assert logits.dtype == torch.float32 and logits.is_contiguous() and dlogits.shape == logits.shape
  _check(lib().wlseg_loss_fwd_bwd(ctypes.byref(hier), _ptr(logits), pitch, ns, nb, ni, h, w, H, W,
                                  _ptr(strong_labels), _ptr(bbox_labels), _ptr(image_labels), _ptr(sums),
                                  _ptr(counts), _ptr(dlogits), _stream()), 'wlseg_loss_fwd_bwd')
  _count()


def loss_fwd_bwd_lists(hier, logits, H, W, strong_labels, box_coords, box_cids, image_vectors, sums, counts, dlogits):
  """loss_fwd_bwd with compact weak labels: box_coords fp32 [nb, max_boxes, 4] + box_cids int32 [nb, max_boxes] for
  the bbox images, image_vectors fp32 [ni, 15] for the image-level ones (batch order: strong, bbox, image)."""
  B, h, w, pitch = logits.shape
  ns = 0 if strong_labels is None else strong_labels.shape[0]
  nb = 0 if box_coords is None else box_coords.shape[0]
  ni = 0 if image_vectors is None else image_vectors.shape[0]
  assert ns + nb + ni == B, 'labels do not cover the batch'
  assert logits.dtype == torch.float32 and logits.is_contiguous() and dlogits.shape == logits.shape
  mb = 0 if box_coords is None else box_coords.shape[1]
  if nb:
    assert box_coords.dtype == torch.float32 and box_cids.dtype == torch.int32 and tuple(box_cids.shape) == (nb, mb)
    box_coords, box_cids = box_coords.contiguous(), box_cids.contiguous()
  if ni:
    assert image_vectors.dtype == torch.float32 and image_vectors.shape[1] == 15
    image_vectors = image_vectors.contiguous()
  _check(lib().wlseg_loss_fwd_bwd_lists(ctypes.byref(hier), _ptr(logits), pitch, ns, nb, ni, h, w, H, W,
                                        _ptr(strong_labels), _ptr(box_coords), _ptr(box_cids), mb, _ptr(image_vectors),
                                        _ptr(sums), _ptr(counts), _ptr(dlogits), _stream()), 'wlseg_loss_fwd_bwd_lists')
  _count()


def loss_finalize(hier, sums, counts, l2_coef, grad_scale, dlogits, losses):
  pitch = dlogits.shape[-1] if dlogits is not None else hier.C1 + hier.Cv + hier.Ch
  npix = 0 if dlogits is None else dlogits.numel() // pitch
  _check(lib().wlseg_loss_finalize(ctypes.byref(hier), _ptr(sums), _ptr(counts), l2_coef, grad_scale, _ptr(dlogits),
                                   pitch, npix, _ptr(losses), _stream()), 'wlseg_loss_finalize')
  _count()


def head_confmat(hier, logits, H, W, labels, num_classes, cm, lut=None, invalid=None, decisions=None):
  """Low-res logits -> hierarchical decisions -> cm[label, lut[decision]] += 1 in one launch (wlseg_head_confmat);
  decisions: optional int32 [N, H, W] output; labels None = decisions only."""
  N, h, w, pitch = logits.shape
  assert logits.dtype == torch.float32 and logits.is_contiguous()
  if labels is not None:
    assert labels.dtype == torch.int32 and labels.is_contiguous() and tuple(labels.shape) == (N, H, W)
    assert cm.dtype == torch.int64 and cm.is_contiguous()
  _check(lib().wlseg_head_confmat(ctypes.byref(hier), _ptr(logits), pitch, N, h, w, H, W, _ptr(labels), num_classes,
                                  _ptr(lut), 0 if lut is None else lut.numel(), _ptr(cm), _ptr(invalid), _ptr(decisions),
                                  _stream()), 'wlseg_head_confmat')
  _count()
  return cm


def confmat_accumulate(labels, decisions, num_classes, cm, lut=None, invalid=None):
  assert labels.dtype == torch.int32 and decisions.dtype == torch.int32 and cm.dtype == torch.int64
  assert labels.numel() == decisions.numel() and labels.is_contiguous() and decisions.is_contiguous()
  assert cm.numel() == num_classes * num_classes
  _check(lib().wlseg_confmat_accumulate(_ptr(labels), _ptr(decisions), labels.numel(), num_classes, _ptr(lut),
                                        0 if lut is None else lut.numel(), _ptr(cm), _ptr(invalid), _stream()),
         'wlseg_confmat_accumulate')
  _count()
  return cm


def sgdm_step(w, g, acc, w_bf16, n_decay, lr_dev, momentum, nesterov, wd, grad_scale=1.0, reg_loss=None):
  _check(lib().wlseg_sgdm_step(_ptr(w), _ptr(g), _ptr(acc), _ptr(w_bf16), w.numel(), n_decay, _ptr(lr_dev), momentum,
                               int(nesterov), wd, grad_scale, _ptr(reg_loss), _stream()), 'wlseg_sgdm_step')
  _count()


def ema_update(biased, shadow, w, decay, inv_correction):
  _check(lib().wlseg_ema_update(_ptr(biased), _ptr(shadow), _ptr(w), w.numel(), decay, inv_correction, _stream()),
         'wlseg_ema_update')
  _count()


def add_inplace(dst, src):
  assert dst.is_contiguous() and src.is_contiguous() and dst.numel() == src.numel() and dst.dtype == src.dtype
  _check(lib().wlseg_add_inplace(_ptr(dst), _ptr(src), dst.numel(), dtype_code(dst.dtype), _stream()),
         'wlseg_add_inplace')
  _count()
  return dst


def resize_crop(x, resized_hw, offset, target_hw, kind):
  """tf.image.resize_images(align_corners=False) to `resized_hw` + crop of the `target_hw` window at `offset`, one pass
  (input_pipelines/utils.py:181-247).  kind: 'bilinear' (fp32 images), 'nearest' (fp32 dense labels or int32 ids)."""
  squeeze = x.dim() == 3
  xx = x.unsqueeze(-1) if squeeze else x
  N, H, W, C = xx.shape
  if kind == 'bilinear':
    assert xx.dtype == torch.float32
    k = 0
  else:
    assert xx.dtype in (torch.float32, torch.int32)
    k = 1 if xx.dtype == torch.float32 else 2
  y = torch.empty((N, target_hw[0], target_hw[1], C), dtype=xx.dtype, device=xx.device)
  _check(lib().wlseg_resize_crop(_ptr(xx.contiguous()), _ptr(y), N, H, W, C, int(resized_hw[0]), int(resized_hw[1]),
                                 int(offset[0]), int(offset[1]), int(target_hw[0]), int(target_hw[1]), k, _stream()),
         'wlseg_resize_crop')
  _count()
  return y.squeeze(-1) if squeeze else y


def eval_inputs(images, lids, sizes, lut, void_id, target_hw, proimages, prolabels, invalid):
  """Raw examples of their own sizes -> the evaluation contract, one launch (wlseg_eval_inputs).  images uint8
  [N, cap_img] (RGB packed HWC per row), lids uint8 [N, cap_lab], sizes int32 [N, 2] = (H, W), lut int32 [<= 256]
  label id -> class id.  Writes proimages fp32 [N, TH, TW, 3] and prolabels int32 [N, TH, TW]; invalid (int64 [1]) +=
  the out-of-range label ids and the examples whose size does not fit their row."""
  N = images.shape[0]
  TH, TW = int(target_hw[0]), int(target_hw[1])
  assert images.dtype == torch.uint8 and lids.dtype == torch.uint8 and images.dim() == 2 and lids.dim() == 2
  assert images.is_contiguous() and lids.is_contiguous() and lids.shape[0] == N
  assert sizes.dtype == torch.int32 and sizes.is_contiguous() and tuple(sizes.shape) == (N, 2)
  assert lut.dtype == torch.int32 and lut.is_contiguous() and lut.dim() == 1
  assert proimages.dtype == torch.float32 and proimages.is_contiguous() and tuple(proimages.shape) == (N, TH, TW, 3)
  assert prolabels.dtype == torch.int32 and prolabels.is_contiguous() and tuple(prolabels.shape) == (N, TH, TW)
  assert invalid.dtype == torch.int64
  _check(lib().wlseg_eval_inputs(_ptr(images), images.shape[1], _ptr(lids), lids.shape[1], _ptr(sizes), N, _ptr(lut),
                                 lut.numel(), int(void_id), TH, TW, _ptr(proimages), _ptr(prolabels), _ptr(invalid),
                                 _stream()), 'wlseg_eval_inputs')
  _count()
  return proimages, prolabels


def train_inputs(arena, offsets, sizes, index, lut, void_id, target_hw, proimages, prolabels, invalid):
  """Arena examples selected by a device index vector -> the per-pixel training contract, one launch
  (wlseg_train_inputs).  arena uint8 [bytes] (example e at offsets[e]: RGB HWC, then its label-id map), offsets int64
  [E], sizes int32 [E, 2] = (H, W), index int32 [N], lut int32 [<= 256] label id -> class id.  Writes proimages fp32
  [N, TH, TW, 3] and prolabels int32 [N, TH, TW]; invalid (int64 [1]) += the out-of-range label ids and indices."""
  N = index.numel()
  E = offsets.numel()
  TH, TW = int(target_hw[0]), int(target_hw[1])
  assert arena.dtype == torch.uint8 and arena.dim() == 1 and arena.is_contiguous()
  assert offsets.dtype == torch.int64 and offsets.is_contiguous() and offsets.dim() == 1
  assert sizes.dtype == torch.int32 and sizes.is_contiguous() and tuple(sizes.shape) == (E, 2)
  assert index.dtype == torch.int32 and index.is_contiguous() and index.dim() == 1
  assert lut.dtype == torch.int32 and lut.is_contiguous() and lut.dim() == 1
  assert proimages.dtype == torch.float32 and proimages.is_contiguous() and tuple(proimages.shape) == (N, TH, TW, 3)
  assert prolabels.dtype == torch.int32 and prolabels.is_contiguous() and tuple(prolabels.shape) == (N, TH, TW)
  assert invalid.dtype == torch.int64
  _check(lib().wlseg_train_inputs(_ptr(arena), _ptr(offsets), _ptr(sizes), E, _ptr(index), N, _ptr(lut), lut.numel(),
                                  int(void_id), TH, TW, _ptr(proimages), _ptr(prolabels), _ptr(invalid), _stream()),
         'wlseg_train_inputs')
  _count()
  return proimages, prolabels


def weak_train_inputs(arena, offsets, sizes, resized, index, crops, target_hw, proimages, labels, invalid, boxes=None,
                      vectors=None):
  """Arena images selected by a device index vector and cut at per-output crop offsets -> one weak part of the training
  contract, one launch (wlseg_weak_train_inputs).  arena uint8 [bytes] (example e: RGB HWC at offsets[e]), offsets int64
  [E], sizes / resized int32 [E, 2] = (H, W) / the aspect-preserving resized size, index int32 [N], crops int32 [N, 2] =
  (oy, ox).  Exactly one of boxes = (box_start int32 [E + 1], box_coords fp32 [B, 4] = xmin, xmax, ymin, ymax,
  box_cids int32 [B]) for the bounding-box part and vectors fp32 [E, 15] for the image-level part.  Writes proimages
  fp32 [N, TH, TW, 3] and labels fp32 [N, TH, TW, 15]; invalid (int64 [1]) += the out-of-range indices and crops."""
  N, E = index.numel(), offsets.numel()
  TH, TW = int(target_hw[0]), int(target_hw[1])
  assert (boxes is None) != (vectors is None), 'one of boxes (bounding-box part) and vectors (image-level part)'
  assert arena.dtype == torch.uint8 and arena.dim() == 1 and arena.is_contiguous()
  assert offsets.dtype == torch.int64 and offsets.is_contiguous() and offsets.dim() == 1
  for t in (sizes, resized):
    assert t.dtype == torch.int32 and t.is_contiguous() and tuple(t.shape) == (E, 2)
  assert index.dtype == torch.int32 and index.is_contiguous() and index.dim() == 1
  assert crops.dtype == torch.int32 and crops.is_contiguous() and tuple(crops.shape) == (N, 2)
  assert proimages.dtype == torch.float32 and proimages.is_contiguous() and tuple(proimages.shape) == (N, TH, TW, 3)
  assert labels.dtype == torch.float32 and labels.is_contiguous() and tuple(labels.shape) == (N, TH, TW, 15)
  assert invalid.dtype == torch.int64
  start = coords = cids = None
  if boxes is not None:
    start, coords, cids = boxes
    assert start.dtype == torch.int32 and start.is_contiguous() and tuple(start.shape) == (E + 1,)
    assert coords.dtype == torch.float32 and coords.is_contiguous() and coords.dim() == 2 and coords.shape[1] == 4
    assert cids.dtype == torch.int32 and cids.is_contiguous() and tuple(cids.shape) == (coords.shape[0],)
  else:
    assert vectors.dtype == torch.float32 and vectors.is_contiguous() and tuple(vectors.shape) == (E, 15)
  _check(lib().wlseg_weak_train_inputs(_ptr(arena), _ptr(offsets), _ptr(sizes), _ptr(resized), E, _ptr(start),
                                       _ptr(coords), _ptr(cids), _ptr(vectors), _ptr(index), _ptr(crops), N, TH, TW,
                                       _ptr(proimages), _ptr(labels), _ptr(invalid), _stream()), 'wlseg_weak_train_inputs')
  _count()
  return proimages, labels
