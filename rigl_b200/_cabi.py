"""ctypes binding of the C ABI in include/rigl_b200.h.

There is no CPU fallback: if librigl_b200.so is missing, `lib()` raises with
the build command.  Tensors are passed as raw device pointers (`data_ptr()`),
streams as the integer `cudaStream_t` of torch's current stream.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'librigl_b200.so')
_lib = None


class RiglError(RuntimeError):
  pass


class LayerDesc(C.Structure):
  _fields_ = [('weights', C.c_void_p), ('score_grow', C.c_void_p), ('mask_bits', C.c_void_p),
              ('noise', C.c_void_p), ('slots', C.c_void_p * 2), ('grow_values', C.c_void_p), ('score_drop', C.c_void_p),
              ('n', C.c_int64), ('n_prune_override', C.c_int32), ('flags', C.c_int32), ('noise_key', C.c_uint32),
              ('reserved', C.c_uint32), ('grad', C.c_void_p)]


class PackDesc(C.Structure):
  _fields_ = [('weights', C.c_void_p), ('mask_bits', C.c_void_p), ('packed', C.c_void_p),
              ('taps', C.c_int32), ('cin', C.c_int32), ('cout', C.c_int32), ('reserved', C.c_int32)]


class SgdDesc(C.Structure):
  _fields_ = [('param', C.c_void_p), ('momentum', C.c_void_p), ('grad', C.c_void_p), ('mask_bits', C.c_void_p),
              ('n', C.c_int64), ('weight_decay', C.c_float), ('grad_scale', C.c_float)]


class ConvDesc(C.Structure):
  _fields_ = [('batch', C.c_int32), ('in_h', C.c_int32), ('in_w', C.c_int32), ('cin', C.c_int32),
              ('out_h', C.c_int32), ('out_w', C.c_int32), ('cout', C.c_int32),
              ('ksize', C.c_int32), ('stride', C.c_int32), ('pad', C.c_int32), ('x_pitch', C.c_int32)]


GROW_ZEROS, GROW_TENSOR, GROW_GRAD_SCALE, GROW_GRAD_SIGN = 0, 1, 2, 3
LAYER_GROW_SCORE_SIGNED, LAYER_DROP_ONLY, LAYER_ALL_ACTIVE = 1, 2, 4

_vp, _i64, _i32, _f32, _sz = C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_size_t

# name -> (restype, argtypes); every symbol include/rigl_b200.h declares.
SIGNATURES = {
    'rigl_version': (C.c_int, []),
    'rigl_last_error': (C.c_char_p, []),
    'rigl_launch_count': (C.c_uint64, []),
    'rigl_mask_words': (_i64, [_i64]),
    'rigl_mask_pack_f32': (C.c_int, [_vp, _i64, _vp, _vp]),
    'rigl_mask_unpack_f32': (C.c_int, [_vp, _i64, _vp, _vp]),
    'rigl_mask_popcount': (C.c_int, [_vp, _i64, _vp, _vp]),
    'rigl_apply_mask_f32': (C.c_int, [_vp, _vp, _i64, _vp, _f32, _vp]),
    'rigl_mask_plan_create': (C.c_int, [C.POINTER(LayerDesc), _i32, C.POINTER(_vp)]),
    'rigl_mask_plan_destroy': (C.c_int, [_vp]),
    'rigl_mask_plan_workspace_bytes': (_sz, [_vp]),
    'rigl_mask_update_run': (C.c_int, [_vp, _f32, _i32, _f32, _f32, _i32, _vp, _sz, _vp]),
    'rigl_mask_update_run_noise': (C.c_int, [_vp, _f32, _i32, _f32, _f32, _i32, _f32, C.c_uint64, _vp, _sz, _vp]),
    'rigl_mask_noise_fill': (C.c_int, [_vp, _i64, C.c_uint32, _f32, C.c_uint64, _vp]),
    'rigl_mask_plan_read_stats': (C.c_int, [_vp, _vp, C.POINTER(C.c_int32), _vp]),
    'rigl_packed_weights_bytes': (_sz, [_i32, _i32, _i32]),
    'rigl_pack_masked_weights': (C.c_int, [_vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    'rigl_pack_plan_create': (C.c_int, [C.POINTER(PackDesc), _i32, C.POINTER(_vp)]),
    'rigl_pack_plan_destroy': (C.c_int, [_vp]),
    'rigl_pack_plan_run': (C.c_int, [_vp, _vp]),
    'rigl_sgd_plan_create': (C.c_int, [C.POINTER(SgdDesc), _i32, C.POINTER(_vp)]),
    'rigl_sgd_plan_destroy': (C.c_int, [_vp]),
    'rigl_sgd_plan_run': (C.c_int, [_vp, _vp, _f32, _i32, _vp]),
    'rigl_conv_workspace_bytes': (_sz, [C.POINTER(ConvDesc)]),
    'rigl_masked_conv2d_fprop': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'rigl_bn_partial_rows': (C.c_int, []),
    'rigl_set_bn_stats_always': (C.c_int, [_i32]),
    'rigl_masked_conv2d_fprop_bnstats': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, C.POINTER(C.c_int), _vp, _sz, _vp]),
    'rigl_masked_conv2d_fprop_affine': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _sz,
                                                  _vp]),
    'rigl_masked_conv2d_dgrad': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _sz, _vp]),
    'rigl_conv2d_wgrad_dense': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _f32, _vp, _sz, _vp]),
    'rigl_im2col_nhwc': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _i64, _vp]),
    'rigl_stem_s2d_supported': (C.c_int, [C.POINTER(ConvDesc)]),
    'rigl_stem_s2d_folded_bytes': (_sz, [C.POINTER(ConvDesc)]),
    'rigl_stem_s2d_packed_bytes': (_sz, [C.POINTER(ConvDesc)]),
    'rigl_stem_s2d_workspace_bytes': (_sz, [C.POINTER(ConvDesc)]),
    'rigl_stem_s2d_fold_input': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp]),
    'rigl_stem_s2d_pack_weights': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp]),
    'rigl_stem_s2d_fprop': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp]),
    'rigl_stem_s2d_wgrad': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _f32, _vp, _sz, _vp]),
    'rigl_smallc_supported': (C.c_int, [C.POINTER(ConvDesc)]),
    'rigl_smallc_padded_bytes': (_sz, [C.POINTER(ConvDesc)]),
    'rigl_smallc_packed_bytes': (_sz, [C.POINTER(ConvDesc)]),
    'rigl_smallc_workspace_bytes': (_sz, [C.POINTER(ConvDesc)]),
    'rigl_smallc_pad_input': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp]),
    'rigl_smallc_pack_weights': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp]),
    'rigl_smallc_fprop': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp]),
    'rigl_smallc_wgrad': (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _f32, _vp, _sz, _vp]),
    'rigl_bn_workspace_bytes': (_sz, [_i64, _i32]),
    'rigl_bn_forward_train': (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _f32, _f32, _i32, _vp, _vp, _vp, _vp,
                                        _vp, _vp, _vp, _vp, _sz, _vp, _vp]),
    'rigl_bn_forward_train_partials': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _f32, _f32, _i32, _vp, _vp,
                                                 _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'rigl_bn_apply': (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp]),
    'rigl_bn_backward': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp,
                                   _vp, _sz, _vp]),
    'rigl_bn_backward2': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp,
                                    _vp, _sz, _vp, _vp]),
    'rigl_depthwise3x3_workspace_bytes': (_sz, [_i32, _i32, _i32, _i32, _i32]),
    'rigl_depthwise3x3_fprop': (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    'rigl_depthwise3x3_dgrad': (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    'rigl_depthwise3x3_wgrad': (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _f32, _vp, _sz, _vp]),
    'rigl_maxpool_same_forward': (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    'rigl_maxpool_same_backward': (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    'rigl_set_force_simt': (C.c_int, [_i32]),
}


def lib():
  """Loads (once) and returns the ctypes handle; fails loudly if absent."""
  global _lib
  if _lib is None:
    if not os.path.exists(LIB_PATH):
      raise RiglError('librigl_b200.so not built: run `python -m rigl_b200.build` '
                      '(or __graft_entry__.build()); there is no CPU fallback')
    handle = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
      fn = getattr(handle, name)
      fn.restype = res
      fn.argtypes = args
    _lib = handle
  return _lib


def check(status, what=''):
  if status != 0:
    msg = lib().rigl_last_error().decode('utf-8', 'replace')
    raise RiglError('%s failed (%d): %s' % (what or 'rigl call', status, msg))


def stream_ptr():
  import torch
  return torch.cuda.current_stream().cuda_stream


def launch_count():
  return int(lib().rigl_launch_count())
