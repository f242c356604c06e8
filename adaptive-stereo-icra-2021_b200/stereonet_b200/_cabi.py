"""ctypes binding of libsnb200.so (include/snb200.h).  Fails loudly when the library is missing: there is no fallback."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SNB200_LIB", os.path.join(os.path.dirname(_HERE), "libsnb200.so"))


class ConvGeom(C.Structure):
  _fields_ = [(n, C.c_int) for n in ("B", "D", "H", "W", "OD", "OH", "OW", "KD", "KH", "KW", "stride", "dil", "pd", "ph", "pw", "transposed")]


class ConvEpilogue(C.Structure):
  _fields_ = [("bias", C.c_void_p), ("scale", C.c_void_p), ("shift", C.c_void_p), ("residual", C.c_void_p),
              ("stats", C.c_void_p), ("lrelu", C.c_int)]


_P, _I, _F, _LL, _D = C.c_void_p, C.c_int, C.c_float, C.c_longlong, C.c_double
_GP, _EP = C.POINTER(ConvGeom), C.POINTER(ConvEpilogue)

# name -> (restype, argtypes); every symbol include/snb200.h declares
SIGNATURES = {
  "snb_last_error": (C.c_char_p, []),
  "snb_version": (_I, []),
  "snb_conv_c32_num_tiles": (_I, [_GP]),
  "snb_prep_conv_weights": (_I, [_P, _P, _I, _I, _I, _I, _P]),
  "snb_cost_volume_fwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
  "snb_cost_volume_bwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
  "snb_conv_c32": (_I, [_P, _P, _P, _GP, _EP, _P]),
  "snb_conv_c32_tc": (_I, [_P, _P, _P, _GP, _EP, _I, _P]),
  "snb_conv_c32_tc_num_tiles": (_I, [_GP]),
  "snb_conv2d_c32_tc": (_I, [_P, _P, _P, _GP, _EP, _I, _P]),
  "snb_conv2d_c32_tc_num_tiles": (_I, [_GP]),
  "snb_conv2d_c32_tc_profile": (_I, [_P, _P, _P, _GP, _EP, _I, _P, _P]),
  "snb_conv_c32_tc_profile": (_I, [_P, _P, _P, _GP, _EP, _I, _P, _P]),
  "snb_conv_c32_ws": (_I, [_P, _P, _P, _GP, _EP, _P]),
  "snb_conv_c32_ws_num_tiles": (_I, [_GP]),
  "snb_conv_c32_ws_f16": (_I, [_P, _P, _P, _GP, _EP, _P]),
  "snb_conv_weights_ws_floats": (_I, [_I]),
  "snb_conv_c32_ws_profile": (_I, [_P, _P, _P, _GP, _EP, _P, _P]),
  "snb_prep_conv_weights_tc": (_I, [_P, _P, _I, _I, _P]),
  "snb_conv_weights_tc_floats": (_I, [_I]),
  "snb_prep_conv_weights_tc_batch": (_I, [_P, _I, _P]),
  "snb_phase_split": (_I, [_P, _P, _I, _I, _I, _P]),
  "snb_phase_merge": (_I, [_P, _P, _I, _I, _I, _P]),
  "snb_conv5x5s2_c3": (_I, [_P, _P, _P, _P, _I, _I, _I, _P]),
  "snb_conv5x5s2_c3_phases": (_I, [_P, _P, _P, _P, _I, _I, _I, _P]),
  "snb_refine_in_conv": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _EP, _P]),
  "snb_refine_in_conv_num_tiles": (_I, [_I, _I, _I]),
  "snb_conv_c32_taps": (_I, [_P, _P, _P, _LL, _I, _I, _P]),
  "snb_tapsum_softargmin": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
  "snb_conv3d_out_softargmin": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
  "snb_tapsum_refine_out": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
  "snb_upsample_bilinear": (_I, [_P, _P, _I, _I, _I, _I, _I, _F, _P]),
  "snb_upsample_bilinear_bwd": (_I, [_P, _P, _I, _I, _I, _I, _I, _F, _P]),
  "snb_bn_finalize": (_I, [_P, _I, _LL, _P, _P, _P, _P, _F, _F, _P, _P, _P, _P, _P]),
  "snb_bn_finalize_ws": (_I, [_P, _I, _LL, _P, _P, _P, _P, _P, _F, _F, _P, _P, _P, _P, _P, _P]),
  "snb_bn_apply": (_I, [_P, _P, _P, _P, _P, _LL, _I, _P]),
  "snb_bwd_num_blocks": (_I, [_LL]),
  "snb_bn_lrelu_bwd_reduce": (_I, [_P, _P, _P, _P, _P, _P, _P, _LL, _I, _P]),
  "snb_bn_lrelu_bwd_apply": (_I, [_P, _P, _P, _P, _P, _P, _P, _LL, _I, _I, _P, _P, _P]),
  "snb_reduce_partials": (_I, [_P, _I, _I, _P, _F, _P]),
  "snb_reduce_wgrad_partials": (_I, [_P, _I, _I, _P, _P]),
  "snb_channel_sum": (_I, [_P, _P, _LL, _P]),
  "snb_conv_c32_wgrad": (_I, [_P, _P, _P, _GP, _P]),
  "snb_conv_c32_wgrad_num_partials": (_I, [_GP]),
  "snb_conv_c32_wgrad_tc": (_I, [_P, _P, _P, _GP, _I, _P]),
  "snb_conv_c32_wgrad_tc_num_partials": (_I, [_GP]),
  "snb_conv_c32_wgrad_tc_debug": (_I, [_P, _P, _P, _GP, _I, _P, _P]),
  "snb_conv5x5s2_c3_wgrad": (_I, [_P, _P, _P, _I, _I, _I, _P]),
  "snb_conv5x5s2_c3_num_tiles": (_I, [_I, _I, _I]),
  "snb_refine_in_wgrad": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P]),
  "snb_softargmin_bwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
  "snb_relu_bwd": (_I, [_P, _P, _P, _LL, _P]),
  "snb_feature_contrast": (_I, [_P, _P, _I, _I, _I, _I, _P]),
  "snb_photo_loss": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _P]),
  "snb_photo_loss_workspace_floats": (_I, [_I, _I, _I]),
  "snb_conv_c32_taps_bwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
  "snb_khamis_loss": (_I, [_P, _P, _P, _P, _P, _LL, _P]),
  "snb_khamis_loss_workspace_floats": (_I, [_LL]),
  "snb_eval_metrics": (_I, [_P, _P, _P, _I, _LL, _P]),
  "snb_multi_gather": (_I, [_P, _P, _P, _I, _P, _P]),
  "snb_adam_clip_step": (_I, [_P, _I, _P, _P, _P, _P, _LL, _LL, _F, _F, _D, _D, _D, _D, _P, _P]),
  "snb_adam_clip_workspace_bytes": (_I, []),
  "snb_conv5x5s2_c32_ws": (_I, [_P, _P, _P, _I, _I, _I, _EP, _P]),
  "snb_conv5x5s2_c32_ws_x": (_I, [_P, _P, _P, _I, _I, _I, _EP, _P]),
  "snb_refine_pack_input": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P]),
  "snb_conv_c4_ws": (_I, [_P, _P, _P, _I, _I, _I, _EP, _P]),
  "snb_bn_running_update": (_I, [_P, _P, _LL, _P, _P, _P, _F, _F, _P]),
  "snb_prep_conv5x5s2_weights_ws": (_I, [_P, _P, _P]),
  "snb_stereonet_num_params": (_I, [_I]),
  "snb_stereonet_weights_bytes": (_LL, [_I]),
  "snb_stereonet_weights_piece": (_I, [_I, _I, C.POINTER(_LL), C.POINTER(_LL)]),
  "snb_stereonet_prepare": (_I, [_P, _I, _P, _P]),
  "snb_stereonet_workspace_bytes": (_LL, [_I, _I, _I, _I, _I, _I]),
  "snb_stereonet_forward": (_I, [_P, _I, _I, _I, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P]),
  "snb_stereonet_forward_f16": (_I, [_P, _I, _I, _I, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P]),
  "snb_stereonet_adapt_state_bytes": (_LL, [_I]),
  "snb_stereonet_adapt_state_piece": (_I, [_I, _I, C.POINTER(_LL), C.POINTER(_LL)]),
  "snb_stereonet_adapt_grad_slot": (_I, [_I, _I, C.POINTER(_LL), C.POINTER(_LL)]),
  "snb_stereonet_adapt_init": (_I, [_P, _I, _P, _P]),
  "snb_stereonet_adapt_workspace_bytes": (_LL, [_I, _I, _I, _I, _I, _I]),
  "snb_stereonet_adapt_forward": (_I, [_P, _P, _I, _I, _I, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
  "snb_stereonet_adapt_update": (_I, [_P, _I, _I, _I, _I, _I, _I, _P, _P, _F, _D, _D, _D, _D, _P]),
  "snb_stereonet_adapt_replay_workspace_bytes": (_LL, [_I, _I, _I, _I, _I, _I, _I]),
  "snb_stereonet_adapt_forward_replay": (_I, [_P, _P, _I, _I, _I, _P, _I, _I, _I, _P, _P, _I, _F, _P, _P, _P, _P, _P, _P, _P, _P]),
  "snb_stereonet_adapt_update_replay": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _F, _D, _D, _D, _D, _P]),
}

_lib = None


def lib():
  """Load (once) and return the C-ABI library."""
  global _lib
  if _lib is None:
    if not os.path.exists(LIB_PATH):
      raise RuntimeError(
          f"stereonet_b200: {LIB_PATH} is missing. Build it with `python adaptive-stereo-icra-2021_b200/build.py` "
          "(nvcc, sm_100a). There is no CPU / eager fallback for this path.")
    l = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
      fn = getattr(l, name)
      fn.restype, fn.argtypes = res, args
    _lib = l
  return _lib


def check(rc, what):
  if rc != 0:
    raise RuntimeError(f"{what} failed: {lib().snb_last_error().decode()}")
