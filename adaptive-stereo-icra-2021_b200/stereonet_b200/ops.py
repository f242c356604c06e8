"""Thin torch-tensor wrappers over the C-ABI (libsnb200.so).  Device memory, streams and shapes are handled here;
every arithmetic instruction runs in the library's CUDA kernels.  Activations are contiguous channels-last fp32
tensors: [B,H,W,32] or [B,D,H,W,32]."""
import ctypes as C

import torch

from . import _cabi
from ._cabi import ConvEpilogue, ConvGeom, check

BN_EPS = 1e-5        # nn.BatchNorm2d/3d defaults used by the reference (stereo_net.py:17,29)
BN_MOMENTUM = 0.1

LAUNCHES = 0         # number of library kernels launched (bench.py reports it as gpu_launches)


def _count(n=1):
  global LAUNCHES
  LAUNCHES += n


def _p(t):
  return None if t is None else C.c_void_p(t.data_ptr())


def _stream(t):
  return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _req(t, name, ndim=None):
  if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
    raise RuntimeError(f"stereonet_b200: `{name}` must be a contiguous fp32 CUDA tensor "
                       f"(got {type(t).__name__} {getattr(t, 'dtype', None)} {getattr(t, 'device', None)})")
  if ndim is not None and t.dim() != ndim:
    raise RuntimeError(f"stereonet_b200: `{name}` must have {ndim} dims, got {tuple(t.shape)}")
  return t


def geom(x_shape, ksize, stride=1, dil=1, pad=None):
  """ConvGeom for a channels-last input of shape [B,H,W,32] (2-D) or [B,D,H,W,32] (3-D), cubic/square kernel."""
  three_d = len(x_shape) == 5
  if three_d:
    B, D, H, W, _ = x_shape
  else:
    B, H, W, _ = x_shape
    D = 1
  if pad is None:
    pad = dil * (ksize - 1) // 2
  OH = (H + 2 * pad - dil * (ksize - 1) - 1) // stride + 1
  OW = (W + 2 * pad - dil * (ksize - 1) - 1) // stride + 1
  g = ConvGeom(B, D, H, W, D, OH, OW, ksize if three_d else 1, ksize, ksize, stride, dil, 1 if three_d else 0, pad, pad, 0)
  if three_d:
    g.OD = D + 2 * 1 - (ksize - 1) - 1 + 1
  return g


def geom_transposed(g):
  """Geometry of the data gradient of conv `g`: reads dy [B,OD,OH,OW], writes dx [B,D,H,W] (snb_conv_geom.transposed)."""
  return ConvGeom(g.B, g.OD, g.OH, g.OW, g.D, g.H, g.W, g.KD, g.KH, g.KW, g.stride, g.dil, g.pd, g.ph, g.pw, 1)


def out_shape(g, three_d):
  return (g.B, g.OD, g.OH, g.OW, 32) if three_d else (g.B, g.OH, g.OW, 32)


def prep_conv_weights(w, mode=0):
  """[Cout,Cin,*k] -> [taps,Cin,Cout] (mode 0) or the flipped/transposed data-gradient layout (mode 1)."""
  w = _req(w.detach().contiguous(), "weight")
  cout, cin = w.shape[0], w.shape[1]
  taps = w[0, 0].numel()
  out = torch.empty((taps, cin, cout) if mode == 0 else (taps, cout, cin), device=w.device, dtype=torch.float32)
  if mode not in (0, 1, 2):
    raise ValueError(mode)
  check(_cabi.lib().snb_prep_conv_weights(_p(w), _p(out), cout, cin, taps, mode, _stream(w)), "snb_prep_conv_weights")
  _count()
  return out


def cost_volume(left, right, D):
  _req(left, "left_features", 4); _req(right, "right_features", 4)
  B, H, W, Cc = left.shape
  if Cc != 32 or right.shape != left.shape:
    raise RuntimeError(f"stereonet_b200: feature maps must be [B,H,W,32] and equal-shaped, got {tuple(left.shape)} {tuple(right.shape)}")
  cost = torch.empty((B, D, H, W, 32), device=left.device, dtype=torch.float32)
  check(_cabi.lib().snb_cost_volume_fwd(_p(left), _p(right), _p(cost), B, D, H, W, _stream(left)), "snb_cost_volume_fwd")
  _count()
  return cost


def cost_volume_bwd(dcost):
  _req(dcost, "dcost", 5)
  B, D, H, W, _ = dcost.shape
  dl = torch.empty((B, H, W, 32), device=dcost.device, dtype=torch.float32)
  dr = torch.empty_like(dl)
  check(_cabi.lib().snb_cost_volume_bwd(_p(dcost), _p(dl), _p(dr), B, D, H, W, _stream(dcost)), "snb_cost_volume_bwd")
  _count()
  return dl, dr


def conv_c32(x, wprep, g, bias=None, scale=None, shift=None, residual=None, lrelu=False, want_stats=False, out=None):
  """32->32 convolution + fused epilogue.  Returns (y, stats) with stats = [ntiles,2,32] partial sums or None."""
  three_d = x.dim() == 5
  _req(x, "x"); _req(wprep, "wprep")
  y = out if out is not None else torch.empty(out_shape(g, three_d), device=x.device, dtype=torch.float32)
  stats = None
  if want_stats:
    nt = _cabi.lib().snb_conv_c32_num_tiles(C.byref(g))
    stats = torch.empty((nt, 2, 32), device=x.device, dtype=torch.float32)
  if residual is not None:
    _req(residual, "residual")
    if residual.shape != y.shape:
      raise RuntimeError("stereonet_b200: residual shape mismatch")
  e = ConvEpilogue(_p(bias), _p(scale), _p(shift), _p(residual), _p(stats), 1 if lrelu else 0)
  check(_cabi.lib().snb_conv_c32(_p(x), _p(wprep), _p(y), C.byref(g), C.byref(e), _stream(x)), "snb_conv_c32")
  _count()
  return y, stats


CONV_F16 = 0x10      # SNB_CONV_F16: fp16-split operands on the round-1 kernels (3-D TMA kernel, 2-D N = 96 walk kernel)
CONV_WS = 0x20       # SNB_CONV_WS: weight image layout of snb_conv_c32_ws, the product kernel


def _fmt_of(fmt):
  """Operand format of the tensor-core convolutions -> (prep mode bits, passes argument).  "ws": snb_conv_c32_ws (product);
  "h": fp16 split on the round-1 kernels; 3: 3xTF32 split; 1: single-pass TF32."""
  if fmt == "ws":
    return CONV_WS, 3
  if fmt == "h":
    return CONV_F16, 3 | CONV_F16
  if fmt in (3, 1):
    return 0, fmt
  raise ValueError(f"unknown tensor-core operand format {fmt!r}")


def prep_conv_weights_tc(w, mode=0, fmt="ws"):
  """[32,32,(3,)3,3] -> tensor-core B-operand image for operand format `fmt` (see _fmt_of / snb_prep_conv_weights_tc)."""
  w = _req(w.detach().contiguous(), "weight")
  if w.shape[0] != 32 or w.shape[1] != 32 or tuple(w.shape[-2:]) != (3, 3):
    raise RuntimeError(f"stereonet_b200: tensor-core conv needs a [32,32,(3,)3,3] weight, got {tuple(w.shape)}")
  kd = 3 if w.dim() == 5 else 1
  bits, _ = _fmt_of(fmt)
  lib = _cabi.lib()
  n = lib.snb_conv_weights_ws_floats(kd) if bits == CONV_WS else lib.snb_conv_weights_tc_floats(kd)
  out = torch.empty((n,), device=w.device, dtype=torch.float32)
  check(lib.snb_prep_conv_weights_tc(_p(w), _p(out), kd, mode | bits, _stream(w)), "snb_prep_conv_weights_tc")
  _count(2 if bits else 1)
  return out


def conv_weights_tc_floats(kd, fmt="ws"):
  lib = _cabi.lib()
  return lib.snb_conv_weights_ws_floats(kd) if fmt == "ws" else lib.snb_conv_weights_tc_floats(kd)


def prep_conv5x5s2_weights_ws(w):
  """[32,32,5,5] weight -> the ten-image set of conv5x5s2_c32_ws (snb_prep_conv5x5s2_weights_ws)."""
  _req(w, "weight", 4)
  if tuple(w.shape) != (32, 32, 5, 5):
    raise RuntimeError(f"stereonet_b200: expected a [32,32,5,5] weight, got {tuple(w.shape)}")
  out = torch.empty((_cabi.lib().snb_conv_weights_ws_floats(5),), device=w.device, dtype=torch.float32)
  check(_cabi.lib().snb_prep_conv5x5s2_weights_ws(_p(w), _p(out), _stream(w)), "snb_prep_conv5x5s2_weights_ws")
  _count(2)
  return out


def conv5x5s2_c32_ws(phases, wimg, bias=None, lrelu=False):
  """5x5 stride-2 pad-2 32->32 conv over the polyphase images [4,B,OH,OW,32] of its input, ONE tensor-core launch."""
  _req(phases, "phases", 5); _req(wimg, "wimg")
  if phases.shape[0] != 4 or phases.shape[-1] != 32:
    raise RuntimeError(f"stereonet_b200: phases must be [4,B,OH,OW,32], got {tuple(phases.shape)}")
  _, B, OH, OW, _ = phases.shape
  y = torch.empty((B, OH, OW, 32), device=phases.device, dtype=torch.float32)
  e = ConvEpilogue(_p(bias), None, None, None, None, 1 if lrelu else 0)
  check(_cabi.lib().snb_conv5x5s2_c32_ws(_p(phases), _p(wimg), _p(y), B, OH, OW, C.byref(e), _stream(phases)), "snb_conv5x5s2_c32_ws")
  _count()
  return y


def conv5x5s2_c32_ws_x(x, wimg, bias=None, lrelu=False):
  """5x5 stride-2 pad-2 32->32 conv straight from the un-split input [B,H,W,32] (strided TMA views; H, W >= 2)."""
  _req(x, "x", 4); _req(wimg, "wimg")
  B, H, W, _ = x.shape
  y = torch.empty((B, (H + 1) // 2, (W + 1) // 2, 32), device=x.device, dtype=torch.float32)
  e = ConvEpilogue(_p(bias), None, None, None, None, 1 if lrelu else 0)
  check(_cabi.lib().snb_conv5x5s2_c32_ws_x(_p(x), _p(wimg), _p(y), B, H, W, C.byref(e), _stream(x)), "snb_conv5x5s2_c32_ws_x")
  _count()
  return y


def prep_conv_weights_tc_batch(table, n):
  """One launch for n weight images; `table` is an int64 device tensor [n,4] (see snb_prep_conv_weights_tc_batch)."""
  check(_cabi.lib().snb_prep_conv_weights_tc_batch(_p(table), n, _stream(table)), "snb_prep_conv_weights_tc_batch")
  _count(2)


def conv_c32_tc(x, wimg, g, bias=None, scale=None, shift=None, residual=None, lrelu=False, want_stats=False, fmt="ws",
                flat=False, out=None, legacy3d=False):
  """Tensor-core (tcgen05) 32->32 'same' 3x3 / 3x3x3 convolution + fused epilogue; returns (y, stats) with stats = [ntiles,2,32]
  partial sums or None.  `fmt` (see _fmt_of) selects the kernel and must match the format `wimg` was prepared in:
  "ws" -> snb_conv_c32_ws (product path, 2-D and 3-D); "h" / 3 / 1 -> the round-1 kernels (2-D: snb_conv2d_c32_tc walk kernel,
  flat=True: the flat-tiled loader-warp kernel; 3-D: the TMA kernel, legacy3d: the loader-warp one) kept as cross-checks."""
  three_d = x.dim() == 5
  _req(x, "x"); _req(wimg, "wimg")
  lib = _cabi.lib()
  bits, passes = _fmt_of(fmt)
  use_ws = bits == CONV_WS
  if use_ws and (flat or legacy3d):
    raise RuntimeError("stereonet_b200: flat / legacy3d select round-1 kernels; use fmt 'h', 3 or 1 with them")
  if fmt == "h" and ((flat and not three_d) or legacy3d):
    raise RuntimeError("stereonet_b200: the fp16 operand split runs on the TMA / walk kernels only")
  if use_ws and want_stats and (scale is not None or lrelu or residual is not None):
    raise RuntimeError("stereonet_b200: snb_conv_c32_ws takes BN statistics of the plain conv + bias output only")
  use2d = (not three_d) and (not flat)
  fn, fn_tiles = (lib.snb_conv2d_c32_tc, lib.snb_conv2d_c32_tc_num_tiles) if use2d else (lib.snb_conv_c32_tc, lib.snb_conv_c32_tc_num_tiles)
  if use_ws:
    fn_tiles = lib.snb_conv_c32_ws_num_tiles
  y = out if out is not None else torch.empty(out_shape(g, three_d), device=x.device, dtype=torch.float32)
  if out is not None:
    _req(out, "out")
    if tuple(out.shape) != tuple(out_shape(g, three_d)):
      raise RuntimeError("stereonet_b200: `out` shape mismatch")
  stats = None
  if want_stats:
    nt = fn_tiles(C.byref(g))
    stats = torch.empty((nt, 2, 32), device=x.device, dtype=torch.float32)
  if residual is not None:
    _req(residual, "residual")
    if residual.shape != y.shape:
      raise RuntimeError("stereonet_b200: residual shape mismatch")
  e = ConvEpilogue(_p(bias), _p(scale), _p(shift), _p(residual), _p(stats), 1 if lrelu else 0)
  if three_d and legacy3d:
    passes |= 0x400                      # diagnostics: 3-D flat-tiled kernel with loader warps instead of the TMA kernel
  if use_ws:
    check(lib.snb_conv_c32_ws(_p(x), _p(wimg), _p(y), C.byref(g), C.byref(e), _stream(x)), "snb_conv_c32_ws")
  else:
    check(fn(_p(x), _p(wimg), _p(y), C.byref(g), C.byref(e), passes, _stream(x)), "snb_conv2d_c32_tc" if use2d else "snb_conv_c32_tc")
  _count()
  return y, stats


def conv_c32_ws_f16(x, wimg, g, bias=None, scale=None, shift=None, residual=None, lrelu=False, out=None):
  """Reduced-precision inference variant of conv_c32_tc(fmt="ws") (snb_conv_c32_ws_f16): one fp16 product per tap, same weight
  image and epilogue, no BatchNorm statistics.  Returns y."""
  three_d = x.dim() == 5
  _req(x, "x"); _req(wimg, "wimg")
  y = out if out is not None else torch.empty(out_shape(g, three_d), device=x.device, dtype=torch.float32)
  if out is not None:
    _req(out, "out")
    if tuple(out.shape) != tuple(out_shape(g, three_d)):
      raise RuntimeError("stereonet_b200: `out` shape mismatch")
  if residual is not None:
    _req(residual, "residual")
    if residual.shape != y.shape:
      raise RuntimeError("stereonet_b200: residual shape mismatch")
  e = ConvEpilogue(_p(bias), _p(scale), _p(shift), _p(residual), None, 1 if lrelu else 0)
  check(_cabi.lib().snb_conv_c32_ws_f16(_p(x), _p(wimg), _p(y), C.byref(g), C.byref(e), _stream(x)), "snb_conv_c32_ws_f16")
  _count()
  return y


def phase_split(x):
  """[B,H,W,32] -> [4,B,ceil(H/2),ceil(W/2),32]: phase a*2+b holds x[:, a::2, b::2] (zero padded to the common size)."""
  _req(x, "x", 4)
  B, H, W, _ = x.shape
  out = torch.empty((4, B, (H + 1) // 2, (W + 1) // 2, 32), device=x.device, dtype=torch.float32)
  check(_cabi.lib().snb_phase_split(_p(x), _p(out), B, H, W, _stream(x)), "snb_phase_split")
  _count()
  return out


def phase_merge(ph, H, W):
  """Inverse of phase_split: [4,B,ceil(H/2),ceil(W/2),32] -> [B,H,W,32]."""
  _req(ph, "phases", 5)
  B = ph.shape[1]
  dx = torch.empty((B, H, W, 32), device=ph.device, dtype=torch.float32)
  check(_cabi.lib().snb_phase_merge(_p(ph), _p(dx), B, H, W, _stream(ph)), "snb_phase_merge")
  _count()
  return dx


def conv5x5s2_c3(img, w, bias):
  _req(img, "rgb_img", 4)
  B, Cc, H, W = img.shape
  if Cc != 3:
    raise RuntimeError(f"stereonet_b200: expected a [B,3,H,W] image, got {tuple(img.shape)}")
  OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
  y = torch.empty((B, OH, OW, 32), device=img.device, dtype=torch.float32)
  check(_cabi.lib().snb_conv5x5s2_c3(_p(img), _p(_req(w.detach(), "w")), _p(bias.detach()), _p(y), B, H, W, _stream(img)),
        "snb_conv5x5s2_c3")
  _count()
  return y


def conv5x5s2_c3_phases(img, w, bias):
  """downsample[0] written as the polyphase images [4,B,OH/2,OW/2,32] of its output (OH, OW even)."""
  _req(img, "rgb_img", 4)
  B, Cc, H, W = img.shape
  OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
  y = torch.empty((4, B, OH // 2, OW // 2, 32), device=img.device, dtype=torch.float32)
  check(_cabi.lib().snb_conv5x5s2_c3_phases(_p(img), _p(_req(w.detach(), "w")), _p(bias.detach()), _p(y), B, H, W, _stream(img)),
        "snb_conv5x5s2_c3_phases")
  _count()
  return y


def refine_in_conv(coarse, rgb, w, bias, scale=None, shift=None, lrelu=False, want_stats=False):
  """Fused upsample + scale + concat + Conv2d(4->32).  Returns (up [B,H,W], z [B,H,W,32], stats)."""
  _req(coarse, "coarse_disparity", 3); _req(rgb, "guidance_rgb", 4)
  B, h, w_ = coarse.shape
  H, W = rgb.shape[-2:]
  up = torch.empty((B, H, W), device=rgb.device, dtype=torch.float32)
  z = torch.empty((B, H, W, 32), device=rgb.device, dtype=torch.float32)
  stats = None
  if want_stats:
    nt = _cabi.lib().snb_refine_in_conv_num_tiles(B, H, W)
    stats = torch.empty((nt, 2, 32), device=rgb.device, dtype=torch.float32)
  e = ConvEpilogue(_p(bias), _p(scale), _p(shift), None, _p(stats), 1 if lrelu else 0)
  check(_cabi.lib().snb_refine_in_conv(_p(coarse), _p(rgb), _p(_req(w.detach(), "w")), _p(up), _p(z), B, h, w_, H, W,
                                       float(W) / float(w_), C.byref(e), _stream(rgb)), "snb_refine_in_conv")
  _count()
  return up, z, stats


def refine_in_weights_ws(w):
  """[32,4,3,3] weight of the refinement's input conv -> the walk kernel's image: the [32,32,3,3] tensor
  W'[co, kw*4 + ch, kh, 0] = w[co, ch, kh, kw] in the "ws" format (layout ops + snb_prep_conv_weights_tc)."""
  _req(w, "weight", 4)
  if tuple(w.shape) != (32, 4, 3, 3):
    raise RuntimeError(f"stereonet_b200: expected a [32,4,3,3] weight, got {tuple(w.shape)}")
  wp = torch.zeros((32, 32, 3, 3), device=w.device, dtype=torch.float32)
  wp[:, :12, :, 0] = w.detach().permute(0, 3, 1, 2).reshape(32, 12, 3)          # [co, kw, ch, kh] -> [co, kw*4+ch, kh]
  return prep_conv_weights_tc(wp, 0, fmt="ws")


def refine_in_conv_ws(coarse, rgb, wimg, bias, scale=None, shift=None, lrelu=False, want_stats=False):
  """Fused upsample + scale + concat, then Conv2d(4->32) on the walk kernel.  Returns (up [B,H,W], z [B,H,W,32], stats)."""
  _req(coarse, "coarse_disparity", 3); _req(rgb, "guidance_rgb", 4); _req(wimg, "wimg")
  B, h, w_ = coarse.shape
  H, W = rgb.shape[-2:]
  lib = _cabi.lib()
  up = torch.empty((B, H, W), device=rgb.device, dtype=torch.float32)
  x4 = torch.empty((B, H, W, 4), device=rgb.device, dtype=torch.float32)
  check(lib.snb_refine_pack_input(_p(coarse), _p(rgb), _p(x4), _p(up), B, h, w_, H, W, float(W) / float(w_), _stream(rgb)),
        "snb_refine_pack_input")
  z = torch.empty((B, H, W, 32), device=rgb.device, dtype=torch.float32)
  stats = None
  if want_stats:
    g = geom((B, H, W, 32), 3)
    stats = torch.empty((lib.snb_conv_c32_ws_num_tiles(C.byref(g)), 2, 32), device=rgb.device, dtype=torch.float32)
  e = ConvEpilogue(_p(bias), _p(scale), _p(shift), None, _p(stats), 1 if lrelu else 0)
  check(lib.snb_conv_c4_ws(_p(x4), _p(wimg), _p(z), B, H, W, C.byref(e), _stream(rgb)), "snb_conv_c4_ws")
  _count(2)
  return up, z, stats


def conv_c32_taps(x, w, ntaps):
  """Channel contraction of a 32->1 conv: x [B,(D),H,W,32] -> taps [B,(D),ntaps,H,W]."""
  _req(x, "x")
  H, W = x.shape[-3], x.shape[-2]
  nslices = x.numel() // (32 * H * W)
  taps = torch.empty(tuple(x.shape[:-3]) + (ntaps, H, W), device=x.device, dtype=torch.float32)
  check(_cabi.lib().snb_conv_c32_taps(_p(x), _p(_req(w.detach(), "w")), _p(taps), nslices, H * W, ntaps, _stream(x)),
        "snb_conv_c32_taps")
  _count()
  return taps


def tapsum_softargmin(taps, bias, want_cost):
  B, D, _, H, W = taps.shape
  pred = torch.empty((B, H, W), device=taps.device, dtype=torch.float32)
  cost = torch.empty((B, D, H, W), device=taps.device, dtype=torch.float32) if want_cost else None
  check(_cabi.lib().snb_tapsum_softargmin(_p(taps), _p(bias.detach()), _p(cost), _p(pred), B, D, H, W, _stream(taps)),
        "snb_tapsum_softargmin")
  _count()
  return cost, pred


def conv3d_out_softargmin(x, w, bias, want_cost=True, want_fcs=False):
  """conv3d_alone + softmax + expectation in one kernel (snb_conv3d_out_softargmin).  x [B,D,H,W,32] -> (cost [B,D,H,W] or
  None, pred [B,H,W], fcs [B,H,W] or None)."""
  _req(x, "x", 5)
  B, D, H, W, _ = x.shape
  pred = torch.empty((B, H, W), device=x.device, dtype=torch.float32)
  cost = torch.empty((B, D, H, W), device=x.device, dtype=torch.float32) if want_cost else None
  fcs = torch.empty((B, H, W), device=x.device, dtype=torch.float32) if want_fcs else None
  check(_cabi.lib().snb_conv3d_out_softargmin(_p(x), _p(_req(w.detach(), "w")), _p(bias.detach()), _p(cost), _p(pred), _p(fcs),
                                              B, D, H, W, _stream(x)), "snb_conv3d_out_softargmin")
  _count()
  return cost, pred, fcs


def tapsum_refine_out(taps, bias, up, relu=True):
  B, _, H, W = taps.shape
  out = torch.empty((B, H, W), device=taps.device, dtype=torch.float32)
  check(_cabi.lib().snb_tapsum_refine_out(_p(taps), _p(None if bias is None else bias.detach()), _p(up), _p(out), B, H, W,
                                          1 if relu else 0, _stream(taps)), "snb_tapsum_refine_out")
  _count()
  return out


def upsample_bilinear(x, H, W, mul):
  _req(x, "x", 3)
  B, h, w = x.shape
  out = torch.empty((B, H, W), device=x.device, dtype=torch.float32)
  check(_cabi.lib().snb_upsample_bilinear(_p(x), _p(out), B, h, w, H, W, float(mul), _stream(x)), "snb_upsample_bilinear")
  _count()
  return out


def upsample_bilinear_bwd(dout, h, w, mul):
  _req(dout, "dout", 3)
  B, H, W = dout.shape
  din = torch.empty((B, h, w), device=dout.device, dtype=torch.float32)
  check(_cabi.lib().snb_upsample_bilinear_bwd(_p(dout), _p(din), B, h, w, H, W, float(mul), _stream(dout)),
        "snb_upsample_bilinear_bwd")
  _count()
  return din


def bn_finalize(stats, count, bn, update_running=True):
  """Reduce conv-epilogue partials into per-channel scale/shift (+ mean, invstd); updates bn's running stats in place."""
  dev = stats.device
  out = torch.empty((4, 32), device=dev, dtype=torch.float32)
  rm = bn.running_mean if update_running else None
  rv = bn.running_var if update_running else None
  scratch = torch.empty((64, 64), device=dev, dtype=torch.float64)
  nbt = bn.num_batches_tracked if (update_running and bn.num_batches_tracked is not None) else None   # += 1 in the same launch
  check(_cabi.lib().snb_bn_finalize_ws(_p(stats), stats.shape[0], int(count), _p(bn.weight.detach()), _p(bn.bias.detach()),
                                       _p(rm), _p(rv), _p(nbt), BN_MOMENTUM, BN_EPS, _p(out[0]), _p(out[1]), _p(out[2]), _p(out[3]),
                                       _p(scratch), _stream(stats)), "snb_bn_finalize_ws")
  _count(2 if stats.shape[0] > 256 else 1)
  return out[0], out[1], out[2], out[3]


def bn_running_update(bn, mean, invstd, count):
  """The running-statistics update of a bn_finalize(..., update_running=False) call, applied later (stream-ordered)."""
  check(_cabi.lib().snb_bn_running_update(_p(mean), _p(invstd), int(count), _p(bn.running_mean), _p(bn.running_var),
                                          _p(bn.num_batches_tracked), BN_MOMENTUM, BN_EPS, _stream(mean)), "snb_bn_running_update")
  _count()


def bn_apply(z, scale, shift, residual=None, lrelu=True):
  y = torch.empty_like(z)
  check(_cabi.lib().snb_bn_apply(_p(z), _p(scale), _p(shift), _p(residual), _p(y), z.numel() // 32, 1 if lrelu else 0,
                                 _stream(z)), "snb_bn_apply")
  _count()
  return y


# ------------------------------------------------------------------------------------------------ backward wrappers
def reduce_partials(partial, mul=1.0):
  """[n, len] per-block partials -> [len] (fixed-order double accumulation on the device)."""
  n = partial.shape[0]
  ln = partial.numel() // n
  out = torch.empty((ln,), device=partial.device, dtype=torch.float32)
  check(_cabi.lib().snb_reduce_partials(_p(partial), n, ln, _p(out), float(mul), _stream(partial)), "snb_reduce_partials")
  _count()
  return out


def reduce_wgrad_partials(part, taps, wshape):
  """[n, taps*1024] per-CTA partials -> weight gradient in PyTorch layout `wshape` = [32,32,*k] (one launch)."""
  out = torch.empty(wshape, device=part.device, dtype=torch.float32)
  check(_cabi.lib().snb_reduce_wgrad_partials(_p(part), part.shape[0], taps, _p(out), _stream(part)), "snb_reduce_wgrad_partials")
  _count()
  return out


def bn_lrelu_bwd(z, dy, scale, shift, mean, invstd, train, lrelu=True):
  """Backward of y = LeakyReLU(z*scale + shift) with (train) batch-stat BatchNorm.  Returns dz, dgamma, dbeta, dbias."""
  _req(z, "z"); _req(dy, "dy")
  npos = z.numel() // 32
  nb = _cabi.lib().snb_bwd_num_blocks(npos)
  part = torch.empty((nb, 64), device=z.device, dtype=torch.float32)
  check(_cabi.lib().snb_bn_lrelu_bwd_reduce(_p(z), _p(dy), _p(scale), _p(shift), _p(mean), _p(invstd), _p(part), npos,
                                            1 if lrelu else 0, _stream(z)), "snb_bn_lrelu_bwd_reduce")
  _count()
  sums = reduce_partials(part)
  dz = torch.empty_like(z)
  dzpart = torch.empty((nb, 32), device=z.device, dtype=torch.float32)
  check(_cabi.lib().snb_bn_lrelu_bwd_apply(_p(z), _p(dy), _p(scale), _p(shift), _p(mean), _p(invstd), _p(sums), npos,
                                           1 if train else 0, 1 if lrelu else 0, _p(dz), _p(dzpart), _stream(z)),
        "snb_bn_lrelu_bwd_apply")
  _count()
  return dz, sums[32:], sums[:32], reduce_partials(dzpart)


def channel_sum(x):
  _req(x, "x")
  npos = x.numel() // 32
  nb = _cabi.lib().snb_bwd_num_blocks(npos)
  part = torch.empty((nb, 32), device=x.device, dtype=torch.float32)
  check(_cabi.lib().snb_channel_sum(_p(x), _p(part), npos, _stream(x)), "snb_channel_sum")
  _count()
  return reduce_partials(part)


def conv_c32_wgrad(x, dz, g, wshape):
  """Weight gradient of a 32->32 conv in PyTorch layout `wshape` = [32,32,*k]."""
  _req(x, "x"); _req(dz, "dz")
  n = _cabi.lib().snb_conv_c32_wgrad_num_partials(C.byref(g))
  taps = g.KD * g.KH * g.KW
  part = torch.empty((n, taps * 1024), device=x.device, dtype=torch.float32)
  check(_cabi.lib().snb_conv_c32_wgrad(_p(x), _p(dz), _p(part), C.byref(g), _stream(x)), "snb_conv_c32_wgrad")
  _count()
  return reduce_wgrad_partials(part, taps, wshape)


def conv_c32_wgrad_tc(x, dz, g, wshape, passes=3):
  """Tensor-core weight gradient of a stride-1 'same' 3x3 / 3x3x3 32->32 conv (snb_conv_c32_wgrad_tc)."""
  _req(x, "x"); _req(dz, "dz")
  n = _cabi.lib().snb_conv_c32_wgrad_tc_num_partials(C.byref(g))
  if n <= 0:
    raise RuntimeError("snb_conv_c32_wgrad_tc_num_partials failed: " + _cabi.lib().snb_last_error().decode())
  taps = g.KD * g.KH * g.KW
  part = torch.empty((n, taps * 1024), device=x.device, dtype=torch.float32)
  check(_cabi.lib().snb_conv_c32_wgrad_tc(_p(x), _p(dz), _p(part), C.byref(g), passes, _stream(x)), "snb_conv_c32_wgrad_tc")
  _count()
  return reduce_wgrad_partials(part, taps, wshape)


def conv5x5s2_c3_wgrad(img, dy):
  B, _, H, W = img.shape
  n = _cabi.lib().snb_conv5x5s2_c3_num_tiles(B, H, W)
  part = torch.empty((n, 75 * 32), device=img.device, dtype=torch.float32)
  check(_cabi.lib().snb_conv5x5s2_c3_wgrad(_p(img), _p(_req(dy, "dy")), _p(part), B, H, W, _stream(img)), "snb_conv5x5s2_c3_wgrad")
  _count()
  return reduce_partials(part).view(3, 5, 5, 32).permute(3, 0, 1, 2).contiguous()


def refine_in_wgrad(coarse, rgb, dz):
  B, h, w_ = coarse.shape
  H, W = rgb.shape[-2:]
  n = _cabi.lib().snb_refine_in_conv_num_tiles(B, H, W)
  part = torch.empty((n, 36 * 32), device=rgb.device, dtype=torch.float32)
  check(_cabi.lib().snb_refine_in_wgrad(_p(coarse), _p(rgb), _p(_req(dz, "dz")), _p(part), B, h, w_, H, W, float(W) / float(w_),
                                        _stream(rgb)), "snb_refine_in_wgrad")
  _count()
  return reduce_partials(part).view(4, 3, 3, 32).permute(3, 0, 1, 2).contiguous()


def softargmin_bwd(cost, pred, dpred, dcost_extra=None):
  B, D, H, W = cost.shape
  dcost = torch.empty_like(cost)
  check(_cabi.lib().snb_softargmin_bwd(_p(_req(cost, "cost")), _p(pred), _p(dpred), _p(dcost_extra), _p(dcost), B, D, H, W,
                                       _stream(cost)), "snb_softargmin_bwd")
  _count()
  return dcost


def relu_bwd(out, dout):
  dres = torch.empty_like(out)
  check(_cabi.lib().snb_relu_bwd(_p(_req(out, "out")), _p(_req(dout, "dout")), _p(dres), out.numel(), _stream(out)), "snb_relu_bwd")
  _count()
  return dres


def conv_c32_taps_bwd(x, w, g, ntaps):
  """Backward of the 32->1 conv given g = d(conv output) [B,(D),H,W].  Returns dx, dw [1,32,*k], db [1]."""
  _req(x, "x"); _req(g, "g")
  if x.dim() == 5:
    B, D, H, W, _ = x.shape
  else:
    B, H, W, _ = x.shape
    D = 1
  npos = B * D * H * W
  nblk = (npos + 127) // 128
  part = torch.empty((nblk, ntaps * 32 + 1), device=x.device, dtype=torch.float32)
  dx = torch.empty_like(x)
  check(_cabi.lib().snb_conv_c32_taps_bwd(_p(x), _p(_req(w.detach(), "w")), _p(g), _p(dx), _p(part), B, D, H, W, ntaps, _stream(x)),
        "snb_conv_c32_taps_bwd")
  _count()
  red = reduce_partials(part)
  dw = red[:ntaps * 32].view(ntaps, 32).t().reshape(w.shape).contiguous()
  return dx, dw, red[ntaps * 32:].clone()


def photo_loss(left, right, disp, smooth_w=1e-3):
  """Fused Monodepth photometric loss (adapt.py:78-86): returns (loss [1 + B], dloss[0]/ddisp [B,H,W]); loss[0] is the
  masked mean over the batch, loss[1 + b] the masked mean over sample b alone (OVS validation, adapt.py:122-142)."""
  _req(left, "left_img", 4); _req(right, "right_img", 4); _req(disp, "disp", 3)
  B, Cc, H, W = left.shape
  if Cc != 3 or right.shape != left.shape or tuple(disp.shape) != (B, H, W):
    raise RuntimeError(f"stereonet_b200: photo_loss expects [B,3,H,W] images and a [B,H,W] disparity, got "
                       f"{tuple(left.shape)} {tuple(right.shape)} {tuple(disp.shape)}")
  loss = torch.empty((1 + B,), device=left.device, dtype=torch.float32)
  ddisp = torch.empty((B, H, W), device=left.device, dtype=torch.float32)
  ws = torch.empty((_cabi.lib().snb_photo_loss_workspace_floats(B, H, W),), device=left.device, dtype=torch.float32)
  check(_cabi.lib().snb_photo_loss(_p(left), _p(right), _p(disp), _p(loss), _p(ddisp), _p(ws), B, H, W, float(smooth_w),
                                   _stream(left)), "snb_photo_loss")
  _count(3)
  return loss, ddisp


def khamis_loss(pred, gt):
  """khamis_robust_loss (loss_functions.py:6-15): returns (loss [1], dloss/dpred like pred)."""
  _req(pred, "pred_disp"); _req(gt, "gt_disp")
  if pred.shape != gt.shape:
    raise RuntimeError(f"stereonet_b200: khamis_loss expects equal shapes, got {tuple(pred.shape)} {tuple(gt.shape)}")
  n = pred.numel()
  loss = torch.empty((1,), device=pred.device, dtype=torch.float32)
  dpred = torch.empty_like(pred)
  ws = torch.empty((_cabi.lib().snb_khamis_loss_workspace_floats(n),), device=pred.device, dtype=torch.float32)
  check(_cabi.lib().snb_khamis_loss(_p(pred), _p(gt), _p(loss), _p(dpred), _p(ws), n, _stream(pred)), "snb_khamis_loss")
  _count(2)
  return loss, dpred


def eval_metrics(pred, gt):
  """Per-sample evaluation sums (train.py:98-107): [B,6] = {sum|e|, #valid, #(|e|>2), #(|e|>3), #(|e|>4), #(|e|>5)} over gt > 0."""
  _req(pred, "pred_disp"); _req(gt, "gt_disp")
  if pred.shape != gt.shape:
    raise RuntimeError(f"stereonet_b200: eval_metrics expects equal shapes, got {tuple(pred.shape)} {tuple(gt.shape)}")
  B = pred.shape[0]
  out = torch.empty((B, 6), device=pred.device, dtype=torch.float32)
  check(_cabi.lib().snb_eval_metrics(_p(pred), _p(gt), _p(out), B, pred.numel() // B, _stream(pred)), "snb_eval_metrics")
  _count()
  return out


def feature_contrast(cost):
  """Feature-contrast score map [B,H,W] of a cost volume [B,D,H,W] (feature_contrast.py:12-23)."""
  _req(cost, "cost_volume", 4)
  B, D, H, W = cost.shape
  out = torch.empty((B, H, W), device=cost.device, dtype=torch.float32)
  check(_cabi.lib().snb_feature_contrast(_p(cost), _p(out), B, D, H, W, _stream(cost)), "snb_feature_contrast")
  _count()
  return out
