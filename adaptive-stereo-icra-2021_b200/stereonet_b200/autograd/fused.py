"""Fused layer entry points used by the nn.Modules: pick the no-grad (inference / validation) kernels or the
autograd.Function wrappers (adaptation step) and keep the derived-tensor caches (repacked weights, folded BN)."""
import torch

from .. import ops

# Derived read-only tensors (repacked weights, folded BN) live ON the owning nn.Module (attribute `_snb_cache`), keyed
# on the in-place version counters of the source parameters, so an optimizer step (adapt.py:393) or load_state_dict
# invalidates them and they die with the module (no process-global state).
# EPOCH covers updates torch's version counters cannot see: a replayed CUDA graph of the adaptation step rewrites the
# parameters in place on the device without touching the Python-side counters (adapt.AdaptStepper bumps it per replay).
EPOCH = 0
# BN_EPOCH does the same for the tensors derived from BatchNorm RUNNING statistics (eval-mode scale / shift): snb_bn_finalize
# updates running_mean / running_var through raw pointers, so their version counters do not move either, and a train-mode
# forward that is NOT followed by an optimizer step (OVS frames whose update is skipped, adapt.py:381-396; no-grad train-mode
# forwards) must still invalidate the folded statistics the next eval-mode forward uses.
BN_EPOCH = 0


def bump_epoch():
  global EPOCH, BN_EPOCH
  EPOCH += 1
  BN_EPOCH += 1


def bump_bn_epoch():
  global BN_EPOCH
  BN_EPOCH += 1


def state_epoch():
  """Changes whenever parameters or BN running statistics may have changed behind torch's version counters."""
  return (EPOCH, BN_EPOCH)


# A torch.cuda.Stream installed here (adapt.AdaptStepper does, around its forward) moves the weight gradients of the conv + BN +
# LeakyReLU layers onto that stream: see functions.WgradToken.
WGRAD_STREAM = None
_TOKEN = {}


def wgrad_token(shape, device):
  """Zero-stride token of `shape` over one persistent float (never written): no allocation, so it can be handed out under a
  stream that is not (yet) part of an ongoing graph capture.  AdaptStepper creates the buffer in its eager warm-up step."""
  buf = _TOKEN.get(device)
  if buf is None:
    buf = _TOKEN[device] = torch.zeros((1,), device=device, dtype=torch.float32)
  return buf.as_strided(tuple(shape), (0,) * len(shape))

# While a list is installed here, train-mode BatchNorm calls do not touch the running statistics; they append
# (bn, mean, invstd, count) instead and flush_deferred_bn() applies the updates later, in call order.  adapt.AdaptStepper uses
# it for the feature pass it runs on a second stream (the left and right passes update the SAME buffers, in that order).
DEFER_BN = None


def bn_finalize(stats, count, bn):
  """Train-mode BatchNorm statistics (ops.bn_finalize) + invalidation of what was derived from the running statistics."""
  if DEFER_BN is not None and bn.running_mean is not None:
    out = ops.bn_finalize(stats, count, bn, update_running=False)
    DEFER_BN.append((bn, out[2], out[3], count))
    return out
  out = ops.bn_finalize(stats, count, bn)
  bump_bn_epoch()
  return out


def flush_deferred_bn(pending):
  for bn, mean, invstd, count in pending:
    ops.bn_running_update(bn, mean, invstd, count)
  if pending:
    bump_bn_epoch()
  del pending[:]


# Fused optimizers (torch.optim.Adam(fused=True), torch._fused_adam_) update parameters in place WITHOUT bumping their
# version counters, so every optimizer step also advances the epoch (global post-step hook; costs one integer add).
def _after_optimizer_step(optimizer, args, kwargs):
  bump_epoch()


try:
  from torch.optim.optimizer import register_optimizer_step_post_hook as _register_step_hook
  _register_step_hook(_after_optimizer_step)
except Exception as exc:  # pragma: no cover
  raise RuntimeError("stereonet_b200 needs torch.optim.optimizer.register_optimizer_step_post_hook "
                     "(PyTorch >= 2.1) to keep its derived-weight caches coherent") from exc


def _cached(owner, key, tensors, make, epoch=None):
  cache = owner.__dict__.setdefault("_snb_cache", {})
  ver = (EPOCH if epoch is None else epoch,) + tuple((t.data_ptr(), t._version) for t in tensors)
  hit = cache.get(key)
  if hit is not None and hit[0] == ver:
    return hit[1]
  val = make()
  cache[key] = (ver, val)
  return val


def clear_cache(module):
  for m in module.modules():
    m.__dict__.pop("_snb_cache", None)


import os

# Kernel / operand format of the stride-1 3x3 / 3x3x3 32->32 tensor-core layers.  "ws" (the product path): snb_conv_c32_ws,
# error-compensated fp16 split (tcgen05 kind::f16, fp32-grade results).  The other values exist for the parity tests and A/B
# measurements only (set with set_conv_backend, never from the environment): "h3" = the fp16 split on the round-1 kernels,
# "tc3" = 3xTF32 split, "tc1" = single-pass TF32 (~1e-3 relative), "ffma" = fp32 CUDA-core kernel.
CONV_BACKEND = "ws"
_FMT = {"ws": "ws", "h3": "h", "tc3": 3, "tc1": 1}
# 3-D layers under the "ws" back end: the 3-D variant of snb_conv_c32_ws (all 27 tap images resident, every raw row brought on
# chip once per three disparity taps and split to fp16 ONCE, in place).  38 us per KITTI filter layer inside a graph against 50 us
# for the TMA kernel of conv3d_c32_tma.cu ("h": the same operand format, weights streamed per window), which stays as the cross-check.
WS_3D_FMT = "ws"


# Reduced-precision inference (runtime.StereoEngine(..., precision="fp16")): the kinds of 32->32 walk-kernel layer, "2d" (3x3, dilated)
# and "3d" (3x3x3), that run on the single-product variant snb_conv_c32_ws_f16 instead of the fp32-grade split.  Empty (the default)
# everywhere but inside the engine's own no-grad eval forward, which sets it to F16_SHIPPED and resets it, as AdaptStepper does with
# DEFER_BN / WGRAD_STREAM.  The nn.Module forward, the grad-enabled paths and AdaptStepper never see it set; a layer that finds it set
# while grad is enabled raises.  F16_SHIPPED is the layer set of snb_stereonet_forward_f16 (csrc/model.cu F16_LAYERS).
F16_LAYERS = frozenset()
F16_SHIPPED = frozenset(("2d", "3d"))


def _f16_guard():
  if F16_LAYERS and torch.is_grad_enabled():
    raise RuntimeError("stereonet_b200: the fp16 inference forward runs under torch.no_grad() only "
                       "(training and the adaptation step stay on the fp32-grade kernels)")


def _fmt(three_d):
  f = _FMT[CONV_BACKEND]
  return WS_3D_FMT if (f == "ws" and three_d) else f


def set_conv_backend(name):
  global CONV_BACKEND
  if name not in ("ws", "h3", "tc3", "tc1", "ffma"):
    raise ValueError(name)
  CONV_BACKEND = name
  bump_epoch()                 # cached weight images are in the previous backend's format


def _tc_kw(three_d=False):
  return dict(fmt=_fmt(three_d))


def wprep_tc(conv, mode=0):
  fmt = _fmt(conv.weight.dim() == 5)
  return _cached(conv, ("wtc", mode, fmt), [conv.weight], lambda: ops.prep_conv_weights_tc(conv.weight, mode, fmt=fmt))


def conv3x3_c32(x, conv, g, **kw):
  """Backend dispatch for the 'same' 3x3(x3) convolution + fused epilogue."""
  if F16_LAYERS and ("3d" if x.dim() == 5 else "2d") in F16_LAYERS:
    _f16_guard()
    if CONV_BACKEND != "ws" or kw.pop("want_stats", False):
      raise RuntimeError("stereonet_b200: the fp16 inference forward needs the 'ws' back end and eval-mode BatchNorm")
    return ops.conv_c32_ws_f16(x, wprep_tc(conv), g, **kw), None
  if CONV_BACKEND == "ffma":
    return ops.conv_c32(x, wprep(conv), g, **kw)
  return ops.conv_c32_tc(x, wprep_tc(conv), g, **_tc_kw(x.dim() == 5), **kw)


def wprep(conv, mode=0):
  return _cached(conv, ("w", mode), [conv.weight], lambda: ops.prep_conv_weights(conv.weight, mode))


def bn_fold(bn):
  """Eval-mode BatchNorm as per-channel scale/shift (running statistics, eps 1e-5)."""
  def make():
    with torch.no_grad():
      scale = bn.weight * torch.rsqrt(bn.running_var + ops.BN_EPS)
      shift = bn.bias - bn.running_mean * scale
      return scale.contiguous(), shift.contiguous()
  return _cached(bn, "fold", [bn.weight, bn.bias, bn.running_mean, bn.running_var], make, epoch=(EPOCH, BN_EPOCH))


def bn_invstd(bn):
  def make():
    with torch.no_grad():
      return torch.rsqrt(bn.running_var + ops.BN_EPS).contiguous()
  return _cached(bn, "invstd", [bn.running_var], make, epoch=(EPOCH, BN_EPOCH))


def conv3x3_c32_dgrad(dy, conv, g, residual=None):
  """Data gradient of a stride-1 'same' 3x3(x3) conv: the same convolution kernels with flipped/transposed weights."""
  if CONV_BACKEND == "ffma":
    return ops.conv_c32(dy, wprep(conv, 1), g, residual=residual)
  return ops.conv_c32_tc(dy, wprep_tc(conv, 1), g, residual=residual, **_tc_kw(dy.dim() == 5))


def conv3x3_c32_wgrad(x, dz, g, wshape):
  """Weight gradient of a stride-1 'same' 3x3(x3) conv: tensor-core kernel unless the FFMA backend is selected."""
  if CONV_BACKEND == "ffma":
    return ops.conv_c32_wgrad(x, dz, g, wshape)
  return ops.conv_c32_wgrad_tc(x, dz, g, wshape, passes=1 if CONV_BACKEND == "tc1" else 3)


def _needs_grad(*tensors_or_modules):
  if not torch.is_grad_enabled():
    return False
  for t in tensors_or_modules:
    if isinstance(t, torch.Tensor):
      if t.requires_grad:
        return True
    elif t is not None:
      if any(p.requires_grad for p in t.parameters()):
        return True
  return False


def _no_backward():
  raise NotImplementedError("stereonet_b200: backward kernels are not wired for this op yet; "
                            "run under torch.no_grad() (there is no eager fallback)")


# ------------------------------------------------------------------------------------------------ feature extractor
def conv5x5s2_first(img, conv):
  if _needs_grad(conv):
    from . import functions
    return functions.Conv5x5s2First.apply(img, conv.weight, conv.bias)
  return ops.conv5x5s2_c3(img, conv.weight, conv.bias)


def wprep_tc_phases(conv, mode):
  """Tensor-core weight images of the four polyphase 3x3 sub-kernels of a 5x5 stride-2 conv (csrc/phase.cu)."""
  fmt = _fmt(False)

  def make():
    w = conv.weight.detach()
    imgs = []
    for a in (0, 1):
      for b in (0, 1):
        sub = w[:, :, a::2, b::2]                                  # [32,32,3|2,3|2]  (layout ops only)
        sub = torch.nn.functional.pad(sub, (0, 3 - sub.shape[3], 0, 3 - sub.shape[2])).contiguous()
        imgs.append(ops.prep_conv_weights_tc(sub, mode, fmt=fmt))
    return imgs
  return _cached(conv, ("wtc_phase", mode, fmt), [conv.weight], make)


def wprep_p4(conv):
  """The ten-image set of a 5x5 stride-2 layer for the one-launch kernel (ops.conv5x5s2_c32_ws)."""
  return _cached(conv, ("wtc_p4", 0, "ws"), [conv.weight], lambda: ops.prep_conv5x5s2_weights_ws(conv.weight.detach().contiguous()))


class WeightPrepBatch:
  """Every tensor-core weight image the adaptation step needs (forward and data-gradient images of all used 3x3 / 3x3x3
  32->32 convolutions, the polyphase images of the 5x5 stride-2 ones) refreshed by ONE launch after an optimizer update,
  instead of ~50 prep launches plus ~50 torch slicing / padding kernels per step.  The images live in one persistent
  buffer; refresh() re-validates the per-module caches (`_cached`) so the layers find them as hits."""

  def __init__(self, nets, modes=(0, 1)):
    self.items = []                      # (conv, cache key, views, source pointer)
    self.backend = (CONV_BACKEND, WS_3D_FMT)
    rows = []
    plan = []
    for net in nets:
      for name, m in net.named_modules():
        if not isinstance(m, (torch.nn.Conv2d, torch.nn.Conv3d)) or ".conv2" in name or name.startswith("conv2"):
          continue                       # BasicBlock.conv2 is constructed but never used (stereo_net.py:40,44-51)
        w = m.weight
        if tuple(w.shape[:2]) != (32, 32):
          continue
        fmt = _fmt(w.dim() == 5)
        fbit = ops._fmt_of(fmt)[0]
        if tuple(w.shape[2:]) in ((3, 3), (3, 3, 3)) and m.stride[0] == 1:
          kd = 3 if w.dim() == 5 else 1
          for mode in modes:
            plan.append((m, ("wtc", mode, fmt), [(kd * 3, mode | fbit, 0, 0, 0)]))
        elif tuple(w.shape[2:]) == (5, 5) and m.stride[0] == 2:
          for mode in modes:
            if mode == 0 and fmt == "ws":          # forward: the one-launch kernel's image set
              plan.append((m, ("wtc_p4", 0, "ws"), [(10, fbit, 2, 0, 0)]))
            else:
              plan.append((m, ("wtc_phase", mode, fmt), [(3, mode | fbit, 1, a, b) for a in (0, 1) for b in (0, 1)]))
    size = lambda nwin, key: ops.conv_weights_tc_floats(5 if nwin == 10 else nwin // 3, key[2])
    total = sum(size(cfg[0], key) for _, key, cfgs in plan for cfg in cfgs)
    dev = plan[0][0].weight.device
    self.buf = torch.empty((total,), device=dev, dtype=torch.float32)
    off = 0
    for m, key, cfgs in plan:
      views = []
      for nwin, mode, kind, a, b in cfgs:
        v = self.buf[off:off + size(nwin, key)]
        off += size(nwin, key)
        views.append(v)
        rows.append([m.weight.data_ptr(), v.data_ptr(), nwin | (mode << 8) | (kind << 16) | (a << 24) | (b << 28), 0])
      self.items.append((m, key, views, m.weight.data_ptr()))
    self.table = torch.tensor(rows, dtype=torch.int64).to(dev)
    self.n = len(rows)

  def valid(self):
    return self.backend == (CONV_BACKEND, WS_3D_FMT) and all(m.weight.data_ptr() == ptr and m.weight.is_contiguous() for m, _, _, ptr in self.items)

  def refresh(self):
    ops.prep_conv_weights_tc_batch(self.table, self.n)
    for m, key, views, _ in self.items:
      ver = (EPOCH, (m.weight.data_ptr(), m.weight._version))
      m.__dict__.setdefault("_snb_cache", {})[key] = (ver, views if key[0] == "wtc_phase" else views[0])


def conv5x5s2_c32(x, conv, bias, phases=None):
  """5x5 stride-2 pad-2 32->32 convolution: FFMA kernel, or four chained tensor-core 3x3 convs over the phase images
  (`phases`: the input already in polyphase form)."""
  if CONV_BACKEND == "ffma":
    g = ops.geom(x.shape, 5, stride=2, dil=1, pad=2)
    y, _ = ops.conv_c32(x, wprep(conv), g, bias=bias)
    return y
  if CONV_BACKEND == "ws" and phases is None and x.shape[1] >= 2 and x.shape[2] >= 2:
    return ops.conv5x5s2_c32_ws_x(x, wprep_p4(conv), bias=bias)          # polyphase images = strided TMA views of x: no split pass
  ph = phases if phases is not None else ops.phase_split(x)
  if CONV_BACKEND == "ws":
    return ops.conv5x5s2_c32_ws(ph, wprep_p4(conv), bias=bias)
  g3 = ops.geom(ph[0].shape, 3, stride=1, dil=1)
  y = None
  for i, wimg in enumerate(wprep_tc_phases(conv, 0)):
    y, _ = ops.conv_c32_tc(ph[i], wimg, g3, bias=bias if i == 0 else None, residual=y, **_tc_kw())
  return y


def conv5x5s2_c32_dgrad(dy, conv, H, W):
  """Data gradient of the above: dx[2i+a][2j+b] = conv3x3_same(dy, flipped/transposed W_ab)[i][j]."""
  if CONV_BACKEND == "ffma":
    g = ops.geom((dy.shape[0], H, W, 32), 5, stride=2, dil=1, pad=2)
    dx, _ = ops.conv_c32(dy, wprep(conv, 2), ops.geom_transposed(g))
    return dx
  g3 = ops.geom(dy.shape, 3, stride=1, dil=1)
  ph = torch.empty((4,) + tuple(dy.shape), device=dy.device, dtype=torch.float32)
  for i, wimg in enumerate(wprep_tc_phases(conv, 1)):
    ops.conv_c32_tc(dy, wimg, g3, out=ph[i], **_tc_kw())
  return ops.phase_merge(ph, H, W)


def downsample_pair(img, conv0, conv1):
  """downsample[0] (3->32) followed by downsample[1] (32->32), both 5x5 stride 2.  Inference with even intermediate size:
  the first layer writes the polyphase images the second one consumes (no separate split pass)."""
  H, W = img.shape[-2:]
  OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
  if CONV_BACKEND != "ffma" and not _needs_grad(conv0, conv1) and OH % 2 == 0 and OW % 2 == 0:
    ph = ops.conv5x5s2_c3_phases(img, conv0.weight, conv0.bias)
    return conv5x5s2_c32(None, conv1, conv1.bias.detach(), phases=ph)
  return conv_plain(conv5x5s2_first(img, conv0), conv1, ksize=5, stride=2)


def conv_plain(x, conv, ksize, stride):
  """Conv2d 32->32 with bias only (downsample[1:], conv_alone)."""
  g = ops.geom(x.shape, ksize, stride=stride, dil=1, pad=ksize // 2)
  _f16_guard()
  if _needs_grad(x, conv):
    from . import functions
    return functions.conv_c32_autograd(x, conv, ksize, stride)
  if ksize == 3 and stride == 1:
    y, _ = conv3x3_c32(x, conv, g, bias=conv.bias.detach())
  elif ksize == 5 and stride == 2:
    y = conv5x5s2_c32(x, conv, conv.bias.detach())
  else:
    y, _ = ops.conv_c32(x, wprep(conv), g, bias=conv.bias.detach())
  return y


# ------------------------------------------------------------------------------------------------ conv + BN + LeakyReLU
def conv_bn_lrelu(x, conv, bn, dil, residual, training):
  """[x +] LeakyReLU(BN(conv(x))) for 3x3 (2-D, dilated) and 3x3x3 convs (stereo_net.py:8-18,21-30,44-51,155-160)."""
  g = ops.geom(x.shape, 3, stride=1, dil=dil)
  _f16_guard()
  if _needs_grad(x, conv, bn):
    from . import functions
    return functions.conv_bn_lrelu_autograd(x, conv, bn, dil, residual, training)
  if not training:
    scale, shift = bn_fold(bn)
    y, _ = conv3x3_c32(x, conv, g, bias=conv.bias.detach(), scale=scale, shift=shift,
                       residual=x if residual else None, lrelu=True)
    return y
  z, stats = conv3x3_c32(x, conv, g, bias=conv.bias.detach(), want_stats=True)
  scale, shift, _, _ = bn_finalize(stats, z.numel() // 32, bn)
  return ops.bn_apply(z, scale, shift, residual=x if residual else None, lrelu=True)


# ------------------------------------------------------------------------------------------------ stereo head
def cost_volume(left, right, D):
  if _needs_grad(left, right):
    from . import functions
    return functions.CostVolume.apply(left, right, D)
  return ops.cost_volume(left, right, D)


def conv3d_out_softargmin(x, conv, want_cost):
  """conv3d_alone + softmax + DisparityRegression (stereo_net.py:187-198).  Training path: one kernel; when the cost volume is
  requested its feature-contrast map comes out of the same epilogue and rides along as `cost._snb_fcs`
  (losses.feature_contrast_mean)."""
  if _needs_grad(x, conv):
    from . import functions
    return functions.conv3d_out_softargmin_autograd(x, conv, want_cost)
  # Inference: the tensor-core tap contraction + gather / soft-argmin pair (head.cu) — 13 us per KITTI frame faster inside the
  # forward than the one-kernel CUDA-core form (head_fused.cu), which the training path uses (it also emits the FCS map).
  taps = ops.conv_c32_taps(x, conv.weight, 27)
  return ops.tapsum_softargmin(taps, conv.bias, want_cost)


def upsample(pred, H, W, mul):
  if _needs_grad(pred):
    from . import functions
    return functions.Upsample.apply(pred, H, W, mul)
  return ops.upsample_bilinear(pred, H, W, mul)


# ------------------------------------------------------------------------------------------------ refinement
def refine_head(coarse, rgb, conv, bn, training):
  if _needs_grad(coarse, conv, bn):
    from . import functions
    return functions.refine_head_autograd(coarse, rgb, conv, bn, training)
  if not training:
    scale, shift = bn_fold(bn)
    if CONV_BACKEND == "ws":
      # the walk kernel over the packed four-channel image: 30 against 39 us per KITTI frame for the im2col tensor-core kernel
      wimg = _cached(conv, ("wtc_c4", 0, "ws"), [conv.weight], lambda: ops.refine_in_weights_ws(conv.weight))
      up, x, _ = ops.refine_in_conv_ws(coarse, rgb, wimg, conv.bias.detach(), scale=scale, shift=shift, lrelu=True)
      return up, x
    up, x, _ = ops.refine_in_conv(coarse, rgb, conv.weight, conv.bias.detach(), scale=scale, shift=shift, lrelu=True)
    return up, x
  up, z, stats = ops.refine_in_conv(coarse, rgb, conv.weight, conv.bias.detach(), want_stats=True)
  scale, shift, _, _ = bn_finalize(stats, z.numel() // 32, bn)
  return up, ops.bn_apply(z, scale, shift, residual=None, lrelu=True)


def refine_tail(x, conv, up):
  if _needs_grad(x, conv, up):
    from . import functions
    return functions.refine_tail_autograd(x, conv, up)
  taps = ops.conv_c32_taps(x, conv.weight, 9)
  return ops.tapsum_refine_out(taps, conv.bias, up)
