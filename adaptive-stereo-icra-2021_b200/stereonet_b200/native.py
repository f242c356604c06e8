"""Bridge to the whole-model C-ABI (snb_stereonet_*, include/snb200.h): the parameter list a C or C++ host hands to
snb_stereonet_prepare, and a weights file such a host can read without Python or torch (examples/stereonet_infer.cpp).
Python users keep runtime.StereoEngine; this module adds no inference wrapper.  NativeAdapt drives the adaptation step
(snb_stereonet_adapt_*: single pass, or with an experience-replay pass) on a pair of modules and converts its Adam state to and from
optim.FusedAdamClip.

Parameter order (param_names): the tensors the eval forward reads, in the reference's state_dict order, feature_net first and
stereo_net second; BasicBlock.conv2.* (constructed, never run) and num_batches_tracked are left out.  2k + 108 tensors.

Weights file (export_weights), little-endian:
  8 bytes   magic b"SNBSTW01"
  4 x int32 k, input_scale, maxdisp, n   (n = number of tensors = len(param_names(k)))
  n times   int32 numel, then numel float32 values (the tensor, contiguous, in PyTorch's layout)
"""
import ctypes as C
import struct

import torch

from . import _cabi

MAGIC = b"SNBSTW01"


def _skipped(name):
  return ".conv2." in name or name.endswith("num_batches_tracked")


def _named_tensors(net):
  return [(n, t) for n, t in net.state_dict(keep_vars=True).items() if not _skipped(n)]


def param_names(k):
  """Ordered names ("feature_net.<key>", "stereo_net.<key>") of the tensors snb_stereonet_prepare reads, taken from the modules'
  own registration order (constructed on the meta device: no memory, no kernels)."""
  from .models.stereo_net import FeatureExtractorNetwork, StereoNet
  with torch.device("meta"):
    f, s = FeatureExtractorNetwork(k), StereoNet(k, 1, 0)
  return ["feature_net." + n for n, _ in _named_tensors(f)] + ["stereo_net." + n for n, _ in _named_tensors(s)]


def _tensors(feature_net, stereo_net):
  if feature_net.k != stereo_net.k:
    raise ValueError(f"feature_net.k = {feature_net.k} but stereo_net.k = {stereo_net.k}")
  ts = [t for _, t in _named_tensors(feature_net)] + [t for _, t in _named_tensors(stereo_net)]
  n = _cabi.lib().snb_stereonet_num_params(feature_net.k)
  if len(ts) != n:
    raise RuntimeError(f"stereonet_b200: the modules hold {len(ts)} tensors, the library expects {n}")
  return ts


def param_pointers(feature_net, stereo_net):
  """ctypes array of the device pointers snb_stereonet_prepare takes as `params` (the modules' own storage, no copies)."""
  ts = _tensors(feature_net, stereo_net)
  for name, t in zip(param_names(feature_net.k), ts):
    if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
      raise RuntimeError(f"stereonet_b200: `{name}` must be a contiguous fp32 CUDA tensor")
  return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def export_weights(feature_net, stereo_net, path):
  """Write the parameters in the file format of the module docstring."""
  ts = _tensors(feature_net, stereo_net)
  with open(path, "wb") as fh:
    fh.write(MAGIC)
    fh.write(struct.pack("<4i", feature_net.k, stereo_net.input_scale, stereo_net.maxdisp, len(ts)))
    for t in ts:
      a = t.detach().to("cpu", torch.float32).contiguous().numpy()
      fh.write(struct.pack("<i", a.size))
      fh.write(a.astype("<f4").tobytes())


def bn_counters(feature_net, stereo_net):
  """ctypes array of the 17 num_batches_tracked counters snb_stereonet_adapt_forward increments, in module order."""
  ts = [m.num_batches_tracked for net in (feature_net, stereo_net) for name, m in net.named_modules()
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm) and ".conv2." not in name]
  return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


class NativeAdapt:
  """State, workspace and pointer arrays of the native adaptation step on (feature_net, stereo_net), whose tensors it updates in
  place.  `flat_grad`, `exp_avg`, `exp_avg_sq` and `step` are views of the state, laid out as optim.FusedAdamClip's buffers."""

  def __init__(self, feature_net, stereo_net, lr=5e-5, betas=(0.9, 0.999), eps=1e-8, clip_norm=1.0):
    self.f, self.s, self.k = feature_net, stereo_net, feature_net.k
    self.lr, self.betas, self.eps, self.clip_norm = float(lr), (float(betas[0]), float(betas[1])), float(eps), clip_norm
    lib = _cabi.lib()
    self.params = param_pointers(feature_net, stereo_net)
    self.counters = bn_counters(feature_net, stereo_net)
    dev = next(feature_net.parameters()).device
    self.state = torch.empty((lib.snb_stereonet_adapt_state_bytes(self.k),), device=dev, dtype=torch.uint8)
    views = []
    for what in range(4):
      off, nb = C.c_longlong(), C.c_longlong()
      _cabi.check(lib.snb_stereonet_adapt_state_piece(self.k, what, C.byref(off), C.byref(nb)), "snb_stereonet_adapt_state_piece")
      views.append(self.state[off.value:off.value + nb.value].view(torch.float32))
    self.flat_grad, self.exp_avg, self.exp_avg_sq, self.step_t = views
    self._ws, self._last = {}, None
    _cabi.check(lib.snb_stereonet_adapt_init(self.params, self.k, self.state.data_ptr(), _stream(dev)), "snb_stereonet_adapt_init")

  def workspace(self, B, H, W, RB=0):
    """The workspace of the forward / update pair at this shape (RB >= 1: with a replay pass of batch RB), allocated once."""
    key = (B, H, W, RB)
    if key not in self._ws:
      lib = _cabi.lib()
      if RB:
        nb = lib.snb_stereonet_adapt_replay_workspace_bytes(self.k, self.s.input_scale, self.s.maxdisp, B, H, W, RB)
      else:
        nb = lib.snb_stereonet_adapt_workspace_bytes(self.k, self.s.input_scale, self.s.maxdisp, B, H, W)
      if nb < 0:
        raise RuntimeError(lib.snb_last_error().decode())
      self._ws[key] = torch.empty((nb,), device=self.state.device, dtype=torch.uint8)
    return self._ws[key]

  def _check(self, t, name, shape):
    if not (isinstance(t, torch.Tensor) and t.device == self.state.device and t.dtype == torch.float32 and t.is_contiguous()
            and tuple(t.shape) == tuple(shape)):
      raise RuntimeError(f"stereonet_b200: `{name}` must be a contiguous fp32 tensor of shape {tuple(shape)} on {self.state.device} "
                         f"(got {type(t).__name__} {tuple(getattr(t, 'shape', ()))} {getattr(t, 'dtype', None)} "
                         f"{getattr(t, 'device', None)})")

  def forward(self, images, loss, disp=None, fcs=None, fcs_mean=None, replay=None, loss_replay=None, er_weight=0.05):
    """images [2,B,3,H,W]; writes loss [1 + B] and the optional outputs disp [B,H,W], fcs [B,h,w], fcs_mean [1].
    replay = (replay_images [2,RB,3,H,W], gt [RB,H,W] or [RB,1,H,W]) adds the experience-replay pass: loss_replay [2] receives
    {Khamis term, loss[0] + er_weight * Khamis term}, and update() then differentiates both passes."""
    if not (isinstance(images, torch.Tensor) and images.dim() == 5 and images.shape[0] == 2 and images.shape[2] == 3):
      raise RuntimeError(f"stereonet_b200: `images` must be [2,B,3,H,W], got {tuple(getattr(images, 'shape', ()))}")
    _, B, _, H, W = images.shape
    h, w = H, W
    for _ in range(self.k):
      h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    self._check(images, "images", images.shape)
    self._check(loss, "loss", (1 + B,))
    for t, name, shape in ((disp, "disp", (B, H, W)), (fcs, "fcs", (B, h, w)), (fcs_mean, "fcs_mean", (1,))):
      if t is not None:
        self._check(t, name, shape)
    p = lambda t: None if t is None else t.data_ptr()
    lib, st = _cabi.lib(), _stream(images.device)
    if replay is None:
      _cabi.check(lib.snb_stereonet_adapt_forward(
          self.params, self.counters, self.k, self.s.input_scale, self.s.maxdisp, images.data_ptr(), B, H, W, self.state.data_ptr(),
          self.workspace(B, H, W).data_ptr(), loss.data_ptr(), p(disp), p(fcs), p(fcs_mean), st), "snb_stereonet_adapt_forward")
      self._last = (B, H, W, 0)
      return
    rimages, gt = replay
    if not (isinstance(rimages, torch.Tensor) and rimages.dim() == 5 and rimages.shape[0] == 2 and rimages.shape[1] >= 1
            and tuple(rimages.shape[2:]) == (3, H, W)):
      raise RuntimeError(f"stereonet_b200: `replay_images` must be [2,RB,3,{H},{W}], got {tuple(getattr(rimages, 'shape', ()))}")
    RB = rimages.shape[1]
    self._check(rimages, "replay_images", rimages.shape)
    self._check(gt, "replay_gt", (RB, 1, H, W) if isinstance(gt, torch.Tensor) and gt.dim() == 4 else (RB, H, W))
    self._check(loss_replay, "loss_replay", (2,))
    _cabi.check(lib.snb_stereonet_adapt_forward_replay(
        self.params, self.counters, self.k, self.s.input_scale, self.s.maxdisp, images.data_ptr(), B, H, W, rimages.data_ptr(),
        gt.data_ptr(), RB, float(er_weight), self.state.data_ptr(), self.workspace(B, H, W, RB).data_ptr(), loss.data_ptr(),
        loss_replay.data_ptr(), p(disp), p(fcs), p(fcs_mean), st), "snb_stereonet_adapt_forward_replay")
    self._last = (B, H, W, RB)

  def update(self):
    """Backward of the last forward (both passes after a replay forward), clip + Adam."""
    if self._last is None:
      raise RuntimeError("stereonet_b200: NativeAdapt.update() needs a forward() first")
    B, H, W, RB = self._last
    lib = _cabi.lib()
    common = (self.state.data_ptr(), self.workspace(B, H, W, RB).data_ptr(), float(self.clip_norm) if self.clip_norm else 0.0,
              self.lr, self.betas[0], self.betas[1], self.eps, _stream(self.state.device))
    if RB:
      _cabi.check(lib.snb_stereonet_adapt_update_replay(self.params, self.k, self.s.input_scale, self.s.maxdisp, B, H, W, RB, *common),
                  "snb_stereonet_adapt_update_replay")
    else:
      _cabi.check(lib.snb_stereonet_adapt_update(self.params, self.k, self.s.input_scale, self.s.maxdisp, B, H, W, *common),
                  "snb_stereonet_adapt_update")

  def to_fused(self, opt):
    """Copy the moments and step into an optim.FusedAdamClip of the same modules (same flat layout)."""
    with torch.no_grad():
      opt.exp_avg.copy_(self.exp_avg); opt.exp_avg_sq.copy_(self.exp_avg_sq); opt.step_t.copy_(self.step_t)

  def from_fused(self, opt):
    with torch.no_grad():
      self.exp_avg.copy_(opt.exp_avg); self.exp_avg_sq.copy_(opt.exp_avg_sq); self.step_t.copy_(opt.step_t)


def _stream(dev):
  return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
