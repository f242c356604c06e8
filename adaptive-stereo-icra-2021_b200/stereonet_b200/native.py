"""Bridge to the whole-model C-ABI (snb_stereonet_*, include/snb200.h): the parameter list a C or C++ host hands to
snb_stereonet_prepare, and a weights file such a host can read without Python or torch (examples/stereonet_infer.cpp).
Python users keep runtime.StereoEngine; this module adds no inference wrapper.

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
