"""The whole-model C-ABI (snb_stereonet_*, csrc/model.cu) against the Python eval path it restates: parameter order (CPU), the
prepared weights, bit-identical outputs over the golden configurations and KITTI sizes, CUDA-graph capture, concurrent calls,
re-preparation, guard bands around every buffer, argument errors, and the torch-free example host."""
import ctypes as C
import json
import os
import subprocess
import threading

import numpy as np
import pytest
import torch

import stereonet_oracle as O
import stereonet_b200 as S
from stereonet_b200 import _cabi, native
from stereonet_b200.losses import feature_contrast_mean
from stereonet_b200.runtime import StereoEngine
from test_oracle_golden import BIG_CASES, CASES, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
SENT = -12345.5
BAND = 1 << 16                    # floats: 256 KB, keeps 256-byte alignment of what sits between the bands

KITTI = {
  "kitti_376x1248_b1": dict(B=1, H=376, W=1248, k=3, s=0),
  "kitti_376x1248_b2": dict(B=2, H=376, W=1248, k=3, s=0),
  "kitti_375x1242_b1": dict(B=1, H=375, W=1242, k=3, s=0),    # odd intermediate width (strided-view branch), 1242 != 156 * 8
}


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("k", [3, 4])
def test_param_names_follow_state_dict_order(k):
  layout = json.load(open(os.path.join(ROOT, "tests", "golden", "state_layout.json")))
  keep = lambda n: ".conv2." not in n and not n.endswith("num_batches_tracked")
  expected = ([f"feature_net.{e[0]}" for e in layout[f"k{k}/feature_net"]["state_dict"] if keep(e[0])]
              + [f"stereo_net.{e[0]}" for e in layout[f"k{k}/stereo_net"]["state_dict"] if keep(e[0])])
  assert native.param_names(k) == expected
  assert _cabi.lib().snb_stereonet_num_params(k) == len(expected) == 2 * k + 108


def test_weights_pieces_are_aligned_and_disjoint():
  lib = _cabi.lib()
  for k in (1, 3, 4):
    total, end = lib.snb_stereonet_weights_bytes(k), 0
    for i in range(lib.snb_stereonet_num_params(k)):
      off, nb = C.c_longlong(), C.c_longlong()
      assert lib.snb_stereonet_weights_piece(k, i, C.byref(off), C.byref(nb)) == 0
      if nb.value:
        assert off.value % 256 == 0 and off.value >= end
        end = off.value + nb.value
    assert end <= total


# ---------------------------------------------------------------------------------------------------------------- helpers
def make_nets(k, s, fsd, ssd):
  f = S.FeatureExtractorNetwork(k).to(DEV)
  n = S.StereoNet(k, 1, s, maxdisp=192).to(DEV)
  f.load_state_dict(fsd, strict=True)
  n.load_state_dict(ssd, strict=True)
  f.eval(); n.eval()
  return f, n


def dims(f, n, B, H, W):
  h, w = H, W
  for _ in range(f.k):
    h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1
  return (n.maxdisp + 1) // 2 ** (n.input_scale + f.k), h, w


def stream_ptr(stream=None):
  return C.c_void_p((stream or torch.cuda.current_stream()).cuda_stream)


def banded(nfloats):
  buf = torch.full((nfloats + 2 * BAND,), SENT, device=DEV, dtype=torch.float32)
  return buf, buf[BAND:BAND + nfloats]


def intact(buf, n):
  return bool((buf[:BAND] == SENT).all().item()) and bool((buf[BAND + n:] == SENT).all().item())


class Native:
  """Prepared weights of one (feature_net, stereo_net) pair and the forward call, through ctypes."""

  def __init__(self, f, n):
    self.f, self.n, self.k = f, n, f.k
    lib = _cabi.lib()
    self.weights = torch.empty((lib.snb_stereonet_weights_bytes(self.k),), device=DEV, dtype=torch.uint8)
    self.prepare()

  def prepare(self):
    _cabi.check(_cabi.lib().snb_stereonet_prepare(native.param_pointers(self.f, self.n), self.k, self.weights.data_ptr(),
                                                   stream_ptr()), "snb_stereonet_prepare")

  def workspace_bytes(self, B, H, W):
    nb = _cabi.lib().snb_stereonet_workspace_bytes(self.k, self.n.input_scale, self.n.maxdisp, B, H, W)
    assert nb > 0, _cabi.lib().snb_last_error()
    return nb

  def call(self, images, ws, disp, coarse=None, cost=None, fcs=None, stream=None):
    B, H, W = images.shape[1], images.shape[-2], images.shape[-1]
    p = lambda t: None if t is None else t.data_ptr()
    return _cabi.lib().snb_stereonet_forward(self.weights.data_ptr(), self.k, self.n.input_scale, self.n.maxdisp, p(images), B, H, W,
                                             p(ws), p(disp), p(coarse), p(cost), p(fcs), stream_ptr(stream))

  def forward(self, images, stream=None):
    """images [2,B,3,H,W] -> dict of fresh output tensors."""
    B, H, W = images.shape[1], images.shape[-2], images.shape[-1]
    D, h, w = dims(self.f, self.n, B, H, W)
    ws = torch.empty((self.workspace_bytes(B, H, W),), device=DEV, dtype=torch.uint8)
    o = dict(disp=torch.empty((B, H, W), device=DEV), coarse=torch.empty((B, H, W), device=DEV),
             cost=torch.empty((B, D, h, w), device=DEV), fcs=torch.empty((B, h, w), device=DEV))
    _cabi.check(self.call(images, ws, **o, stream=stream), "snb_stereonet_forward")
    return o


def python_path(f, n, left, right):
  """StereoEngine's graph-replayed eval forward (what a Python user runs) and the feature-contrast map of its cost volume."""
  eng = StereoEngine(f, n, output_cost_volume=True)
  out = eng(left, right)
  s, k = n.input_scale, f.k
  cost = out[f"cost_volume_l/{s + k}"]
  return dict(disp=out[f"pred_disp_l/{s}"][:, 0].clone(), coarse=out[f"pred_disp_l/{s + k}"][:, 0].clone(), cost=cost.clone(),
              fcs=feature_contrast_mean(cost).clone())


def golden_setup(cfg):
  fsd, ssd, left, right, _ = build(dict(cfg, sharpen=cfg.get("sharpen", 40.0)))
  f, n = make_nets(cfg["k"], cfg["s"], fsd, ssd)
  return f, n, left.to(DEV), right.to(DEV)


def random_setup(cfg, seed=5):
  fsd, ssd = O.make_feature_state(cfg["k"], 11), O.make_stereo_state(22, sharpen=40.0)
  f, n = make_nets(cfg["k"], cfg["s"], fsd, ssd)
  g = torch.Generator(device=DEV).manual_seed(seed)
  pair = torch.rand((2, cfg["B"], 3, cfg["H"], cfg["W"]), device=DEV, generator=g)
  return f, n, pair[0].contiguous(), pair[1].contiguous()


ALL = {**{k: dict(v) for k, v in CASES.items()}, **{k: dict(v) for k, v in BIG_CASES.items()}, **KITTI}


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("k", [3, 4])
def test_prepare_matches_python_caches(k):
  """Folded BN bit-identical to fused.bn_fold; every weight image bit-identical to what the Python path caches on the modules."""
  f, n, left, right = golden_setup(dict(k=k, s=0, B=1, H=64, W=256))
  nat = Native(f, n)
  with torch.no_grad():
    f.eval(); n.eval()
    n(left, f(left), f(right), "l")                  # fills the modules' _snb_cache
  torch.cuda.synchronize()
  wf = nat.weights.view(torch.float32)
  mods = dict(f.named_modules(prefix="feature_net")); mods.update(n.named_modules(prefix="stereo_net"))
  lib = _cabi.lib()
  seen = {"fold": 0, "image": 0, "raw": 0}
  for i, name in enumerate(native.param_names(k)):
    off, nb = C.c_longlong(), C.c_longlong()
    assert lib.snb_stereonet_weights_piece(k, i, C.byref(off), C.byref(nb)) == 0
    piece = wf[off.value // 4:(off.value + nb.value) // 4]
    mname, leaf = name.rsplit(".", 1)
    m = mods[mname]
    if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
      if leaf in ("weight", "bias"):
        scale, shift = m._snb_cache["fold"][1]
        assert torch.equal(piece, scale if leaf == "weight" else shift), name
        seen["fold"] += 1
      else:
        assert nb.value == 0
      continue
    cache = getattr(m, "_snb_cache", {})
    key = next((kk for kk in (("wtc", 0, "ws"), ("wtc_p4", 0, "ws"), ("wtc_c4", 0, "ws")) if kk in cache), None)
    if leaf == "weight" and key is not None:
      img = cache[key][1]
      assert piece.numel() == img.numel(), name
      # the 3-D and P4 sets end with their scale slot and three floats that are never written
      ncmp = img.numel() - 3 if img.numel() % 8 == 4 else img.numel()
      assert torch.equal(piece[:ncmp], img[:ncmp]), name
      seen["image"] += 1
    else:
      src = dict(m.named_parameters(recurse=False))[leaf].detach().flatten()
      assert torch.equal(piece, src), name
      seen["raw"] += 1
  assert seen["fold"] == 2 * 17 and seen["image"] == 18 + (k - 1)     # 17 "ws" images + the C4 image + the P4 sets


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ALL))
def test_forward_bit_identical_to_python_path(name):
  cfg = ALL[name]
  f, n, left, right = (random_setup if name in KITTI else golden_setup)(cfg)
  ref = python_path(f, n, left, right)
  got = Native(f, n).forward(torch.stack([left, right]).contiguous())
  torch.cuda.synchronize()
  for key in ("disp", "coarse", "cost", "fcs"):
    assert torch.equal(got[key], ref[key]), (name, key, (got[key] - ref[key]).abs().max().item())


@pytest.mark.gpu
def test_graph_capture_threads_and_reprepare():
  cfg = KITTI["kitti_375x1242_b1"]
  f, n, left, right = random_setup(cfg)
  images = torch.stack([left, right]).contiguous()
  nat = Native(f, n)
  eager = nat.forward(images)
  torch.cuda.synchronize()

  # captured into a CUDA graph and replayed
  B, H, W = cfg["B"], cfg["H"], cfg["W"]
  ws = torch.empty((nat.workspace_bytes(B, H, W),), device=DEV, dtype=torch.uint8)
  outs = {k_: torch.empty_like(v) for k_, v in eager.items()}
  g = torch.cuda.CUDAGraph()
  with torch.cuda.graph(g):
    assert nat.call(images, ws, **outs) == 0
  for _ in range(2):
    g.replay()
  torch.cuda.synchronize()
  for key in eager:
    assert torch.equal(outs[key], eager[key]), key

  # two host threads, two streams, separate workspaces and outputs
  streams = [torch.cuda.Stream(device=DEV) for _ in range(2)]
  wss = [torch.empty_like(ws) for _ in range(2)]
  res = [{k_: torch.empty_like(v) for k_, v in eager.items()} for _ in range(2)]
  rcs = [None, None]
  for s_ in streams:
    s_.wait_stream(torch.cuda.current_stream())

  def run(i):
    rc = 0
    for _ in range(3):
      rc |= nat.call(images, wss[i], **res[i], stream=streams[i])
    rcs[i] = rc
  th = [threading.Thread(target=run, args=(i,)) for i in range(2)]
  for t in th:
    t.start()
  for t in th:
    t.join()
  torch.cuda.synchronize()
  assert rcs == [0, 0]
  for r in res:
    for key in eager:
      assert torch.equal(r[key], eager[key]), key

  # a parameter and a running statistic change, prepare again: the output follows the Python path with the new values
  with torch.no_grad():
    f.residual_blocks[2].conv1[0][0].weight.mul_(1.25)
    n.filter[1][0][1].running_var.mul_(0.5)
    n.edge_aware_refinements[0].conv2d_out.bias.add_(0.5)
  nat.prepare()
  got = nat.forward(images)
  ref = python_path(f, n, left, right)
  torch.cuda.synchronize()
  for key in ("disp", "coarse", "cost", "fcs"):
    assert torch.equal(got[key], ref[key]), key
  assert not torch.equal(got["disp"], eager["disp"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["k3_ragged", "kitti_375x1242_b1", "k4_sharp"])
def test_writes_stay_inside_buffers(name):
  cfg = ALL[name]
  f, n, left, right = (random_setup if name in KITTI else golden_setup)(cfg)
  images = torch.stack([left, right]).contiguous()
  nat = Native(f, n)
  full = nat.forward(images)
  B, H, W = cfg["B"], cfg["H"], cfg["W"]
  D, h, w = dims(f, n, B, H, W)
  nws = nat.workspace_bytes(B, H, W) // 4
  sizes = dict(disp=B * H * W, coarse=B * H * W, cost=B * D * h * w, fcs=B * h * w)
  for optional in (True, False):
    wbuf, ws = banded(nws)
    bufs = {key: banded(sz) for key, sz in sizes.items() if optional or key == "disp"}
    outs = {key: v for key, (_, v) in bufs.items()}
    assert nat.call(images, ws, **outs) == 0, _cabi.lib().snb_last_error()
    torch.cuda.synchronize()
    assert intact(wbuf, nws), "workspace"
    for key, (buf, v) in bufs.items():
      assert intact(buf, sizes[key]), key
      assert bool((v != SENT).all().item()), key              # every output element was written
      assert torch.equal(v.view_as(full[key]), full[key]), key


@pytest.mark.gpu
def test_argument_errors_launch_nothing():
  cfg = CASES["k3_ragged"]
  f, n, left, right = golden_setup(cfg)
  images = torch.stack([left, right]).contiguous()
  nat = Native(f, n)
  B, H, W = cfg["B"], cfg["H"], cfg["W"]
  lib = _cabi.lib()
  ws = torch.empty((nat.workspace_bytes(B, H, W) + 256,), device=DEV, dtype=torch.uint8)
  disp = torch.full((B, H, W), SENT, device=DEV)
  torch.cuda.synchronize()
  st = stream_ptr()

  def fwd(k=3, maxdisp=192, img=images.data_ptr(), wsp=ws.data_ptr(), dp=disp.data_ptr(), fcs=None):
    return lib.snb_stereonet_forward(nat.weights.data_ptr(), k, 0, maxdisp, img, B, H, W, wsp, dp, None, None, fcs, st)

  cases = [
    (lambda: fwd(img=None), "images"),
    (lambda: fwd(dp=None), "disp"),
    (lambda: fwd(wsp=None), "workspace"),
    (lambda: fwd(wsp=ws.data_ptr() + 16), "workspace"),
    (lambda: fwd(maxdisp=1000), "maxdisp"),
    (lambda: fwd(k=0), "k"),
    (lambda: fwd(fcs=disp.data_ptr()), "cost"),
    (lambda: lib.snb_stereonet_forward(None, 3, 0, 192, images.data_ptr(), B, H, W, ws.data_ptr(), disp.data_ptr(), None, None,
                                       None, st), "weights"),
    (lambda: lib.snb_stereonet_prepare(None, 3, nat.weights.data_ptr(), st), "params"),
    (lambda: lib.snb_stereonet_prepare(native.param_pointers(f, n), 0, nat.weights.data_ptr(), st), "k"),
    (lambda: lib.snb_stereonet_prepare(native.param_pointers(f, n), 3, nat.weights.data_ptr() + 16, st), "weights"),
  ]
  for call, word in cases:
    assert call() != 0
    msg = lib.snb_last_error().decode()
    assert f"`{word}`" in msg or f"{word} " in msg, (word, msg)
  ptrs = native.param_pointers(f, n)
  ptrs[5] = None
  assert lib.snb_stereonet_prepare(ptrs, 3, nat.weights.data_ptr(), st) != 0
  assert "params[5]" in lib.snb_last_error().decode()
  assert lib.snb_stereonet_workspace_bytes(3, 0, 1000, B, H, W) == -1
  torch.cuda.synchronize()
  assert bool((disp == SENT).all().item())                   # nothing ran
  assert fwd() == 0                                          # and the same arguments, corrected, do


@pytest.mark.gpu
def test_example_host_matches_python_path(tmp_path):
  """examples/stereonet_infer.cpp (no torch): reads the exported weights and raw images, graph-replays the forward, writes the
  disparity — bit-identical to the Python path."""
  import importlib.util
  spec = importlib.util.spec_from_file_location("snb200_build", os.path.join(ROOT, "adaptive-stereo-icra-2021_b200", "build.py"))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  exe = mod.build_example(str(tmp_path / "stereonet_infer"))
  cfg = CASES["k3_b2_sharp"]
  f, n, left, right = golden_setup(cfg)
  B, H, W = cfg["B"], cfg["H"], cfg["W"]
  native.export_weights(f, n, str(tmp_path / "w.bin"))
  torch.stack([left, right]).cpu().numpy().astype("<f4").tofile(str(tmp_path / "img.bin"))
  r = subprocess.run([exe, str(tmp_path / "w.bin"), str(tmp_path / "img.bin"), str(B), str(H), str(W), str(tmp_path / "disp.bin"), "5"],
                     capture_output=True, text=True, timeout=300)
  assert r.returncode == 0, r.stdout + r.stderr
  assert "ms per frame" in r.stdout
  got = torch.from_numpy(np.fromfile(str(tmp_path / "disp.bin"), dtype="<f4").reshape(B, H, W))
  ref = python_path(f, n, left, right)["disp"].cpu()
  assert torch.equal(got, ref)
