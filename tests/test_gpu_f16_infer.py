"""The opt-in reduced-precision inference forward: snb_conv_c32_ws_f16 (one fp16 product per tap) against an fp64 reference of the
same layer, the whole model (snb_stereonet_forward_f16 / StereoEngine(precision="fp16")) against the oracle with the errors printed
and bounded, native against Python bit for bit, CUDA-graph capture, guard bands, argument errors and the example host.  These numbers
are reported apart from the fp32 parity contract that every other test holds the default path to."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import stereonet_oracle as O
from stereonet_b200 import _cabi, ops
from stereonet_b200.autograd import fused
from stereonet_b200.runtime import StereoEngine
from test_gpu_kernels import cl, uncl, rnd
from test_gpu_native import (ALL, KITTI, SENT, Native, banded, dims, golden_setup, intact, make_nets, random_setup, stream_ptr,
                             python_path)
from test_oracle_golden import BIG_CASES, CASES, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
LAYER_TOL = 3e-3          # single-pass tolerance of test_gpu_conv_tc.py: max error <= 3e-3 x max |output|

# Whole model against the oracle (refined and coarse disparity, px).  The sanity bounds of the single-pass TF32 cross-check
# (test_gpu_e2e.py::test_conv_backends_agree[tc1]) are |dEPE| <= 0.1 and median |d disp| <= 0.5.  The bounds below are twice the
# largest value measured over MODEL_CASES on an NVIDIA B200 (DESIGN.md section 4.2f16): |dEPE| 0.0152, median 0.0737, p99 0.887,
# max 2.97 px.
BOUNDS = dict(depe=0.03, median=0.15, p99=1.8, max=6.0)

MODEL_CASES = ["T_320x960_k3", "k4_320x960", "k3s1_160x480", "k3_ragged", "k3_b2_sharp", "k4_sharp",
               "kitti_376x1248_b1", "kitti_376x1248_b2", "kitti_375x1242_b1"]
LAYER_SETS = {"2d": frozenset(("2d",)), "3d": frozenset(("3d",)), "both": frozenset(("2d", "3d"))}


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_engine_precision_is_checked():
  with pytest.raises(ValueError, match="precision"):
    StereoEngine(None, None, precision="bf16")
  assert fused.F16_LAYERS == frozenset()
  assert fused.F16_SHIPPED <= LAYER_SETS["both"]


# ---------------------------------------------------------------------------------------------------------------- layers
def _layer(x, w, b, scale, shift, residual, lrelu, dil, three_d):
  """fp64 reference of one 32->32 'same' layer with the walk kernel's epilogue (NCHW / NCDHW)."""
  conv = F.conv3d if three_d else F.conv2d
  z = conv(x.double(), w.double(), b.double(), padding=dil, dilation=dil)
  shp = (1, 32) + (1,) * (z.dim() - 2)
  if scale is not None:
    z = z * scale.double().view(shp) + shift.double().view(shp)
  if lrelu:
    z = F.leaky_relu(z, 0.2)
  if residual is not None:
    z = z + residual.double()
  return z


def _run_layer(x, w, b, scale, shift, residual, lrelu, dil, three_d):
  g = ops.geom(tuple(cl(x).shape), 3, dil=dil)
  wimg = ops.prep_conv_weights_tc(w.to(DEV), 0, fmt="ws")
  kw = dict(bias=b.to(DEV), scale=None if scale is None else scale.to(DEV), shift=None if shift is None else shift.to(DEV),
            lrelu=lrelu)
  xc = cl(x)                     # a residual that is the input takes the kernel's on-chip path, any other one the TMA-loaded tile
  rc = None if residual is None else (xc if residual is x else cl(residual))
  y16 = ops.conv_c32_ws_f16(xc, wimg, g, residual=rc, **kw)
  y32, _ = ops.conv_c32_tc(xc, wimg, g, residual=rc, fmt="ws", **kw)
  return uncl(y16), uncl(y32)


def _check_layer(got, ref, y32, what):
  err = (got.double() - ref).abs().max().item()
  mag = ref.abs().max().item()
  print(f"[f16 layer] {what}: max err / max |out| = {err / mag:.3e}")
  assert err <= LAYER_TOL * mag, f"{what}: {err:.3e} vs {mag:.3e}"
  assert not torch.equal(got, y32), f"{what}: identical to the fp32-grade kernel (the variant did not run)"


@pytest.mark.gpu
@pytest.mark.parametrize("xscale", [1e-2, 1.0, 1e2])
@pytest.mark.parametrize("epi", ["bias", "bn_lrelu_residual", "residual_tile"])
@pytest.mark.parametrize("dil", [1, 2, 4, 8])
def test_layer_2d_vs_fp64(dil, epi, xscale):
  x, w, b = rnd(1, 32, 37, 300, seed=1) * xscale, rnd(32, 32, 3, 3, seed=2, scale=0.1), rnd(32, seed=3) * xscale
  scale, shift, residual, lrelu = None, None, None, False
  if epi != "bias":
    scale, shift, lrelu = rnd(32, seed=4).abs() + 0.5, rnd(32, seed=5) * xscale, True
    residual = x if epi == "bn_lrelu_residual" else rnd(1, 32, 37, 300, seed=6) * xscale
  got, y32 = _run_layer(x, w, b, scale, shift, residual, lrelu, dil, False)
  _check_layer(got, _layer(x, w, b, scale, shift, residual, lrelu, dil, False), y32, f"2-D dil={dil} {epi} xscale={xscale}")


@pytest.mark.gpu
@pytest.mark.parametrize("xscale", [1e-2, 1.0, 1e2])
@pytest.mark.parametrize("H,W", [(9, 40), (7, 45), (47, 156)])        # H*W = 360, 315 (ragged), 7332 (KITTI coarse size)
@pytest.mark.parametrize("epi", ["bias", "bn_lrelu"])
def test_layer_3d_vs_fp64(H, W, epi, xscale):
  x, w, b = rnd(1, 32, 24, H, W, seed=1) * xscale, rnd(32, 32, 3, 3, 3, seed=2, scale=0.05), rnd(32, seed=3) * xscale
  scale, shift, lrelu = (None, None, False) if epi == "bias" else (rnd(32, seed=4).abs() + 0.5, rnd(32, seed=5) * xscale, True)
  got, y32 = _run_layer(x, w, b, scale, shift, None, lrelu, 1, True)
  _check_layer(got, _layer(x, w, b, scale, shift, None, lrelu, 1, True), y32, f"3-D {H}x{W} {epi} xscale={xscale}")


@pytest.mark.gpu
def test_layer_rejects_stats_by_name():
  lib = _cabi.lib()
  x = torch.randn(1, 16, 40, 32, device=DEV)
  w = ops.prep_conv_weights_tc(torch.randn(32, 32, 3, 3, device=DEV) * 0.1, 0, fmt="ws")
  y = torch.full_like(x, SENT)
  g = ops.geom(tuple(x.shape), 3)
  stats = torch.zeros((lib.snb_conv_c32_ws_num_tiles(C.byref(g)), 2, 32), device=DEV)
  e = _cabi.ConvEpilogue(None, None, None, None, C.c_void_p(stats.data_ptr()), 0)
  torch.cuda.synchronize()
  assert lib.snb_conv_c32_ws_f16(x.data_ptr(), w.data_ptr(), y.data_ptr(), C.byref(g), C.byref(e), stream_ptr()) != 0
  assert "`stats`" in lib.snb_last_error().decode()
  torch.cuda.synchronize()
  assert bool((y == SENT).all().item())                      # nothing ran
  with torch.no_grad():                                      # the Python switch refuses train-mode statistics as well
    fused.F16_LAYERS = fused.F16_SHIPPED
    try:
      with pytest.raises(RuntimeError, match="eval-mode"):
        fused.conv3x3_c32(x, torch.nn.Conv2d(32, 32, 3, padding=1).to(DEV), g, want_stats=True)
    finally:
      fused.F16_LAYERS = frozenset()


# ---------------------------------------------------------------------------------------------------------------- whole model
def oracle_setup(name):
  """Weights and the synthetic pair with ground truth, as the e2e `kitti` fixture builds them (sharpened conv3d_alone)."""
  if name in KITTI:
    cfg = dict(KITTI[name], sharpen=40.0)
    fsd, ssd = O.make_feature_state(cfg["k"], 11), O.make_stereo_state(22, sharpen=40.0)
    left, right, gt = O.make_stereo_pair(cfg["B"], cfg["H"], cfg["W"], seed=1000, max_disp_px=60.0)
  else:
    cfg = dict(BIG_CASES.get(name) or CASES[name])
    fsd, ssd, left, right, gt = build(cfg)
  return cfg, fsd, ssd, left, right, gt


def disp_stats(got, ref, gt):
  d = (got - ref).abs().flatten().double()
  return dict(max=d.max().item(), median=d.median().item(), p99=torch.quantile(d, 0.99).item(),
              depe=abs(O.epe(got, gt).item() - O.epe(ref, gt).item()))


def _with_layers(layers, fn):
  old = fused.F16_LAYERS
  fused.F16_LAYERS = layers
  try:
    with torch.no_grad():
      return fn()
  finally:
    fused.F16_LAYERS = old


@pytest.mark.gpu
@pytest.mark.parametrize("name", MODEL_CASES)
def test_model_vs_oracle(name):
  """The three layer sets (2-D only, 3-D only, both) on the module forward, and the shipped forward (StereoEngine fp16), against
  the oracle: max, median, p99 |d disp| and |d EPE| of the refined and the coarse disparity."""
  cfg, fsd, ssd, left, right, gt = oracle_setup(name)
  f, n = make_nets(cfg["k"], cfg["s"], fsd, ssd)
  s, k = cfg["s"], cfg["k"]
  with torch.no_grad():
    ref = O.predict_disparity_left(fsd, ssd, left, right, k, s)
  l, r = left.to(DEV), right.to(DEV)
  keys = {"refined": f"pred_disp_l/{s}", "coarse": f"pred_disp_l/{s + k}"}
  for tag, layers in LAYER_SETS.items():
    out = _with_layers(layers, lambda: n(l, f(l), f(r), "l", output_cost_volume=True))
    for which, key in keys.items():
      st = disp_stats(out[key].cpu(), ref[key], gt)
      print(f"[f16 model] {name} layers={tag} {which}: " + " ".join(f"{a}={v:.3e}" for a, v in st.items()))
  out = StereoEngine(f, n, output_cost_volume=True, precision="fp16")(l, r)
  for which, key in keys.items():
    st = disp_stats(out[key].cpu(), ref[key], gt)
    print(f"[f16 model] {name} shipped {which}: " + " ".join(f"{a}={v:.3e}" for a, v in st.items()))
    for a, bound in BOUNDS.items():
      if bound is not None:
        assert st[a] <= bound, (name, which, a, st[a], bound)


# ---------------------------------------------------------------------------------------------------------------- native
class NativeF16(Native):
  def call(self, images, ws, disp, coarse=None, cost=None, fcs=None, stream=None):
    B, H, W = images.shape[1], images.shape[-2], images.shape[-1]
    p = lambda t: None if t is None else t.data_ptr()
    return _cabi.lib().snb_stereonet_forward_f16(self.weights.data_ptr(), self.k, self.n.input_scale, self.n.maxdisp, p(images), B,
                                                 H, W, p(ws), p(disp), p(coarse), p(cost), p(fcs), stream_ptr(stream))


def python_f16(f, n, left, right):
  from stereonet_b200.losses import feature_contrast_mean
  out = StereoEngine(f, n, output_cost_volume=True, precision="fp16")(left, right)
  s, k = n.input_scale, f.k
  cost = out[f"cost_volume_l/{s + k}"]
  return dict(disp=out[f"pred_disp_l/{s}"][:, 0].clone(), coarse=out[f"pred_disp_l/{s + k}"][:, 0].clone(), cost=cost.clone(),
              fcs=feature_contrast_mean(cost).clone())


def setup(name):
  return (random_setup if name in KITTI else golden_setup)(ALL[name])


@pytest.mark.gpu
@pytest.mark.parametrize("name", MODEL_CASES)
def test_native_bit_identical_to_engine(name):
  f, n, left, right = setup(name)
  ref = python_f16(f, n, left, right)
  got = NativeF16(f, n).forward(torch.stack([left, right]).contiguous())
  torch.cuda.synchronize()
  for key in ("disp", "coarse", "cost", "fcs"):
    assert torch.equal(got[key], ref[key]), (name, key, (got[key] - ref[key]).abs().max().item())
  default = python_path(f, n, left, right)                   # the default forward is untouched by the fp16 engine
  fp32 = Native(f, n).forward(torch.stack([left, right]).contiguous())
  torch.cuda.synchronize()
  assert fused.F16_LAYERS == frozenset()
  for key in ("disp", "coarse", "cost", "fcs"):
    assert torch.equal(fp32[key], default[key]), (name, key)
  assert not torch.equal(got["disp"], fp32["disp"])


@pytest.mark.gpu
def test_graph_capture_matches_eager():
  f, n, left, right = setup("kitti_375x1242_b1")
  images = torch.stack([left, right]).contiguous()
  nat = NativeF16(f, n)
  eager = nat.forward(images)
  B, H, W = images.shape[1], images.shape[-2], images.shape[-1]
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


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["k3_ragged", "kitti_375x1242_b1", "k4_sharp"])
def test_writes_stay_inside_buffers(name):
  f, n, left, right = setup(name)
  images = torch.stack([left, right]).contiguous()
  nat = NativeF16(f, n)
  full = nat.forward(images)
  cfg = ALL[name]
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
      assert bool((v != SENT).all().item()), key
      assert torch.equal(v.view_as(full[key]), full[key]), key


@pytest.mark.gpu
def test_argument_errors_launch_nothing():
  cfg = CASES["k3_ragged"]
  f, n, left, right = golden_setup(cfg)
  images = torch.stack([left, right]).contiguous()
  nat = NativeF16(f, n)
  B, H, W = cfg["B"], cfg["H"], cfg["W"]
  lib = _cabi.lib()
  ws = torch.empty((nat.workspace_bytes(B, H, W) + 256,), device=DEV, dtype=torch.uint8)
  disp = torch.full((B, H, W), SENT, device=DEV)
  torch.cuda.synchronize()
  st = stream_ptr()

  def fwd(k=3, maxdisp=192, img=images.data_ptr(), wsp=ws.data_ptr(), dp=disp.data_ptr(), fcs=None, weights=nat.weights.data_ptr()):
    return lib.snb_stereonet_forward_f16(weights, k, 0, maxdisp, img, B, H, W, wsp, dp, None, None, fcs, st)

  cases = [(lambda: fwd(img=None), "images"), (lambda: fwd(dp=None), "disp"), (lambda: fwd(wsp=None), "workspace"),
           (lambda: fwd(wsp=ws.data_ptr() + 16), "workspace"), (lambda: fwd(maxdisp=1000), "maxdisp"), (lambda: fwd(k=0), "k"),
           (lambda: fwd(fcs=disp.data_ptr()), "cost"), (lambda: fwd(weights=None), "weights")]
  for call, word in cases:
    assert call() != 0
    msg = lib.snb_last_error().decode()
    assert "snb_stereonet_forward_f16" in msg and (f"`{word}`" in msg or f"{word} " in msg), (word, msg)
  torch.cuda.synchronize()
  assert bool((disp == SENT).all().item())
  assert fwd() == 0


@pytest.mark.gpu
def test_engine_refuses_train_mode_and_grad():
  f, n, left, right = golden_setup(CASES["k3_ragged"])
  f.train()
  with pytest.raises(RuntimeError, match="eval-mode"):
    StereoEngine(f, n, precision="fp16")(left, right)
  f.eval()
  assert fused.F16_LAYERS == frozenset()
  fused.F16_LAYERS = fused.F16_SHIPPED                       # set with grad enabled: every layer entry point refuses
  try:
    with pytest.raises(RuntimeError, match="no_grad"):
      f(left)
  finally:
    fused.F16_LAYERS = frozenset()


@pytest.mark.gpu
def test_example_host_f16_matches_native(tmp_path):
  import importlib.util
  spec = importlib.util.spec_from_file_location("snb200_build", os.path.join(ROOT, "adaptive-stereo-icra-2021_b200", "build.py"))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  exe = mod.build_example(str(tmp_path / "stereonet_infer"))
  cfg = CASES["k3_b2_sharp"]
  f, n, left, right = golden_setup(cfg)
  B, H, W = cfg["B"], cfg["H"], cfg["W"]
  from stereonet_b200 import native
  native.export_weights(f, n, str(tmp_path / "w.bin"))
  images = torch.stack([left, right]).contiguous()
  images.cpu().numpy().astype("<f4").tofile(str(tmp_path / "img.bin"))
  r = subprocess.run([exe, str(tmp_path / "w.bin"), str(tmp_path / "img.bin"), str(B), str(H), str(W), str(tmp_path / "disp.bin"), "5",
                      "f16"], capture_output=True, text=True, timeout=300)
  assert r.returncode == 0, r.stdout + r.stderr
  assert "f16" in r.stdout and "ms per frame" in r.stdout
  got = torch.from_numpy(np.fromfile(str(tmp_path / "disp.bin"), dtype="<f4").reshape(B, H, W))
  ref = NativeF16(f, n).forward(images)["disp"].cpu()
  assert torch.equal(got, ref)
