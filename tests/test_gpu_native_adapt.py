"""The single-pass adaptation step of the C-ABI (snb_stereonet_adapt_*, csrc/adapt.cu) against the Python step it restates,
AdaptStepper(f, s, make_optimizer(f, s, lr, fused=True), two_streams=False): the bucket layout (CPU); bit-identical losses,
parameters, BatchNorm buffers, gradient bucket and Adam state over consecutive frames, with a skipped update, under CUDA-graph
capture; interoperation with the inference API and optim.FusedAdamClip; the reference goldens; guard bands and argument errors."""
import ctypes as C

import numpy as np
import pytest
import torch

import stereonet_oracle as O
import stereonet_b200 as S
from stereonet_b200 import _cabi, native
from stereonet_b200.adapt import AdaptStepper, make_optimizer
from stereonet_b200.losses import feature_contrast_mean, monodepth_single_loss
from stereonet_b200.optim import FusedAdamClip
from test_gpu_native import DEV, SENT, Native, banded, intact, python_path, stream_ptr
from test_oracle_golden import CASES, build, summ

LR = 5e-5

ADAPT = {
  "k3_96x256": dict(k=3, s=0, B=1, H=96, W=256, frames=3),
  "k4_320x960": dict(k=4, s=0, B=1, H=320, W=960, frames=3),
  "k3_s1_160x480": dict(k=3, s=1, B=1, H=160, W=480, frames=3),
  "k3_375x1242": dict(k=3, s=0, B=1, H=375, W=1242, frames=3),     # odd sizes: strided views over odd extents
  "k3_split_3x64": dict(k=3, s=0, B=1, H=3, W=64, frames=3),       # downsample[2] input of height 1: the phase-split branch
  "k3_b2_128x320": dict(k=3, s=0, B=2, H=128, W=320, frames=3),
  "kitti_376x1248": dict(k=3, s=0, B=1, H=376, W=1248, frames=1),
}


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("k", [3, 4])
def test_grad_slots_follow_fused_adam_layout(k):
  """params[i] -> bucket slot as optim.FusedAdamClip lays out its flat buffers (stereo_net first, no .conv2.)."""
  f, s = S.FeatureExtractorNetwork(k), S.StereoNet(k, 1, 0)
  expected, off = {}, 0
  for prefix, net in (("stereo_net.", s), ("feature_net.", f)):
    for n, p in net.named_parameters():
      if ".conv2." not in n:
        expected[prefix + n] = (off, p.numel())
        off += p.numel()
  lib = _cabi.lib()
  names = native.param_names(k)
  for i, name in enumerate(names):
    o, c = C.c_longlong(), C.c_longlong()
    assert lib.snb_stereonet_adapt_grad_slot(k, i, C.byref(o), C.byref(c)) == 0
    if name in expected:
      assert (o.value, c.value) == expected[name], name
    else:
      assert c.value == 0 and name.endswith(("running_mean", "running_var")), name
  assert set(expected) <= set(names)
  offs = []
  for what in range(4):
    o, nb = C.c_longlong(), C.c_longlong()
    assert lib.snb_stereonet_adapt_state_piece(k, what, C.byref(o), C.byref(nb)) == 0
    assert nb.value == (4 if what == 3 else 4 * off) and o.value % 256 == 0
    offs.append((o.value, o.value + nb.value))
  assert all(a[1] <= b[0] for a, b in zip(offs, offs[1:]))
  assert offs[-1][1] <= lib.snb_stereonet_adapt_state_bytes(k)
  assert lib.snb_stereonet_adapt_grad_slot(k, len(names), C.byref(o), C.byref(c)) != 0


# ---------------------------------------------------------------------------------------------------------------- helpers
def nets(cfg, fsd=None, ssd=None):
  fsd = fsd if fsd is not None else O.make_feature_state(cfg["k"], 11)
  ssd = ssd if ssd is not None else O.make_stereo_state(22, sharpen=40.0)
  f = S.FeatureExtractorNetwork(cfg["k"]).to(DEV)
  n = S.StereoNet(cfg["k"], 1, cfg["s"], maxdisp=192).to(DEV)
  f.load_state_dict(fsd, strict=True)
  n.load_state_dict(ssd, strict=True)
  return f, n


def twin(f, n, cfg):
  return nets(cfg, {k: v.clone() for k, v in f.state_dict().items()}, {k: v.clone() for k, v in n.state_dict().items()})


def frames(cfg, count, seed=7):
  g = torch.Generator(device=DEV).manual_seed(seed)
  return [torch.rand((2, cfg["B"], 3, cfg["H"], cfg["W"]), device=DEV, generator=g) for _ in range(count)]


def python_stepper(f, n, clip):
  return AdaptStepper(f, n, make_optimizer(f, n, lr=LR, fused=True), clip_grad_norm=clip, two_streams=False)


def outputs(cfg):
  B, H, W = cfg["B"], cfg["H"], cfg["W"]
  return dict(loss=torch.empty((1 + B,), device=DEV), disp=torch.empty((B, H, W), device=DEV), fcs_mean=torch.empty((1,), device=DEV))


def coarse_hw(cfg):
  h, w = cfg["H"], cfg["W"]
  for _ in range(cfg["k"]):
    h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1
  return h, w


def assert_same_model(fa, na, fb, nb):
  for (ka, a), (kb, b) in zip(list(fa.state_dict().items()) + list(na.state_dict().items()),
                              list(fb.state_dict().items()) + list(nb.state_dict().items())):
    assert ka == kb and torch.equal(a, b), (ka, (a.double() - b.double()).abs().max().item())


def assert_same_optimizer(nat, opt):
  for key, a, b in (("flat_grad", nat.flat_grad, opt.flat_grad), ("exp_avg", nat.exp_avg, opt.exp_avg),
                    ("exp_avg_sq", nat.exp_avg_sq, opt.exp_avg_sq), ("step", nat.step_t, opt.step_t)):
    assert torch.equal(a, b), (key, (a - b).abs().max().item())


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("clip", [True, False])
@pytest.mark.parametrize("name", list(ADAPT))
def test_update_frames_bit_identical_to_python_step(name, clip):
  cfg = ADAPT[name]
  fp, np_ = nets(cfg)
  fn, nn_ = twin(fp, np_, cfg)
  stepper = python_stepper(fp, np_, clip)
  nat = native.NativeAdapt(fn, nn_, lr=LR, clip_norm=1.0 if clip else None)
  s = cfg["s"]
  for img in frames(cfg, cfg["frames"]):
    loss_py, fcs_py, out_py = stepper.step(img[0], img[1])
    o = outputs(cfg)
    fcs = torch.empty((cfg["B"],) + coarse_hw(cfg), device=DEV)
    nat.forward(img, o["loss"], o["disp"], fcs, o["fcs_mean"])
    nat.update()
    torch.cuda.synchronize()
    assert torch.equal(o["loss"][0], loss_py), (o["loss"][0].item(), loss_py.item())
    assert torch.equal(o["disp"], out_py[f"pred_disp_l/{s}"][:, 0].detach())
    # the feature-contrast map the EMA of adapt.py:352-353 reads, as losses.feature_contrast_mean gives it for the Python step
    fcs_map_py = feature_contrast_mean(out_py[f"cost_volume_l/{s + cfg['k']}"])
    assert torch.equal(fcs, fcs_map_py), (fcs - fcs_map_py).abs().max().item()
    # its mean: a fixed-order double sum here, torch's float reduction there
    assert torch.allclose(o["fcs_mean"][0], fcs_py.float(), rtol=1e-5, atol=1e-6)
    assert o["fcs_mean"][0].item() == pytest.approx(fcs.double().mean().item(), rel=1e-6)
    assert_same_model(fp, np_, fn, nn_)
    assert_same_optimizer(nat, stepper.optimizer)


@pytest.mark.gpu
def test_update_skip_update():
  """A frame whose update the host skips still runs the train-mode forward: BatchNorm statistics and counters move."""
  cfg = ADAPT["k3_96x256"]
  fp, np_ = nets(cfg)
  fn, nn_ = twin(fp, np_, cfg)
  stepper = python_stepper(fp, np_, True)
  nat = native.NativeAdapt(fn, nn_, lr=LR)
  for i, img in enumerate(frames(cfg, 3, seed=9)):
    o = outputs(cfg)
    if i == 1:
      fp.train(); np_.train()
      stepper._refresh_weights()
      loss_py = monodepth_single_loss(img[0], img[1], stepper.predict(img[0], img[1]), 0)    # grad enabled, no backward
      nat.forward(img, o["loss"])
    else:
      loss_py = stepper.step(img[0], img[1])[0]
      nat.forward(img, o["loss"])
      nat.update()
    torch.cuda.synchronize()
    assert torch.equal(o["loss"][0], loss_py.detach())
    assert_same_model(fp, np_, fn, nn_)
    assert_same_optimizer(nat, stepper.optimizer)


@pytest.mark.gpu
def test_graph_capture_matches_eager():
  cfg = ADAPT["k3_375x1242"]
  B, H, W = cfg["B"], cfg["H"], cfg["W"]
  fe, ne = nets(cfg)
  fg, ng = twin(fe, ne, cfg)
  eager = native.NativeAdapt(fe, ne, lr=LR)
  graph = native.NativeAdapt(fg, ng, lr=LR)
  images = torch.empty((2, B, 3, H, W), device=DEV)
  og = outputs(cfg)
  graph.workspace(B, H, W)
  torch.cuda.synchronize()
  before = {k: v.clone() for k, v in list(fg.state_dict().items()) + list(ng.state_dict().items())}
  g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
  with torch.cuda.graph(g1):
    graph.forward(images, og["loss"], og["disp"], fcs_mean=og["fcs_mean"])
  with torch.cuda.graph(g2):
    graph.update()
  torch.cuda.synchronize()
  for k, v in list(fg.state_dict().items()) + list(ng.state_dict().items()):
    assert torch.equal(v, before[k]), k                          # capturing ran nothing
  for img in frames(cfg, 3, seed=11):
    images.copy_(img)
    g1.replay(); g2.replay()
    oe = outputs(cfg)
    eager.forward(img, oe["loss"], oe["disp"], fcs_mean=oe["fcs_mean"])
    eager.update()
    torch.cuda.synchronize()
    for key in oe:
      assert torch.equal(og[key], oe[key]), key
    assert_same_model(fe, ne, fg, ng)
    for a, b in ((graph.flat_grad, eager.flat_grad), (graph.exp_avg, eager.exp_avg), (graph.exp_avg_sq, eager.exp_avg_sq),
                 (graph.step_t, eager.step_t)):
      assert torch.equal(a, b)


@pytest.mark.gpu
def test_inference_api_and_fused_adam_interop():
  cfg = ADAPT["k3_b2_128x320"]
  fp, np_ = nets(cfg)
  fn, nn_ = twin(fp, np_, cfg)
  stepper = python_stepper(fp, np_, True)
  nat = native.NativeAdapt(fn, nn_, lr=LR)
  for img in frames(cfg, 2, seed=13):
    stepper.step(img[0], img[1])
    nat.forward(img, outputs(cfg)["loss"])
    nat.update()
  torch.cuda.synchronize()
  # the updated tensors feed the eval API; StereoEngine on modules loaded from them gives the same bits
  f2, n2 = twin(fn, nn_, cfg)
  f2.eval(); n2.eval(); fn.eval(); nn_.eval()
  left, right = frames(cfg, 1, seed=17)[0]
  ref = python_path(f2, n2, left, right)
  got = Native(fn, nn_).forward(torch.stack([left, right]).contiguous())
  torch.cuda.synchronize()
  for key in ("disp", "coarse", "cost", "fcs"):
    assert torch.equal(got[key], ref[key]), key
  # the Adam state converts to FusedAdamClip (and so to torch.optim.Adam's state_dict) and back
  opt = FusedAdamClip(nn_, fn, lr=LR)
  nat.to_fused(opt)
  sa, sb = opt.state_dict(), stepper.optimizer.state_dict()
  assert sa["param_groups"] == sb["param_groups"] and sa["state"].keys() == sb["state"].keys()
  for i in sa["state"]:
    for key in ("step", "exp_avg", "exp_avg_sq"):
      assert torch.equal(sa["state"][i][key], sb["state"][i][key]), (i, key)
  other = native.NativeAdapt(*twin(fn, nn_, cfg), lr=LR)
  other.from_fused(opt)
  assert torch.equal(other.exp_avg, nat.exp_avg) and torch.equal(other.exp_avg_sq, nat.exp_avg_sq)
  assert torch.equal(other.step_t, nat.step_t)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n, c in CASES.items() if c["train"]])
def test_bucket_vs_reference_golden(name):
  """Independent of the Python path: the native bucket (no clipping) against the reference's own gradients, with the bands of
  tests/test_gpu_backward.py::test_adapt_step_vs_reference_golden (see there for why they are this wide)."""
  import os
  from test_gpu_backward import GOLD, TRAIN_SHARPEN_RATIO
  cfg = dict(CASES[name])
  g = np.load(os.path.join(GOLD, name + ".npz"))
  fsd, _, left, right, _ = build(cfg)
  ssd = O.make_stereo_state(seed=22, sharpen=cfg["sharpen"] * TRAIN_SHARPEN_RATIO)
  f, n = nets(cfg, fsd, ssd)
  nat = native.NativeAdapt(f, n, lr=LR, clip_norm=None)
  o = outputs(cfg)
  nat.forward(torch.stack([left, right]).to(DEV).contiguous(), o["loss"])
  nat.update()
  torch.cuda.synchronize()
  assert abs(o["loss"][0].item() - float(g["train/loss"])) < 2e-5
  lib = _cabi.lib()
  for i, full in enumerate(native.param_names(cfg["k"])):
    o_, c_ = C.c_longlong(), C.c_longlong()
    lib.snb_stereonet_adapt_grad_slot(cfg["k"], i, C.byref(o_), C.byref(c_))
    if c_.value == 0:
      continue
    tag, pname = ("s" if full.startswith("stereo_net.") else "f"), full.split(".", 1)[1]
    if pname.endswith(".0.0.bias") or pname == "conv3d_alone.bias" or f"grad_none/{tag}/{pname}" in g.files:
      continue
    grad = nat.flat_grad[o_.value:o_.value + c_.value].cpu()
    ref, got = g[f"grad_sum/{tag}/{pname}"], summ(grad)
    if ref[2] < 1e-6:
      assert got[2] < 1e-5, pname
      continue
    assert abs(got[2] - ref[2]) / (ref[2] + 1e-12) <= (6e-2 if c_.value == 1 else 3e-2), (pname, got, ref)
    key = f"grad/{tag}/{pname}"
    if key in g.files:
      a, b = grad.numpy().astype(np.float64), g[key].ravel().astype(np.float64)
      assert float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30)) >= 0.997, key
      assert np.abs(a - b).max() <= 1.2e-1 * (np.abs(b).max() + 1e-12), key


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["k3_split_3x64", "k3_375x1242"])
def test_writes_stay_inside_buffers(name):
  cfg = ADAPT[name]
  B, H, W, k = cfg["B"], cfg["H"], cfg["W"], cfg["k"]
  h, w = H, W
  for _ in range(k):
    h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1
  lib = _cabi.lib()
  img = frames(cfg, 1, seed=19)[0]
  fr, nr = nets(cfg)
  ref = native.NativeAdapt(fr, nr, lr=LR)
  oref = dict(outputs(cfg), fcs=torch.empty((B, h, w), device=DEV))
  ref.forward(img, oref["loss"], oref["disp"], oref["fcs"], oref["fcs_mean"])
  ref.update()
  sizes = dict(loss=1 + B, disp=B * H * W, fcs=B * h * w, fcs_mean=1)
  nstate = lib.snb_stereonet_adapt_state_bytes(k) // 4
  nws = lib.snb_stereonet_adapt_workspace_bytes(k, cfg["s"], 192, B, H, W) // 4
  for optional in (True, False):
    f, n = nets(cfg)
    sbuf, state = banded(nstate)
    wbuf, ws = banded(nws)
    bufs = {key: banded(sz) for key, sz in sizes.items() if optional or key == "loss"}
    p = lambda key: bufs[key][1].data_ptr() if key in bufs else None
    params, st = native.param_pointers(f, n), stream_ptr()
    assert lib.snb_stereonet_adapt_init(params, k, state.data_ptr(), st) == 0
    assert lib.snb_stereonet_adapt_forward(params, native.bn_counters(f, n), k, cfg["s"], 192, img.data_ptr(), B, H, W, state.data_ptr(),
                                           ws.data_ptr(), p("loss"), p("disp"), p("fcs"), p("fcs_mean"), st) == 0, lib.snb_last_error()
    assert lib.snb_stereonet_adapt_update(params, k, cfg["s"], 192, B, H, W, state.data_ptr(), ws.data_ptr(), 1.0, LR, 0.9, 0.999, 1e-8,
                                          st) == 0, lib.snb_last_error()
    torch.cuda.synchronize()
    assert intact(sbuf, nstate), "state"
    assert intact(wbuf, nws), "workspace"
    for key, (buf, v) in bufs.items():
      assert intact(buf, sizes[key]), key
      assert torch.equal(v, oref[key].flatten()), key
    assert_same_model(fr, nr, f, n)


@pytest.mark.gpu
def test_argument_errors_launch_nothing():
  cfg = ADAPT["k3_96x256"]
  B, H, W = cfg["B"], cfg["H"], cfg["W"]
  f, n = nets(cfg)
  nat = native.NativeAdapt(f, n, lr=LR)
  img = frames(cfg, 1)[0]
  ws = nat.workspace(B, H, W)
  lib = _cabi.lib()
  loss = torch.full((1 + B,), SENT, device=DEV)
  before = {k: v.clone() for k, v in list(f.state_dict().items()) + list(n.state_dict().items())}
  torch.cuda.synchronize()
  st = stream_ptr()

  def fwd(k=3, maxdisp=192, params=nat.params, im=img.data_ptr(), state=nat.state.data_ptr(), wsp=ws.data_ptr(), lp=loss.data_ptr(),
          fcs=None):
    return lib.snb_stereonet_adapt_forward(params, nat.counters, k, 0, maxdisp, im, B, H, W, state, wsp, lp, None, fcs, None, st)

  def upd(k=3, s=0, maxdisp=192, b=B, h=H, w=W, params=nat.params, state=nat.state.data_ptr(), wsp=ws.data_ptr(), beta1=0.9):
    return lib.snb_stereonet_adapt_update(params, k, s, maxdisp, b, h, w, state, wsp, 1.0, LR, beta1, 0.999, 1e-8, st)

  bad = native.param_pointers(f, n)
  bad[7] = None
  odd = native.param_pointers(f, n)
  odd[3] = odd[3] + 4
  cases = [
    (lambda: fwd(im=None), "images"),
    (lambda: fwd(lp=None), "loss"),
    (lambda: fwd(wsp=None), "workspace"),
    (lambda: fwd(wsp=ws.data_ptr() + 16), "workspace"),
    (lambda: fwd(state=nat.state.data_ptr() + 64), "state"),
    (lambda: fwd(params=None), "params"),
    (lambda: fwd(params=bad), "params[7]"),
    (lambda: fwd(params=odd), "params[3]"),
    (lambda: fwd(k=0), "k"),
    (lambda: fwd(maxdisp=1000), "maxdisp"),
    (lambda: fwd(maxdisp=15, fcs=loss.data_ptr()), "fcs"),
    (lambda: upd(wsp=None), "workspace"),
    (lambda: upd(state=None), "state"),
    (lambda: upd(params=bad), "params[7]"),
    (lambda: upd(k=17), "k"),
    (lambda: upd(maxdisp=-1), "maxdisp"),
    (lambda: upd(beta1=1.0), "beta1"),
    (lambda: lib.snb_stereonet_adapt_init(nat.params, 3, nat.state.data_ptr() + 16, st), "state"),
  ]
  for call, word in cases:
    assert call() != 0, word
    msg = lib.snb_last_error().decode()
    assert f"`{word}`" in msg or f"{word} " in msg, (word, msg)
  assert lib.snb_stereonet_adapt_workspace_bytes(3, 0, 1000, B, H, W) == -1
  torch.cuda.synchronize()
  assert bool((loss == SENT).all().item())                    # nothing ran
  for k, v in list(f.state_dict().items()) + list(n.state_dict().items()):
    assert torch.equal(v, before[k]), k
  assert fwd() == 0                                           # and the same arguments, corrected, do
  # an update must carry its forward's arguments: anything else is rejected by name before any launch (a larger shape would
  # otherwise write past a workspace sized for the forward)
  torch.cuda.synchronize()
  after = {k: v.clone() for k, v in list(f.state_dict().items()) + list(n.state_dict().items())}
  grad0 = nat.flat_grad.clone()
  other = torch.empty((ws.numel() + 512,), device=DEV, dtype=torch.uint8)
  alt = native.param_pointers(f, n)
  alt[5] = alt[6]
  mismatched = [
    (lambda: upd(h=H + 2), "H"),
    (lambda: upd(w=W - 8), "W"),
    (lambda: upd(b=2), "B"),
    (lambda: upd(s=1), "input_scale"),
    (lambda: upd(maxdisp=100), "maxdisp"),
    (lambda: upd(k=4, params=native.param_pointers(*nets(dict(cfg, k=4)))), "k"),
    (lambda: upd(state=nat.state.data_ptr() + 256), "state"),
    (lambda: upd(params=alt), "params[5]"),
    (lambda: upd(wsp=other.data_ptr() + 256), "workspace"),
  ]
  for call, word in mismatched:
    assert call() != 0, word
    msg = lib.snb_last_error().decode()
    assert f"`{word}`" in msg, (word, msg)
  torch.cuda.synchronize()
  assert torch.equal(nat.flat_grad, grad0)
  for k, v in list(f.state_dict().items()) + list(n.state_dict().items()):
    assert torch.equal(v, after[k]), k
  assert upd() == 0
  with pytest.raises(RuntimeError, match="images"):
    nat.forward(img.transpose(3, 4), loss)                   # the Python helper checks shapes, dtype and layout
  with pytest.raises(RuntimeError, match="loss"):
    nat.forward(img, loss[:1])


@pytest.mark.gpu
def test_example_host_matches_native_api(tmp_path):
  """examples/stereonet_adapt.cpp (no torch): adapts over raw frames and writes the weights file, which equals the same frames
  through the native API from Python."""
  import importlib.util
  import os
  import subprocess
  from test_gpu_native import ROOT
  spec = importlib.util.spec_from_file_location("snb200_build", os.path.join(ROOT, "adaptive-stereo-icra-2021_b200", "build.py"))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  exe = mod.build_example(str(tmp_path / "stereonet_adapt"), "stereonet_adapt")
  cfg = ADAPT["k3_b2_128x320"]
  B, H, W = cfg["B"], cfg["H"], cfg["W"]
  f, n = nets(cfg)
  native.export_weights(f, n, str(tmp_path / "w.bin"))
  imgs = frames(cfg, 2, seed=23)
  torch.stack(imgs).cpu().numpy().astype("<f4").tofile(str(tmp_path / "img.bin"))
  r = subprocess.run([exe, str(tmp_path / "w.bin"), str(tmp_path / "img.bin"), str(B), str(H), str(W), "2", str(tmp_path / "out.bin")],
                     capture_output=True, text=True, timeout=300)
  assert r.returncode == 0, r.stdout + r.stderr
  assert r.stdout.count("loss") == 2
  nat = native.NativeAdapt(f, n, lr=LR)
  for img in imgs:
    nat.forward(img, outputs(cfg)["loss"])
    nat.update()
  torch.cuda.synchronize()
  native.export_weights(f, n, str(tmp_path / "ref.bin"))
  assert (tmp_path / "out.bin").read_bytes() == (tmp_path / "ref.bin").read_bytes()
