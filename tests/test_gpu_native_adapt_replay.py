"""The experience-replay adaptation step of the C-ABI (snb_stereonet_adapt_forward_replay / _update_replay, csrc/adapt.cu) against
the Python step it restates, AdaptStepper(f, s, make_optimizer(f, s, lr, fused=True), two_streams=False).step(left, right,
replay=(rl, rr, gt)): bit-identical losses, disparity, parameters, BatchNorm buffers, gradient bucket and Adam state over consecutive
frames with changing replay samples, an all-invalid replay frame, a skipped update, CUDA-graph capture; the reference's own ER step
(tests/golden/rows_f3_f4.npz); guard bands, argument errors and the example host."""
import math

import numpy as np
import pytest
import torch

import stereonet_oracle as O
from stereonet_b200 import _cabi, native
from stereonet_b200.losses import feature_contrast_mean, khamis_robust_loss, monodepth_single_loss
from test_gpu_native import DEV, SENT, banded, intact, stream_ptr
from test_gpu_native_adapt import LR, assert_same_model, assert_same_optimizer, coarse_hw, frames, nets, outputs, python_stepper, twin

ER_WEIGHT = 0.05

ADAPT_ER = {
  "k3_96x256": dict(k=3, s=0, B=1, RB=1, H=96, W=256, frames=3),
  "k3_b2_128x320": dict(k=3, s=0, B=2, RB=1, H=128, W=320, frames=3),
  "k3_rb2_96x256": dict(k=3, s=0, B=1, RB=2, H=96, W=256, frames=3),
  "k4_320x960": dict(k=4, s=0, B=1, RB=1, H=320, W=960, frames=3),
  "k3_s1_160x480": dict(k=3, s=1, B=1, RB=1, H=160, W=480, frames=3),
  "k3_375x1242": dict(k=3, s=0, B=1, RB=1, H=375, W=1242, frames=3),     # odd sizes: strided views over odd extents
  "k3_split_3x64": dict(k=3, s=0, B=1, RB=1, H=3, W=64, frames=3),       # downsample[2] input of height 1: the phase-split branch
  "kitti_376x1248": dict(k=3, s=0, B=1, RB=1, H=376, W=1248, frames=1),
}


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_replay_workspace_bytes():
  """The replay pair's workspace holds both passes' activations: more than the single pass's, growing with RB; RB < 1 and the
  shapes the calls reject give -1."""
  lib = _cabi.lib()
  plain = lib.snb_stereonet_adapt_workspace_bytes(3, 0, 192, 1, 96, 256)
  one = lib.snb_stereonet_adapt_replay_workspace_bytes(3, 0, 192, 1, 96, 256, 1)
  two = lib.snb_stereonet_adapt_replay_workspace_bytes(3, 0, 192, 1, 96, 256, 2)
  assert 0 < plain < one < two and one % 256 == 0
  assert lib.snb_stereonet_adapt_replay_workspace_bytes(3, 0, 192, 1, 96, 256, 0) == -1
  assert b"`RB`" in lib.snb_last_error()
  assert lib.snb_stereonet_adapt_replay_workspace_bytes(3, 0, 1000, 1, 96, 256, 1) == -1


# ---------------------------------------------------------------------------------------------------------------- helpers
def replay_samples(cfg, count, seed=31):
  """`count` stored samples (images [2,RB,3,H,W], gt [RB,H,W]); the gt has an invalid band (gt = 0) over the first quarter of the
  columns and is positive elsewhere."""
  g = torch.Generator(device=DEV).manual_seed(seed)
  RB, H, W = cfg["RB"], cfg["H"], cfg["W"]
  out = []
  for _ in range(count):
    img = torch.rand((2, RB, 3, H, W), device=DEV, generator=g)
    gt = torch.rand((RB, H, W), device=DEV, generator=g) * 40.0 + 0.5
    gt[:, :, :max(1, W // 4)] = 0.0
    out.append((img, gt))
  return out


def record_predictions(stepper):
  """Keep what every AdaptStepper.predict call returns (per step: the stream pass, then the replay pass)."""
  seen, predict = [], stepper.predict

  def wrapped(left, right):
    out = predict(left, right)
    seen.append(out)
    return out
  stepper.predict = wrapped
  return seen


def replay_outputs(cfg):
  return dict(outputs(cfg), loss_replay=torch.empty((2,), device=DEV))


def python_terms(cfg, img, rimg, gt, out, out_er):
  """The photometric loss of the stream pass and the Khamis term of the replay pass the Python step formed (same kernels, same
  inputs: the same bits)."""
  s = cfg["s"]
  with torch.no_grad():
    return (monodepth_single_loss(img[0], img[1], out, s), khamis_robust_loss(out_er[f"pred_disp_l/{s}"], gt))


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("clip", [True, False])
@pytest.mark.parametrize("name", list(ADAPT_ER))
def test_replay_frames_bit_identical_to_python_step(name, clip):
  cfg = ADAPT_ER[name]
  fp, np_ = nets(cfg)
  fn, nn_ = twin(fp, np_, cfg)
  stepper = python_stepper(fp, np_, clip)
  seen = record_predictions(stepper)
  nat = native.NativeAdapt(fn, nn_, lr=LR, clip_norm=1.0 if clip else None)
  s = cfg["s"]
  for img, (rimg, gt) in zip(frames(cfg, cfg["frames"]), replay_samples(cfg, cfg["frames"])):
    total_py = stepper.step(img[0], img[1], replay=(rimg[0], rimg[1], gt))[0]
    out_py, out_er = seen[-2], seen[-1]
    loss_py, khamis_py = python_terms(cfg, img, rimg, gt, out_py, out_er)
    o = replay_outputs(cfg)
    fcs = torch.empty((cfg["B"],) + coarse_hw(cfg), device=DEV)
    nat.forward(img, o["loss"], o["disp"], fcs, o["fcs_mean"], replay=(rimg, gt), loss_replay=o["loss_replay"], er_weight=ER_WEIGHT)
    nat.update()
    torch.cuda.synchronize()
    assert torch.equal(o["loss"][0], loss_py), (o["loss"][0].item(), loss_py.item())
    assert torch.equal(o["loss_replay"][0], khamis_py), (o["loss_replay"][0].item(), khamis_py.item())
    assert torch.equal(o["loss_replay"][1], total_py), (o["loss_replay"][1].item(), total_py.item())
    assert torch.equal(o["disp"], out_py[f"pred_disp_l/{s}"][:, 0].detach())
    assert torch.equal(fcs, feature_contrast_mean(out_py[f"cost_volume_l/{s + cfg['k']}"]))
    assert_same_model(fp, np_, fn, nn_)
    assert_same_optimizer(nat, stepper.optimizer)


@pytest.mark.gpu
def test_all_invalid_replay_gt():
  """A replay sample without one valid pixel: the Khamis term is 0 and the update still equals the Python step's."""
  cfg = ADAPT_ER["k3_96x256"]
  fp, np_ = nets(cfg)
  fn, nn_ = twin(fp, np_, cfg)
  stepper = python_stepper(fp, np_, True)
  nat = native.NativeAdapt(fn, nn_, lr=LR)
  samples = replay_samples(cfg, 2, seed=37)
  samples[1] = (samples[1][0], torch.zeros_like(samples[1][1]))
  for i, (img, (rimg, gt)) in enumerate(zip(frames(cfg, 2, seed=41), samples)):
    total_py = stepper.step(img[0], img[1], replay=(rimg[0], rimg[1], gt))[0]
    o = replay_outputs(cfg)
    nat.forward(img, o["loss"], replay=(rimg, gt), loss_replay=o["loss_replay"])
    nat.update()
    torch.cuda.synchronize()
    if i == 1:
      assert o["loss_replay"][0].item() == 0.0
    assert torch.equal(o["loss_replay"][1], total_py)
    assert_same_model(fp, np_, fn, nn_)
    assert_same_optimizer(nat, stepper.optimizer)


@pytest.mark.gpu
def test_replay_skip_update():
  """A frame whose update the host skips still runs both train-mode passes: BatchNorm statistics and counters move as in the
  Python grad-enabled forwards (stream pass first)."""
  cfg = ADAPT_ER["k3_96x256"]
  fp, np_ = nets(cfg)
  fn, nn_ = twin(fp, np_, cfg)
  stepper = python_stepper(fp, np_, True)
  nat = native.NativeAdapt(fn, nn_, lr=LR)
  for i, (img, (rimg, gt)) in enumerate(zip(frames(cfg, 3, seed=43), replay_samples(cfg, 3, seed=47))):
    o = replay_outputs(cfg)
    if i == 1:
      fp.train(); np_.train()
      stepper._refresh_weights()
      out = stepper.predict(img[0], img[1])                                     # grad enabled, no backward
      out_er = stepper.predict(rimg[0], rimg[1])
      loss_py, khamis_py = python_terms(cfg, img, rimg, gt, out, out_er)
      total_py = loss_py + ER_WEIGHT * khamis_py
      nat.forward(img, o["loss"], replay=(rimg, gt), loss_replay=o["loss_replay"])
    else:
      total_py = stepper.step(img[0], img[1], replay=(rimg[0], rimg[1], gt))[0]
      nat.forward(img, o["loss"], replay=(rimg, gt), loss_replay=o["loss_replay"])
      nat.update()
    torch.cuda.synchronize()
    assert torch.equal(o["loss_replay"][1], total_py.detach())
    assert_same_model(fp, np_, fn, nn_)
    assert_same_optimizer(nat, stepper.optimizer)
  counts = {n: int(v) for n, v in list(fn.state_dict().items()) + list(nn_.state_dict().items()) if n.endswith("num_batches_tracked")}
  fnames = {n for n in fn.state_dict() if n.endswith("num_batches_tracked")}
  for n, v in counts.items():
    assert v == (0 if ".conv2." in n else (12 if n in fnames else 6)), (n, v)  # three frames: 4 and 2 per frame


@pytest.mark.gpu
def test_replay_step_vs_reference_golden():
  """Independent of the Python path: the native ER step against the reference's own (tests/golden/rows_f3_f4.npz, er/*), with the
  inputs and bands of tests/test_gpu_adapt_rows.py::test_replay_step_vs_reference_golden."""
  import os
  import stereonet_b200 as S
  gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rows_f3_f4.npz"))
  H, W = 96, 256
  f = S.FeatureExtractorNetwork(3).to(DEV); s = S.StereoNet(3, 1, 0).to(DEV)
  f.load_state_dict(O.make_feature_state(3, 11)); s.load_state_dict(O.make_stereo_state(22, sharpen=10.0))
  l, r, _ = O.make_stereo_pair(1, H, W, seed=1000, max_disp_px=40.0)
  rl, rr, rgt = O.make_stereo_pair(1, H, W, seed=1001, max_disp_px=40.0)
  nat = native.NativeAdapt(f, s, lr=5e-5, clip_norm=1.0)
  loss = torch.empty((2,), device=DEV)
  loss_replay = torch.empty((2,), device=DEV)
  nat.forward(torch.stack([l, r]).to(DEV).contiguous(), loss, replay=(torch.stack([rl, rr]).to(DEV).contiguous(), rgt.to(DEV)),
              loss_replay=loss_replay, er_weight=0.05)
  nat.update()
  torch.cuda.synchronize()
  assert abs(loss[0].item() - float(gold["er/loss_mono"])) < 2e-5
  assert abs(loss_replay[0].item() - float(gold["er/loss_replay"])) < 2e-4 * float(gold["er/loss_replay"])
  n_clip = sum(p.numel() for n, p in s.named_parameters() if ".conv2." not in n)     # the bucket's stereo_net slots
  gn = math.sqrt(float((nat.flat_grad[:n_clip].double() ** 2).sum().item()))
  assert abs(gn - float(gold["er/grad_norm_stereo"])) <= 1.5e-2 * float(gold["er/grad_norm_stereo"]), gn
  for key in gold.files:
    if key.startswith("er/post/") and ("running_" in key or "num_batches" in key):
      _, _, tag, n = key.split("/", 3)
      v = (s if tag == "s" else f).state_dict()[n].cpu().numpy()
      if "num_batches" in key:
        assert int(v) == int(gold[key]) == (0 if ".conv2." in n else (2 if tag == "s" else 4)), key
      else:
        assert np.abs(v - gold[key]).max() <= 1e-4 * max(1.0, np.abs(gold[key]).max()), key
  d = np.abs(s.conv3d_alone.weight.detach().cpu().numpy() - gold["er/post/s/conv3d_alone.weight"])
  assert d.max() <= 2.1 * 5e-5 and (d <= 3e-6).mean() >= 0.97, (d.max(), (d <= 3e-6).mean())


@pytest.mark.gpu
def test_replay_graph_capture_matches_eager():
  cfg = ADAPT_ER["k3_rb2_96x256"]
  B, RB, H, W = cfg["B"], cfg["RB"], cfg["H"], cfg["W"]
  fe, ne = nets(cfg)
  fg, ng = twin(fe, ne, cfg)
  eager = native.NativeAdapt(fe, ne, lr=LR)
  graph = native.NativeAdapt(fg, ng, lr=LR)
  images = torch.empty((2, B, 3, H, W), device=DEV)
  rimages = torch.empty((2, RB, 3, H, W), device=DEV)
  gt = torch.empty((RB, H, W), device=DEV)
  og = replay_outputs(cfg)
  graph.workspace(B, H, W, RB)
  torch.cuda.synchronize()
  before = {k: v.clone() for k, v in list(fg.state_dict().items()) + list(ng.state_dict().items())}
  g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
  with torch.cuda.graph(g1):
    graph.forward(images, og["loss"], og["disp"], fcs_mean=og["fcs_mean"], replay=(rimages, gt), loss_replay=og["loss_replay"])
  with torch.cuda.graph(g2):
    graph.update()
  torch.cuda.synchronize()
  for k, v in list(fg.state_dict().items()) + list(ng.state_dict().items()):
    assert torch.equal(v, before[k]), k                          # capturing ran nothing
  for img, (rimg, g) in zip(frames(cfg, 3, seed=53), replay_samples(cfg, 3, seed=59)):
    images.copy_(img); rimages.copy_(rimg); gt.copy_(g)
    g1.replay(); g2.replay()
    oe = replay_outputs(cfg)
    eager.forward(img, oe["loss"], oe["disp"], fcs_mean=oe["fcs_mean"], replay=(rimg, g), loss_replay=oe["loss_replay"])
    eager.update()
    torch.cuda.synchronize()
    for key in oe:
      assert torch.equal(og[key], oe[key]), key
    assert_same_model(fe, ne, fg, ng)
    for a, b in ((graph.flat_grad, eager.flat_grad), (graph.exp_avg, eager.exp_avg), (graph.exp_avg_sq, eager.exp_avg_sq),
                 (graph.step_t, eager.step_t)):
      assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["k3_split_3x64", "k3_375x1242"])
def test_replay_writes_stay_inside_buffers(name):
  cfg = ADAPT_ER[name]
  B, RB, H, W, k = cfg["B"], cfg["RB"], cfg["H"], cfg["W"], cfg["k"]
  h, w = coarse_hw(cfg)
  lib = _cabi.lib()
  img = frames(cfg, 1, seed=61)[0]
  rimg, gt = replay_samples(cfg, 1, seed=67)[0]
  fr, nr = nets(cfg)
  ref = native.NativeAdapt(fr, nr, lr=LR)
  oref = dict(replay_outputs(cfg), fcs=torch.empty((B, h, w), device=DEV))
  ref.forward(img, oref["loss"], oref["disp"], oref["fcs"], oref["fcs_mean"], replay=(rimg, gt), loss_replay=oref["loss_replay"])
  ref.update()
  sizes = dict(loss=1 + B, loss_replay=2, disp=B * H * W, fcs=B * h * w, fcs_mean=1)
  nstate = lib.snb_stereonet_adapt_state_bytes(k) // 4
  nws = lib.snb_stereonet_adapt_replay_workspace_bytes(k, cfg["s"], 192, B, H, W, RB) // 4
  for optional in (True, False):
    f, n = nets(cfg)
    sbuf, state = banded(nstate)
    wbuf, ws = banded(nws)
    bufs = {key: banded(sz) for key, sz in sizes.items() if optional or key in ("loss", "loss_replay")}
    p = lambda key: bufs[key][1].data_ptr() if key in bufs else None
    params, st = native.param_pointers(f, n), stream_ptr()
    assert lib.snb_stereonet_adapt_init(params, k, state.data_ptr(), st) == 0
    assert lib.snb_stereonet_adapt_forward_replay(
        params, native.bn_counters(f, n), k, cfg["s"], 192, img.data_ptr(), B, H, W, rimg.data_ptr(), gt.data_ptr(), RB, ER_WEIGHT,
        state.data_ptr(), ws.data_ptr(), p("loss"), p("loss_replay"), p("disp"), p("fcs"), p("fcs_mean"), st) == 0, lib.snb_last_error()
    assert lib.snb_stereonet_adapt_update_replay(params, k, cfg["s"], 192, B, H, W, RB, state.data_ptr(), ws.data_ptr(), 1.0, LR, 0.9,
                                                 0.999, 1e-8, st) == 0, lib.snb_last_error()
    torch.cuda.synchronize()
    assert intact(sbuf, nstate), "state"
    assert intact(wbuf, nws), "workspace"
    for key, (buf, v) in bufs.items():
      assert intact(buf, sizes[key]), key
      assert torch.equal(v, oref[key].flatten()), key
    assert_same_model(fr, nr, f, n)


@pytest.mark.gpu
def test_replay_argument_errors_launch_nothing():
  cfg = ADAPT_ER["k3_96x256"]
  B, RB, H, W = cfg["B"], cfg["RB"], cfg["H"], cfg["W"]
  f, n = nets(cfg)
  nat = native.NativeAdapt(f, n, lr=LR)
  img = frames(cfg, 1)[0]
  rimg, gt = replay_samples(cfg, 1)[0]
  ws = nat.workspace(B, H, W, RB)
  lib = _cabi.lib()
  loss = torch.full((1 + B,), SENT, device=DEV)
  loss_replay = torch.full((2,), SENT, device=DEV)
  state_dict = lambda: {k: v.clone() for k, v in list(f.state_dict().items()) + list(n.state_dict().items())}
  before = state_dict()
  torch.cuda.synchronize()
  st = stream_ptr()

  def fwdr(rim=rimg.data_ptr(), g=gt.data_ptr(), rb=RB, er=ER_WEIGHT, lr=loss_replay.data_ptr()):
    return lib.snb_stereonet_adapt_forward_replay(nat.params, nat.counters, 3, 0, 192, img.data_ptr(), B, H, W, rim, g, rb, er,
                                                  nat.state.data_ptr(), ws.data_ptr(), loss.data_ptr(), lr, None, None, None, st)

  def fwd():
    return lib.snb_stereonet_adapt_forward(nat.params, nat.counters, 3, 0, 192, img.data_ptr(), B, H, W, nat.state.data_ptr(),
                                           ws.data_ptr(), loss.data_ptr(), None, None, None, st)

  def updr(rb=RB):
    return lib.snb_stereonet_adapt_update_replay(nat.params, 3, 0, 192, B, H, W, rb, nat.state.data_ptr(), ws.data_ptr(), 1.0, LR, 0.9,
                                                 0.999, 1e-8, st)

  def upd():
    return lib.snb_stereonet_adapt_update(nat.params, 3, 0, 192, B, H, W, nat.state.data_ptr(), ws.data_ptr(), 1.0, LR, 0.9, 0.999,
                                          1e-8, st)

  def rejected(cases):
    for call, word in cases:
      assert call() != 0, word
      msg = lib.snb_last_error().decode()
      assert f"`{word}`" in msg, (word, msg)

  rejected([
    (lambda: fwdr(rim=None), "replay_images"),
    (lambda: fwdr(rim=rimg.data_ptr() + 4), "replay_images"),
    (lambda: fwdr(g=None), "replay_gt"),
    (lambda: fwdr(rb=0), "RB"),
    (lambda: fwdr(er=-0.5), "er_weight"),
    (lambda: fwdr(er=float("nan")), "er_weight"),
    (lambda: fwdr(er=float("inf")), "er_weight"),
    (lambda: fwdr(lr=None), "loss_replay"),
  ])
  torch.cuda.synchronize()
  assert bool((loss == SENT).all().item()) and bool((loss_replay == SENT).all().item())     # nothing ran
  after = state_dict()
  for k, v in after.items():
    assert torch.equal(v, before[k]), k
  # an update must match its forward: a replay update takes the forward's RB, and each forward has its own update
  for forward, mismatched in ((fwdr, [(lambda: updr(rb=2), "RB"), (upd, "replay")]), (fwd, [(updr, "RB")])):
    assert forward() == 0
    torch.cuda.synchronize()
    after, grad0 = state_dict(), nat.flat_grad.clone()
    rejected(mismatched)
    torch.cuda.synchronize()
    assert torch.equal(nat.flat_grad, grad0)
    for k, v in state_dict().items():
      assert torch.equal(v, after[k]), k
  assert upd() == 0                                          # and the same calls, matched, do run
  assert fwdr() == 0 and updr() == 0
  torch.cuda.synchronize()
  o = replay_outputs(cfg)
  with pytest.raises(RuntimeError, match="loss_replay"):
    nat.forward(img, o["loss"], replay=(rimg, gt))           # the Python helper checks shapes, dtype and layout
  with pytest.raises(RuntimeError, match="replay_images"):
    nat.forward(img, o["loss"], replay=(rimg[:, :, :, :H - 1], gt), loss_replay=o["loss_replay"])
  with pytest.raises(RuntimeError, match="replay_gt"):
    nat.forward(img, o["loss"], replay=(rimg, gt[:, :, :W - 1]), loss_replay=o["loss_replay"])
  with pytest.raises(RuntimeError, match="replay_gt"):
    nat.forward(img, o["loss"], replay=(rimg, gt.double()), loss_replay=o["loss_replay"])


@pytest.mark.gpu
def test_example_host_replay_matches_native_api(tmp_path):
  """examples/stereonet_adapt.cpp with the replay arguments (no torch): frame f replays stored sample f % N; the weights file it
  writes equals the same frames and replay sequence through NativeAdapt from Python."""
  import importlib.util
  import os
  import subprocess
  from test_gpu_native import ROOT
  spec = importlib.util.spec_from_file_location("snb200_build", os.path.join(ROOT, "adaptive-stereo-icra-2021_b200", "build.py"))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  exe = mod.build_example(str(tmp_path / "stereonet_adapt"), "stereonet_adapt")
  cfg = ADAPT_ER["k3_b2_128x320"]
  B, RB, H, W, N, nframes = cfg["B"], cfg["RB"], cfg["H"], cfg["W"], 2, 3
  f, n = nets(cfg)
  native.export_weights(f, n, str(tmp_path / "w.bin"))
  imgs = frames(cfg, nframes, seed=71)
  samples = replay_samples(cfg, N, seed=73)
  torch.stack(imgs).cpu().numpy().astype("<f4").tofile(str(tmp_path / "img.bin"))
  torch.stack([s[0] for s in samples]).cpu().numpy().astype("<f4").tofile(str(tmp_path / "rimg.bin"))
  torch.stack([s[1] for s in samples]).cpu().numpy().astype("<f4").tofile(str(tmp_path / "rgt.bin"))
  args = [str(tmp_path / "w.bin"), str(tmp_path / "img.bin"), str(B), str(H), str(W), str(nframes), str(tmp_path / "out.bin"), "5e-5",
          str(tmp_path / "rimg.bin"), str(tmp_path / "rgt.bin"), str(RB), str(N)]
  r = subprocess.run([exe] + args, capture_output=True, text=True, timeout=300)
  assert r.returncode == 0, r.stdout + r.stderr
  assert r.stdout.count("khamis") == nframes and r.stdout.count("total") == nframes, r.stdout
  nat = native.NativeAdapt(f, n, lr=LR)
  for i, img in enumerate(imgs):
    rimg, gt = samples[i % N]
    nat.forward(img, outputs(cfg)["loss"], replay=(rimg, gt), loss_replay=torch.empty((2,), device=DEV), er_weight=ER_WEIGHT)
    nat.update()
  torch.cuda.synchronize()
  native.export_weights(f, n, str(tmp_path / "ref.bin"))
  assert (tmp_path / "out.bin").read_bytes() == (tmp_path / "ref.bin").read_bytes()
