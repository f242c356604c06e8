"""Shared-model data-parallel adaptation through the C-ABI (snb_stereonet_adapt_backward[_replay] + the host's all-reduce of the
state's dp_flat piece + snb_stereonet_adapt_apply, csrc/adapt.cu): the state layout around the all-reduce span (CPU); backward +
apply(1) bit-identical to the update; two replicas on one GPU, summed by hand as a two-rank NCCL SUM would, against
optim.FusedAdamClip; two NCCL ranks against AdaptStepper(..., dp_bucket=parallel.DPBucket(...)); the torch-free multi-GPU host
examples/stereonet_adapt_dp.cpp; argument errors and guard bands."""
import ctypes as C
import os
import subprocess
import sys

import pytest
import torch

import stereonet_b200 as S
from stereonet_b200 import _cabi, native, parallel
from stereonet_b200.optim import FusedAdamClip
from test_gpu_native import DEV, ROOT, banded, intact, stream_ptr
from test_gpu_native_adapt import LR, assert_same_model, assert_same_optimizer, frames, nets, outputs, twin
from test_gpu_native_adapt_replay import ER_WEIGHT, replay_outputs, replay_samples

N_STATS = 17 * 2 * 32
KITTI = dict(k=3, s=0, B=1, RB=1, H=376, W=1248)
SMALL = dict(k=3, s=0, B=1, RB=1, H=96, W=256)


def piece(k, what):
  o, nb = C.c_longlong(), C.c_longlong()
  assert _cabi.lib().snb_stereonet_adapt_state_piece(k, what, C.byref(o), C.byref(nb)) == 0, _cabi.lib().snb_last_error()
  return o.value, nb.value


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("k", [3, 4])
def test_dp_span_layout(k):
  """Piece 4 (running statistics) sits right after the bucket, piece 5 covers both: DPBucket.flat's layout and size."""
  with torch.device("meta"):
    f, s = S.FeatureExtractorNetwork(k), S.StereoNet(k, 1, 0)
  n_total = sum(p.numel() for p in parallel.used_parameters(s, f))
  assert sum(b.numel() for b in parallel.used_bn_buffers(s, f)) == N_STATS
  (g0, gb), (s0, sb), (d0, db) = piece(k, 0), piece(k, 4), piece(k, 5)
  assert gb == 4 * n_total
  assert (s0, sb) == (g0 + 4 * n_total, 4 * N_STATS)
  assert (d0, db) == (g0, 4 * (n_total + N_STATS))
  if k == 3:
    assert n_total + N_STATS == 289154
  offs = [piece(k, what) for what in range(4)]                # pieces 0-3: aligned, in order, after the span
  assert all(o % 256 == 0 for o, _ in offs)
  assert offs[1][0] >= d0 + db
  assert all(a[0] + a[1] <= b[0] for a, b in zip(offs, offs[1:]))
  assert offs[-1][0] + offs[-1][1] <= _cabi.lib().snb_stereonet_adapt_state_bytes(k)
  o, nb = C.c_longlong(), C.c_longlong()
  assert _cabi.lib().snb_stereonet_adapt_state_piece(k, 6, C.byref(o), C.byref(nb)) != 0
  assert b"`what`" in _cabi.lib().snb_last_error()


# ---------------------------------------------------------------------------------------------------------------- helpers
def stats_of(f, n):
  return torch.cat([b.detach().reshape(-1) for b in parallel.used_bn_buffers(n, f)])


def forward(nat, cfg, img, sample):
  if sample is None:
    nat.forward(img, outputs(cfg)["loss"])
  else:
    nat.forward(img, outputs(cfg)["loss"], replay=sample, loss_replay=torch.empty((2,), device=DEV), er_weight=ER_WEIGHT)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("replay", [False, True])
def test_world_one_equals_update(replay):
  """forward -> backward -> apply(1) leaves what forward -> update leaves: parameters, running statistics, counters, bucket,
  moments and step; backward's statistics piece is the running statistics in used_bn_buffers order."""
  cfg = KITTI
  fu, nu = nets(cfg)
  fd, nd = twin(fu, nu, cfg)
  upd = native.NativeAdapt(fu, nu, lr=LR)
  dp = native.NativeAdapt(fd, nd, lr=LR)
  samples = replay_samples(cfg, 3, seed=83) if replay else [None] * 3
  for img, sample in zip(frames(cfg, 3, seed=79), samples):
    forward(upd, cfg, img, sample)
    upd.update()
    forward(dp, cfg, img, sample)
    dp.backward()
    torch.cuda.synchronize()
    assert torch.equal(dp.bn_stats, stats_of(fd, nd))
    dp.apply(1)
    torch.cuda.synchronize()
    assert_same_model(fu, nu, fd, nd)
    for a, b in ((upd.flat_grad, dp.flat_grad), (upd.exp_avg, dp.exp_avg), (upd.exp_avg_sq, dp.exp_avg_sq), (upd.step_t, dp.step_t)):
      assert torch.equal(a, b)


@pytest.mark.gpu
def test_two_replicas_on_one_gpu():
  """Two replicas, their own frames and replay samples; dp_flat = a + b on both (a two-rank NCCL SUM), then apply(2): identical
  replicas, equal to FusedAdamClip.step(grad_scale=0.5) on the summed bucket with the statistics fl(sum * 0.5)."""
  cfg = dict(SMALL, B=2, H=128, W=320)
  fa, na = nets(cfg)
  fb, nb = twin(fa, na, cfg)
  a = native.NativeAdapt(fa, na, lr=LR)
  b = native.NativeAdapt(fb, nb, lr=LR)
  for step in range(2):
    for nat, seed in ((a, 89), (b, 97)):
      img = frames(cfg, 1, seed=seed + step)[0]
      forward(nat, cfg, img, replay_samples(cfg, 1, seed=seed + 50 + step)[0])
      nat.backward()
    torch.cuda.synchronize()
    # the reference: replica a's modules and Adam state as they stand before the apply, one FusedAdamClip step on the sum
    fr, nr = twin(fa, na, cfg)
    opt = FusedAdamClip(nr, fr, lr=LR)
    a.to_fused(opt)
    total = a.dp_flat + b.dp_flat
    a.dp_flat.copy_(total)
    b.dp_flat.copy_(total)
    n = opt.n_total
    with torch.no_grad():
      opt.flat_grad.copy_(total[:n])
      stats = total[n:].clone()
      stats.mul_(1.0 / 2)
      off = 0
      for buf in parallel.used_bn_buffers(nr, fr):
        buf.copy_(stats[off:off + buf.numel()].view_as(buf))
        off += buf.numel()
    opt.step(grad_scale=0.5, packed=True)
    a.apply(2)
    b.apply(2)
    torch.cuda.synchronize()
    assert_same_model(fa, na, fb, nb)
    assert_same_model(fa, na, fr, nr)
    assert_same_optimizer(a, opt)
    for x, y in ((a.exp_avg, b.exp_avg), (a.exp_avg_sq, b.exp_avg_sq), (a.step_t, b.step_t)):
      assert torch.equal(x, y)


DP_SNIPPET = r'''
import os, sys
import torch, torch.distributed as dist
ROOT = sys.argv[1]
for p in (ROOT, os.path.join(ROOT, "adaptive-stereo-icra-2021_b200"), os.path.join(ROOT, "oracle")):
  sys.path.insert(0, p)
import stereonet_oracle as O
import stereonet_b200 as S
from stereonet_b200 import native, parallel
from stereonet_b200.adapt import AdaptStepper, make_optimizer
LR = 5e-5
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
cfg = dict(k=3, s=0, B=1, RB=1, H=96, W=256)
g = torch.Generator(device=dev).manual_seed(101 + rank)        # a different stream and replay sample per rank
steps = []
for i in range(3):
  img = torch.rand((2, 1, 3, cfg["H"], cfg["W"]), device=dev, generator=g)
  rimg = torch.rand((2, 1, 3, cfg["H"], cfg["W"]), device=dev, generator=g)
  gt = torch.rand((1, cfg["H"], cfg["W"]), device=dev, generator=g) * 40.0 + 0.5
  steps.append((img, rimg, gt))
models = {}
for name in ("native", "python"):
  f, s = S.FeatureExtractorNetwork(3).to(dev), S.StereoNet(3, 1, 0, maxdisp=192).to(dev)
  f.load_state_dict(O.make_feature_state(3, 11)); s.load_state_dict(O.make_stereo_state(22, sharpen=40.0))
  models[name] = (f, s)
f, s = models["native"]
nat = native.NativeAdapt(f, s, lr=LR)
for img, rimg, gt in steps:
  nat.forward(img, torch.empty((2,), device=dev), replay=(rimg, gt), loss_replay=torch.empty((2,), device=dev), er_weight=0.05)
  nat.update(dp_group=dist.group.WORLD)
f, s = models["python"]
opt = make_optimizer(f, s, lr=LR, fused=True)
bucket = parallel.DPBucket(opt, s, f)
st = AdaptStepper(f, s, opt, cfg["H"], cfg["W"])
for img, rimg, gt in steps:
  st.step(img[0], img[1], replay=(rimg[0], rimg[1], gt), dp_bucket=bucket)
torch.cuda.synchronize()
flat = lambda f, s: torch.cat([t.detach().double().reshape(-1) for net in (s, f) for t in net.state_dict().values()])
a, b = flat(*models["native"]), flat(*models["python"])
assert torch.equal(a, b), ("native != python", float((a - b).abs().max()))
assert torch.equal(nat.exp_avg, opt.exp_avg) and torch.equal(nat.exp_avg_sq, opt.exp_avg_sq) and torch.equal(nat.step_t, opt.step_t)
gathered = [torch.empty_like(a) for _ in range(world)]
dist.all_gather(gathered, a)
for x in gathered[1:]:
  assert torch.equal(x, gathered[0]), ("replicas diverged", float((x - gathered[0]).abs().max()))
assert models["native"][1].filter[0][0][1].num_batches_tracked.item() == 6
dist.barrier()
dist.destroy_process_group()
if rank == 0:
  print("NATIVE_DP_OK")
'''


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_match_python_dp_step():
  """Two NCCL ranks, three replay steps each: NativeAdapt.update(dp_group=...) against AdaptStepper(..., dp_bucket=...) on the same
  frames; identical replicas, native equal to Python bit for bit."""
  env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29573", WORLD_SIZE="2")
  procs = [subprocess.Popen([sys.executable, "-c", DP_SNIPPET, ROOT], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                            stderr=subprocess.STDOUT, text=True) for r in range(2)]
  outs = []
  try:
    for p in procs:
      outs.append(p.communicate(timeout=600)[0])
  finally:
    for p in procs:
      if p.poll() is None:
        p.kill()
        p.wait()
  assert all(p.returncode == 0 for p in procs), "\n".join(o[-3000:] for o in outs)
  assert "NATIVE_DP_OK" in outs[0]


def build_example(tmp_path, name):
  import importlib.util
  spec = importlib.util.spec_from_file_location("snb200_build", os.path.join(ROOT, "adaptive-stereo-icra-2021_b200", "build.py"))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  return mod.build_example(str(tmp_path / name), name)


@pytest.mark.gpu
@pytest.mark.parametrize("replay", [False, True])
def test_example_host_one_gpu_matches_single_host(tmp_path, replay):
  """examples/stereonet_adapt_dp.cpp with G = 1 writes the weights file examples/stereonet_adapt.cpp writes on the same frames."""
  single, dp = build_example(tmp_path, "stereonet_adapt"), build_example(tmp_path, "stereonet_adapt_dp")
  cfg = dict(SMALL, B=2, H=128, W=320)
  B, H, W, N, nframes = cfg["B"], cfg["H"], cfg["W"], 2, 3
  native.export_weights(*nets(cfg), str(tmp_path / "w.bin"))
  torch.stack(frames(cfg, nframes, seed=103)).cpu().numpy().astype("<f4").tofile(str(tmp_path / "img.bin"))
  args = [str(tmp_path / "w.bin"), str(tmp_path / "img.bin"), str(B), str(H), str(W), str(nframes)]
  tail = []
  if replay:
    samples = replay_samples(cfg, N, seed=107)
    torch.stack([s[0] for s in samples]).cpu().numpy().astype("<f4").tofile(str(tmp_path / "rimg.bin"))
    torch.stack([s[1] for s in samples]).cpu().numpy().astype("<f4").tofile(str(tmp_path / "rgt.bin"))
    tail = ["5e-5", str(tmp_path / "rimg.bin"), str(tmp_path / "rgt.bin"), str(cfg["RB"]), str(N)]
  r1 = subprocess.run([single] + args + [str(tmp_path / "single.bin")] + tail, capture_output=True, text=True, timeout=300)
  assert r1.returncode == 0, r1.stdout + r1.stderr
  r2 = subprocess.run([dp, "1"] + args + [str(tmp_path / "dp.bin")] + tail, capture_output=True, text=True, timeout=300)
  assert r2.returncode == 0, r2.stdout + r2.stderr
  assert "1 replicas identical" in r2.stdout and "us per step" in r2.stdout, r2.stdout
  assert r2.stdout.count("rank 0 loss") == nframes, r2.stdout
  assert (tmp_path / "dp.bin").read_bytes() == (tmp_path / "single.bin").read_bytes()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_example_host_two_gpus_identical_replicas(tmp_path):
  dp = build_example(tmp_path, "stereonet_adapt_dp")
  cfg = dict(SMALL)
  B, H, W, G = cfg["B"], cfg["H"], cfg["W"], 2
  native.export_weights(*nets(cfg), str(tmp_path / "w.bin"))
  torch.stack(frames(cfg, 2 * G, seed=109)).cpu().numpy().astype("<f4").tofile(str(tmp_path / "img.bin"))   # [2][G][2][B][3][H][W]
  samples = replay_samples(cfg, 3, seed=113)
  torch.stack([s[0] for s in samples]).cpu().numpy().astype("<f4").tofile(str(tmp_path / "rimg.bin"))
  torch.stack([s[1] for s in samples]).cpu().numpy().astype("<f4").tofile(str(tmp_path / "rgt.bin"))
  r = subprocess.run([dp, str(G), str(tmp_path / "w.bin"), str(tmp_path / "img.bin"), str(B), str(H), str(W), "3", str(tmp_path / "o.bin"),
                      "5e-5", str(tmp_path / "rimg.bin"), str(tmp_path / "rgt.bin"), "1", "3"], capture_output=True, text=True, timeout=600)
  assert r.returncode == 0, r.stdout + r.stderr
  assert f"{G} replicas identical" in r.stdout, r.stdout


@pytest.mark.gpu
def test_argument_errors_launch_nothing():
  cfg = SMALL
  B, RB, H, W = cfg["B"], cfg["RB"], cfg["H"], cfg["W"]
  f, n = nets(cfg)
  nat = native.NativeAdapt(f, n, lr=LR)
  img = frames(cfg, 1, seed=127)[0]
  rimg, gt = replay_samples(cfg, 1, seed=131)[0]
  lib, st = _cabi.lib(), stream_ptr()
  ws, wsr = nat.workspace(B, H, W), nat.workspace(B, H, W, RB)
  state_dict = lambda: {k: v.clone() for k, v in list(f.state_dict().items()) + list(n.state_dict().items())}

  def bwd(wsp=ws.data_ptr()):
    return lib.snb_stereonet_adapt_backward(nat.params, 3, 0, 192, B, H, W, nat.state.data_ptr(), wsp, st)

  def bwdr(rb=RB, wsp=wsr.data_ptr()):
    return lib.snb_stereonet_adapt_backward_replay(nat.params, 3, 0, 192, B, H, W, rb, nat.state.data_ptr(), wsp, st)

  def apply(world=1, params=nat.params):
    return lib.snb_stereonet_adapt_apply(params, 3, nat.state.data_ptr(), world, 1.0, LR, 0.9, 0.999, 1e-8, st)

  def fwd(wsp=ws.data_ptr()):
    return lib.snb_stereonet_adapt_forward(nat.params, nat.counters, 3, 0, 192, img.data_ptr(), B, H, W, nat.state.data_ptr(), wsp,
                                           outputs(cfg)["loss"].data_ptr(), None, None, None, st)

  def fwdr():
    o = replay_outputs(cfg)
    return lib.snb_stereonet_adapt_forward_replay(nat.params, nat.counters, 3, 0, 192, img.data_ptr(), B, H, W, rimg.data_ptr(),
                                                  gt.data_ptr(), RB, ER_WEIGHT, nat.state.data_ptr(), wsr.data_ptr(), o["loss"].data_ptr(),
                                                  o["loss_replay"].data_ptr(), None, None, None, st)

  def rejected(cases):
    torch.cuda.synchronize()
    before, span = state_dict(), nat.dp_flat.clone()
    for call, word in cases:
      assert call() != 0, word
      msg = lib.snb_last_error().decode()
      assert f"`{word}`" in msg, (word, msg)
    torch.cuda.synchronize()
    assert torch.equal(nat.dp_flat, span)                   # nothing ran
    for k, v in state_dict().items():
      assert torch.equal(v, before[k]), k

  alt = native.param_pointers(f, n)
  alt[5] = alt[6]
  # no forward on this address (the records are keyed by address, and torch's allocator hands out 512-byte aligned blocks that an
  # earlier test's workspace may have held)
  rejected([(lambda: bwd(wsp=ws.data_ptr() + 256), "workspace"), (lambda: bwdr(wsp=wsr.data_ptr() + 256), "workspace")])
  assert fwdr() == 0
  rejected([(lambda: bwd(wsp=wsr.data_ptr()), "replay"), (lambda: bwdr(rb=2), "RB")])
  assert bwdr() == 0
  rejected([(lambda: apply(world=0), "world"), (lambda: apply(params=alt), "params[5]")])
  assert apply() == 0
  rejected([(lambda: apply(), "state")])                     # applied: no backward since
  assert fwd() == 0
  rejected([(lambda: bwdr(wsp=ws.data_ptr()), "RB")])
  assert bwd() == 0
  assert lib.snb_stereonet_adapt_update(nat.params, 3, 0, 192, B, H, W, nat.state.data_ptr(), ws.data_ptr(), 1.0, LR, 0.9, 0.999, 1e-8,
                                        st) == 0                # an update consumes the bucket too
  rejected([(lambda: apply(), "state")])
  with pytest.raises(RuntimeError, match="forward"):
    native.NativeAdapt(*twin(f, n, cfg), lr=LR).backward()


@pytest.mark.gpu
@pytest.mark.parametrize("replay", [False, True])
def test_backward_apply_write_inside_buffers(replay):
  cfg = dict(SMALL, H=375, W=1242)
  B, RB, H, W, k = cfg["B"], cfg["RB"], cfg["H"], cfg["W"], cfg["k"]
  lib = _cabi.lib()
  img = frames(cfg, 1, seed=137)[0]
  rimg, gt = replay_samples(cfg, 1, seed=139)[0]
  fr, nr = nets(cfg)
  ref = native.NativeAdapt(fr, nr, lr=LR)
  forward(ref, cfg, img, (rimg, gt) if replay else None)
  ref.update()
  nstate = lib.snb_stereonet_adapt_state_bytes(k) // 4
  nws = (lib.snb_stereonet_adapt_replay_workspace_bytes(k, 0, 192, B, H, W, RB) if replay
         else lib.snb_stereonet_adapt_workspace_bytes(k, 0, 192, B, H, W)) // 4
  f, n = nets(cfg)
  sbuf, state = banded(nstate)
  wbuf, ws = banded(nws)
  params, st = native.param_pointers(f, n), stream_ptr()
  loss, loss_replay = torch.empty((1 + B,), device=DEV), torch.empty((2,), device=DEV)
  assert lib.snb_stereonet_adapt_init(params, k, state.data_ptr(), st) == 0
  if replay:
    assert lib.snb_stereonet_adapt_forward_replay(
        params, native.bn_counters(f, n), k, 0, 192, img.data_ptr(), B, H, W, rimg.data_ptr(), gt.data_ptr(), RB, ER_WEIGHT,
        state.data_ptr(), ws.data_ptr(), loss.data_ptr(), loss_replay.data_ptr(), None, None, None, st) == 0, lib.snb_last_error()
    assert lib.snb_stereonet_adapt_backward_replay(params, k, 0, 192, B, H, W, RB, state.data_ptr(), ws.data_ptr(), st) == 0
  else:
    assert lib.snb_stereonet_adapt_forward(params, native.bn_counters(f, n), k, 0, 192, img.data_ptr(), B, H, W, state.data_ptr(),
                                           ws.data_ptr(), loss.data_ptr(), None, None, None, st) == 0, lib.snb_last_error()
    assert lib.snb_stereonet_adapt_backward(params, k, 0, 192, B, H, W, state.data_ptr(), ws.data_ptr(), st) == 0
  assert lib.snb_stereonet_adapt_apply(params, k, state.data_ptr(), 1, 1.0, LR, 0.9, 0.999, 1e-8, st) == 0, lib.snb_last_error()
  torch.cuda.synchronize()
  assert intact(sbuf, nstate), "state"
  assert intact(wbuf, nws), "workspace"
  assert_same_model(fr, nr, f, n)
