#!/usr/bin/env python
"""bench.py — StereoNet forward (BASELINE.json configs[1]: KITTI 376x1248, D=192, k=3, batch 1 per GPU) and the other
BASELINE.json configurations as extra keyed entries of the same JSON line.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    # the reference's own modules on the host CPU cores

A step = one pass of the hot path over one synthetic stereo pair per GPU: feature_net(L), feature_net(R),
stereo_net(L, fl, fr, 'l').  Prints ONE JSON line on rank 0 (contract in the task statement / DESIGN.md §6):

  value / ms_per_step   configs[1], device-resident inputs, CUDA-graph replay, CUDA events, max over ranks
  e2e                   configs[1] through StereoEngine.infer_host_async: pinned host images in, host disparity out, every step
  adapt                 configs[2] (N = 1: one stream) / configs[4] (N > 1: shared-model data parallel, one stream + one
                        reservoir-replay sample per rank and step, ONE NCCL all-reduce over [gradients | BN statistics])
  sceneflow_b32         configs[3]: 32 x 3 x 540 x 960 split over the ranks (strong scaling entry)
  timing_configs        configs[0] (T = 1x3x320x960 k=3) and the reference's own timing recipes (test/test_stereo_net.py,
                        evaluation/stereonet_timing.py): k=4 at 320x960, k=3 / input_scale 1 at 160x480, 320x1216 k=4 fwd and fwd+bwd
  roofline / kernels    per-kernel event timings with an L2 flush before every launch; DRAM traffic from the committed ncu capture
  cpu_baseline          the reference modules (oracle/_ref) — or the oracle port where they are absent — on the host cores

Every timed region runs exactly its number of steps (--steps for `value` and `e2e`); with --min-seconds S > 0 a region instead
grows until it lasts at least S seconds.  --dump-outputs DIR writes the outputs of the last step of the `value` region as
DIR/<name>.npy (float32, '/' in a name becomes '_'): seeded inputs and weights make two builds comparable output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "adaptive-stereo-icra-2021_b200")
for p in (ROOT, PKG):
  if p not in sys.path:
    sys.path.insert(0, p)

import torch  # noqa: E402

H, W, K_DOWN, MAXDISP = 376, 1248, 3, 192
METRIC = "StereoNet pairs/s @KITTI 376x1248 D=192"
WORKLOAD = "StereoNet k=3 D=192 fp32 forward, KITTI 1x3x376x1248 per GPU (BASELINE.json configs[1])"


def peaks():
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(path):
    d = json.load(open(path))
    return dict(hbm=d["hbm_gbs"], tensor=d["bf16_tflops"], tensor_sustained=d.get("bf16_tflops_sustained"), src="measured")
  return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, src="fallback")


# ------------------------------------------------------------------------------------------------- synthetic data
def synthetic_pair(seed, h=H, w=W, batch=1, slope=60.0):
  """Textured left image, ground-plane disparity ramp d(y) = 4 + slope * y / (h - 1), right = left warped by it (SURVEY.md §8d).
  Returns (left, right, gt_disp_l).  Plain torch on the host; no oracle import on the product path."""
  import torch.nn.functional as F
  g = torch.Generator().manual_seed(seed)
  noise = torch.randn((batch, 3, h, w), generator=g)
  low = F.avg_pool2d(F.avg_pool2d(noise, 9, 1, 4), 9, 1, 4) * 6.0
  left = (0.5 + 0.25 * low + 0.1 * torch.randn((batch, 3, h, w), generator=g)).clamp(0, 1)
  ramp = 4.0 + slope * torch.arange(h, dtype=torch.float32) / (h - 1)
  rows, cols = torch.meshgrid(torch.arange(h), torch.arange(w), indexing="ij")
  flow = torch.stack([cols, rows], dim=-1).float().expand(batch, -1, -1, -1).clone()
  flow[..., 0] = flow[..., 0] + ramp.view(1, h, 1)
  flow[..., 0] = (2 * flow[..., 0] / w) - 1.0
  flow[..., 1] = (2 * flow[..., 1] / h) - 1.0
  right = F.grid_sample(left, flow, mode="bilinear", padding_mode="border", align_corners=False)
  gt = ramp.view(1, 1, h, 1).expand(batch, 1, h, w).contiguous()
  return left.contiguous(), right.contiguous(), gt


# ------------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
  Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
      "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

  def __init__(self, index):
    self.index, self.rows, self.proc = index, [], None

  def start(self):
    try:
      self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits", "-lms", "25"], stdout=subprocess.PIPE, text=True)
      self.thread = threading.Thread(target=self._read, daemon=True)
      self.thread.start()
    except Exception:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append([c.strip() for c in line.split(",")])

  def stop(self):
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except Exception:
      self.proc.kill()
    sm, mx, reasons = [], None, set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for r in self.rows:
      try:
        sm.append(float(r[0])); mx = float(r[1])
        for n, v in zip(names, r[3:7]):
          if v.lower().startswith("active"):
            reasons.add(n)
      except Exception:
        pass
    sm.sort()
    # under load = upper half of the samples (the sampler also sees the idle gaps around the regions)
    med = sm[(len(sm) * 3) // 4] if sm else None
    return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------- reference arm (CPU)
def _host_cores():
  cores = os.cpu_count() or 1
  try:
    cores = len(os.sched_getaffinity(0))
  except Exception:
    pass
  return cores


def _oracle():
  sys.path.insert(0, os.path.join(ROOT, "oracle"))
  import stereonet_oracle as O
  import make_ref
  return O, make_ref.load()


def cpu_reference(steps, warmup, budget_s):
  """The reference's forward on the host cores, eval / no-grad, same shapes and seeded weights as the GPU arm; each step = one
  KITTI-sized pair.  kind = "reference": the unmodified modules vendored into oracle/_ref (stereo_net.py:54-207);
  kind = "port": the oracle's restatement, where oracle/_ref is absent."""
  O, ref = _oracle()
  cores = _host_cores()
  torch.set_num_threads(cores)
  fsd, ssd = O.make_feature_state(K_DOWN, 11), O.make_stereo_state(22, sharpen=40.0)
  left, right, _ = synthetic_pair(1000)
  if ref is not None:
    sn = ref[0]
    fnet, snet = sn.FeatureExtractorNetwork(K_DOWN), sn.StereoNet(K_DOWN, 1, 0, maxdisp=MAXDISP)
    fnet.load_state_dict(fsd); snet.load_state_dict(ssd)
    fnet.eval(); snet.eval()
    run = lambda: snet(left, fnet(left), fnet(right), "l", output_cost_volume=True)
    kind, what = "reference", "the unmodified reference modules (oracle/_ref: adaptive_stereo/models/stereo_net.py)"
  else:
    run = lambda: O.predict_disparity_left(fsd, ssd, left, right, K_DOWN)
    kind, what = "port", "the oracle port"
  done, t_total = 0, 0.0
  with torch.no_grad():
    for _ in range(warmup):
      run()
    t_begin = time.perf_counter()
    while done < steps:
      t0 = time.perf_counter()
      run()
      t_total += time.perf_counter() - t0
      done += 1
      if time.perf_counter() - t_begin > budget_s:
        break
  return dict(value=done / t_total, unit="pairs/s", cores=cores, kind=kind, steps=done, ms_per_step=1e3 * t_total / done,
              sample=f"{done} full forward passes of {what} (torch CPU fp32, {cores} threads) on one synthetic KITTI pair")


def cpu_reference_adapt(steps):
  """One adaptation step on the host cores (adapt.py:313-337,381-394): reference modules + their own Monodepth loss, clip, Adam."""
  O, ref = _oracle()
  cores = torch.get_num_threads()
  left, right, _ = synthetic_pair(1000)
  fsd0, ssd0 = O.make_feature_state(K_DOWN, 11), O.make_stereo_state(22, sharpen=10.0)
  if ref is not None:
    sn, lw, lf, _ = ref
    fnet, snet = sn.FeatureExtractorNetwork(K_DOWN), sn.StereoNet(K_DOWN, 1, 0, maxdisp=MAXDISP)
    fnet.load_state_dict(fsd0); snet.load_state_dict(ssd0)
    fnet.train(); snet.train()
    opt = torch.optim.Adam([{"params": snet.parameters()}, {"params": fnet.parameters()}], lr=5e-5)
    warper = lw.LinearWarping(H, W, torch.device("cpu"))

    def step():
      o = snet(left, fnet(left), fnet(right), "l", output_cost_volume=True)
      lw_img, mask = warper(right, o["pred_disp_l/0"], right_to_left=True)
      loss = lf.monodepth_loss(o["pred_disp_l/0"], left, lw_img, smoothness_weight=1e-3)[0][mask].mean()
      opt.zero_grad(); loss.backward()
      torch.nn.utils.clip_grad_norm_(snet.parameters(), 1.0)
      opt.step()
    kind = "reference"
  else:
    fsd, ssd, adam = O.clone_state(fsd0, True), O.clone_state(ssd0, True), {}
    step = lambda: O.adapt_step(fsd, ssd, left, right, K_DOWN, adam)
    kind = "port"
  step()
  t0 = time.perf_counter()
  for _ in range(steps):
    step()
  dt = (time.perf_counter() - t0) / steps
  return {"value": 1.0 / dt, "unit": "steps/s", "cores": cores, "kind": kind, "sample": f"{steps} adaptation steps ({kind})"}


# ------------------------------------------------------------------------------------------------- GPU arm
def time_kernel(fn, iters, flush, stream):
  """Average duration (ms) of fn() alone, L2 flushed before every launch, CUDA events on the launching stream."""
  evs = []
  for _ in range(3):
    fn()
  for _ in range(iters):
    flush.zero_()                       # > L2 (126 MB): evicts the kernel's inputs/outputs
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream); fn(); b.record(stream)
    evs.append((a, b))
  torch.cuda.synchronize()
  ts = sorted(a.elapsed_time(b) for a, b in evs)
  return sum(ts) / len(ts), ts[len(ts) // 2]


def dump_outputs(outputs, out_dir):
  """outputs: the dict of device tensors the forward returns (KITTI size: ~4.5 MB in all) -> out_dir/<name>.npy, float32."""
  import numpy as np
  os.makedirs(out_dir, exist_ok=True)
  for name, t in outputs.items():
    np.save(os.path.join(out_dir, name.replace("/", "_") + ".npy"), t.detach().float().cpu().numpy())


class Timer:
  """Timed regions of exactly `min_steps` steps, or with `min_seconds` > 0 of at least `min_steps` steps AND `min_seconds`: a probe of
  a few steps sizes the region (the step count is agreed over the ranks).  The region runs between a barrier + synchronize on both
  sides, CUDA events, max over ranks."""

  def __init__(self, dev, world, min_seconds):
    self.dev, self.world, self.min_seconds = dev, world, min_seconds
    self.stream = torch.cuda.current_stream(dev)

  def barrier(self):
    import torch.distributed as dist
    torch.cuda.synchronize()
    if self.world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def _max(self, v):
    import torch.distributed as dist
    t = torch.tensor([v], device=self.dev, dtype=torch.float64)
    if self.world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())

  def run(self, step, min_steps, warmup, finish=None, max_steps=200000):
    for _ in range(max(warmup, 3)):
      step()
    if finish:
      finish()
    steps = min_steps
    if self.min_seconds > 0:
      self.barrier()
      a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      a.record(self.stream)
      for _ in range(5):
        step()
      if finish:
        finish()
      b.record(self.stream)
      torch.cuda.synchronize()
      probe_ms = self._max(a.elapsed_time(b) / 5)
      steps = int(min(max_steps, max(min_steps, self.min_seconds * 1e3 / max(probe_ms, 1e-3) + 1)))
    for attempt in range(3):
      self.barrier()
      a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      a.record(self.stream)
      for _ in range(steps):
        step()
      if finish:
        finish()
      b.record(self.stream)
      self.barrier()
      ms = self._max(a.elapsed_time(b))               # the same number on every rank, so every rank takes the same decision
      if ms >= self.min_seconds * 1e3 or steps >= max_steps:
        break
      steps = int(min(max_steps, steps * self.min_seconds * 1e3 / max(ms, 1e-3) * 1.03 + 1))      # the probe over-estimated a step
    return steps, ms


def gpu_arm(args):
  import stereonet_b200 as S
  from stereonet_b200 import ops, parallel
  from stereonet_b200.autograd import fused
  from stereonet_b200.runtime import StereoEngine
  from stereonet_b200.adapt import AdaptStepper, make_optimizer
  from stereonet_b200.reservoir import ReplayReservoir
  import torch.distributed as dist

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  if world != args.gpus and world > 1:
    raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)
  tm = Timer(dev, world, args.min_seconds)
  stream = tm.stream

  def make_nets(k=K_DOWN, s=0):
    torch.manual_seed(123)                                   # the reference's seed (adapt.py:29, train.py:141)
    return S.FeatureExtractorNetwork(k).to(dev), S.StereoNet(k, 1, s, maxdisp=MAXDISP).to(dev)

  fnet, snet = make_nets()
  fnet.eval(); snet.eval()
  engine = StereoEngine(fnet, snet, output_cost_volume=True, use_graph=not args.no_graph)

  left, right, _ = synthetic_pair(1000 + rank)
  shape = tuple(left.shape)
  left_pin, right_pin = left.pin_memory(), right.pin_memory()
  out_pin = torch.empty((1, 1, H, W), dtype=torch.float32).pin_memory()
  e = engine._entry(shape, dev)
  e["left"].copy_(left_pin); e["right"].copy_(right_pin)
  launches = engine.run_static(shape, dev)[1]

  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()

  # ---- configs[1], device-resident throughput: inputs already in HBM, graph replays
  last = {}

  def step_dev():
    last["out"] = engine.run_static(shape, dev)[0]
  steps_dev, ms_dev = tm.run(step_dev, args.steps, args.warmup)
  if args.dump_outputs and rank == 0:
    dump_outputs(last["out"], args.dump_outputs)          # what the last timed step returned

  # ---- configs[1], end to end through the public engine API: pinned host images in, host disparity out, every step
  # (a) streaming API: H2D of frame i+1 / forward of frame i / D2H of frame i-1 overlap (throughput = the headline e2e);
  # (b) blocking API: the three phases of one frame back to back (latency).
  steps_e2e, ms_e2e = tm.run(lambda: engine.infer_host_async(left_pin, right_pin, out_pin), args.steps, args.warmup, finish=engine.synchronize)
  steps_seq, ms_seq = tm.run(lambda: engine.infer_host(left_pin, right_pin, out_pin), max(args.steps // 2, 10), 3)

  # ---- configs[3]: SceneFlow-shaped batch 32 x 3 x 540 x 960 split over the ranks (strong scaling), eval forward, CUDA graph
  sf = None
  if not args.skip_sceneflow:
    lo, hi = parallel.shard_range(32, rank, world)
    nb = hi - lo
    pairs = [synthetic_pair(3000 + lo + i, 540, 960)[:2] for i in range(min(nb, 2))]          # 2 distinct samples, tiled over the shard
    sl = torch.cat([pairs[i % len(pairs)][0] for i in range(nb)]).to(dev)
    sr = torch.cat([pairs[i % len(pairs)][1] for i in range(nb)]).to(dev)
    eng_sf = StereoEngine(fnet, snet, output_cost_volume=False, use_graph=not args.no_graph)
    es = eng_sf._entry(tuple(sl.shape), dev)
    es["left"].copy_(sl); es["right"].copy_(sr)
    steps_sf, ms_sf = tm.run(lambda: eng_sf.run_static(tuple(sl.shape), dev), 5, 3)
    sf = {"metric": "StereoNet pairs/s @SceneFlow 540x960 D=192, global batch 32 (BASELINE.json configs[3])",
          "value": 32 * steps_sf / (ms_sf / 1e3), "unit": "pairs/s", "ms_per_batch": ms_sf / steps_sf, "steps": steps_sf,
          "pairs_per_gpu": nb, "scaling": "strong", "parallelism": f"batch 32 sharded {world}-way, no collective"}
    del eng_sf, es, sl, sr
    torch.cuda.empty_cache()

  # ---- online-adaptation step: train-mode fwd + photometric loss + bwd + clip + Adam, all in libsnb200 kernels.
  # N = 1 -> configs[2] (one stream).  N > 1 -> configs[4]: shared-model data parallel, one stream per rank, one replay sample per
  # rank and step drawn from the rank's reservoir, ONE NCCL all-reduce per step over [gradients | BN running statistics].
  adapt = None
  if not args.skip_adapt:
    fa, sa = make_nets()
    fa.train(); sa.train()
    opt = make_optimizer(fa, sa, lr=5e-5, fused=True)
    bucket = parallel.DPBucket(opt, sa, fa) if world > 1 else None
    stepper = AdaptStepper(fa, sa, opt, H, W, clip_grad_norm=True, use_graph=not args.no_graph, two_streams=not args.adapt_single_stream)
    frames = [tuple(t.to(dev) for t in synthetic_pair(1000 + 100 * rank + i, slope=60.0 - 2.0 * i)) for i in range(4)]   # a drifting ramp
    it = [0]
    if world > 1:
      res = ReplayReservoir(8, seed=rank)
      for i in range(8):
        l_, r_, g_ = synthetic_pair(7000 + 100 * rank + i, slope=30.0 + 3.0 * i)
        res.add(l_.to(dev), r_.to(dev), g_.to(dev), i)

      def step_adapt():
        l_, r_, _ = frames[it[0] % len(frames)]; it[0] += 1
        stepper.step(l_, r_, replay=res.sample(), dp_bucket=bucket)
    else:
      def step_adapt():
        l_, r_, _ = frames[it[0] % len(frames)]; it[0] += 1
        stepper.step(l_, r_)
    n0 = ops.LAUNCHES
    steps_ad, ms_ad = tm.run(step_adapt, max(50, args.steps // 2), 3)
    adapt = {"metric": "online adaptation steps/s @KITTI 376x1248 (train-mode fwd + Monodepth loss + bwd + clip + Adam lr 5e-5)"
                       + (" — BASELINE.json configs[2]" if world == 1 else " with one reservoir-replay pass per step — BASELINE.json configs[4]"),
             "value": world * steps_ad / (ms_ad / 1e3), "unit": "steps/s", "ms_per_step": ms_ad / steps_ad, "steps": steps_ad,
             "library_launches_per_step": stepper.launches_per_step or (ops.LAUNCHES - n0) // max(it[0], 1),
             "cuda_graph": not args.no_graph,
             "parallelism": "single stream" if world == 1 else
                            f"shared-model DP x{world}: one stream + one replay sample per rank, one NCCL all-reduce of "
                            f"{bucket.flat.numel()} floats (gradients of the used parameters + BN running statistics) per step",
             "optimizer": "optim.FusedAdamClip (snb_multi_gather + snb_adam_clip_step: clip on the stereo_net group + Adam, 5 launches)"}
    # N = 1: also the ER step (two passes per update) so the single-GPU line has the configs[4] workload per rank
    if world == 1:
      res = ReplayReservoir(8, seed=0)
      for i in range(8):
        l_, r_, g_ = synthetic_pair(7000 + i, slope=30.0 + 3.0 * i)
        res.add(l_.to(dev), r_.to(dev), g_.to(dev), i)

      def step_er():
        l_, r_, _ = frames[it[0] % len(frames)]; it[0] += 1
        stepper.step(l_, r_, replay=res.sample())
      steps_er, ms_er = tm.run(step_er, 30, 3)
      adapt["with_replay"] = {"value": steps_er / (ms_er / 1e3), "unit": "steps/s", "ms_per_step": ms_er / steps_er, "steps": steps_er,
                              "note": "adapt.py:339-349: a second full train-mode pass on a reservoir sample + Khamis loss, per update"}
    del stepper, opt, fa, sa
    torch.cuda.empty_cache()

  clocks = sampler.stop() if rank == 0 else None          # sampled across the timed regions above

  result = None
  if rank == 0:
    pk = peaks()
    # ---- the reference's own test / timing configurations (rank 0; single-GPU recipes): graph-replayed forward, and fwd + bwd + Adam
    timing = {}
    if world == 1 and not args.skip_timing_configs:
      t1 = Timer(dev, 1, min(args.min_seconds, 1.0))
      for name, (k, s, h, w) in {"T_320x960_k3 (configs[0], test_stereo_net.py:17-22)": (3, 0, 320, 960),
                                 "k4_320x960 (test_stereo_net.py:46-53, experiments/adaptation/*.sh)": (4, 0, 320, 960),
                                 "k3_s1_160x480 (test_stereo_net.py:55-62)": (3, 1, 160, 480),
                                 "k4_320x1216 (stereonet_timing.py:22-41)": (4, 0, 320, 1216)}.items():
        fk, sk = make_nets(k, s)
        fk.eval(); sk.eval()
        eng = StereoEngine(fk, sk, output_cost_volume=False, use_graph=not args.no_graph)
        l_, r_, _ = synthetic_pair(11, h, w)
        en = eng._entry(tuple(l_.shape), dev)
        en["left"].copy_(l_); en["right"].copy_(r_)
        n_, ms_ = t1.run(lambda: eng.run_static(tuple(l_.shape), dev), 20, 3)
        timing[name] = {"forward_ms": ms_ / n_, "pairs_per_s": n_ / (ms_ / 1e3), "steps": n_}
      fk, sk = make_nets(4, 0)
      fk.train(); sk.train()
      stp = AdaptStepper(fk, sk, make_optimizer(fk, sk, lr=1e-4, fused=True), 320, 1216, clip_grad_norm=False, use_graph=not args.no_graph)
      l_, r_, _ = synthetic_pair(12, 320, 1216)
      l_, r_ = l_.to(dev), r_.to(dev)
      n_, ms_ = t1.run(lambda: stp.step(l_, r_), 20, 3)
      timing["k4_320x1216 fwd+bwd+Adam lr 1e-4 (stereonet_timing.py:44-72)"] = {"step_ms": ms_ / n_, "steps_per_s": n_ / (ms_ / 1e3), "steps": n_}
      del stp, fk, sk, eng
      torch.cuda.empty_cache()

    # ---- per-kernel roofline numbers, each kernel timed alone with an L2 flush before every launch
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev, dtype=torch.float32)
    hc, wc, D = (H - 1) // 8 + 1, (W - 1) // 8 + 1, (MAXDISP + 1) // 8
    with torch.no_grad():
      fl = torch.randn(1, hc, wc, 32, device=dev); fr = torch.randn(1, hc, wc, 32, device=dev)
      cv_ms, _ = time_kernel(lambda: ops.cost_volume(fl, fr, D), 20, flush, stream)
      cv_bytes = 4 * 32 * hc * wc * (2 + D)
      # back to back over rotating outputs totalling > 2x L2: every launch writes memory no earlier launch left in L2 — the way
      # the kernel runs inside the forward (launch latency and the staging round trip overlap the previous launch's stores)
      nrot = 14
      outs = [torch.empty((1, D, hc, wc, 32), device=dev) for _ in range(nrot)]
      import ctypes as C
      from stereonet_b200 import _cabi
      def cv_rot(i):
        _cabi.check(_cabi.lib().snb_cost_volume_fwd(ops._p(fl), ops._p(fr), ops._p(outs[i % nrot]), 1, D, hc, wc, ops._stream(fl)), "cv")
      for i in range(nrot):
        cv_rot(i)
      torch.cuda.synchronize()
      ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      ea.record(stream)
      for i in range(8 * nrot):
        cv_rot(i)
      eb.record(stream)
      torch.cuda.synchronize()
      cvr_ms = ea.elapsed_time(eb) / (8 * nrot)
      del outs
      fl8 = torch.randn(8, hc, wc, 32, device=dev); fr8 = torch.randn(8, hc, wc, 32, device=dev)
      cv8_ms, _ = time_kernel(lambda: ops.cost_volume(fl8, fr8, D), 20, flush, stream)    # 195 MB > L2: fixed costs amortised
      x3 = torch.randn(1, D, hc, wc, 32, device=dev)
      conv3, bn3 = snet.filter[0][0][0], snet.filter[0][0][1]
      f3_ms, _ = time_kernel(lambda: fused.conv_bn_lrelu(x3, conv3, bn3, 1, False, False), 10, flush, stream)
      f3_flops = 2 * 27 * 32 * 32 * D * hc * wc
      x2 = torch.randn(1, H, W, 32, device=dev)
      blk = snet.edge_aware_refinements[0].residual_astrous_blocks[2]
      r2_ms, _ = time_kernel(lambda: blk.forward_cl(x2), 10, flush, stream)
      r2_flops = 2 * 9 * 32 * 32 * H * W
      hd_ms, _ = time_kernel(lambda: ops.conv3d_out_softargmin(x3, snet.conv3d_alone.weight, snet.conv3d_alone.bias, True, True), 20, flush, stream)
      hd_bytes = 4 * hc * wc * (32 * D + 1 + D + 1)
      tp_ms, _ = time_kernel(lambda: ops.conv_c32_taps(x3, snet.conv3d_alone.weight, 27), 20, flush, stream)
      taps27 = ops.conv_c32_taps(x3, snet.conv3d_alone.weight, 27)
      ts_ms, _ = time_kernel(lambda: ops.tapsum_softargmin(taps27, snet.conv3d_alone.bias, True), 20, flush, stream)
      tp_bytes, ts_bytes = 4 * hc * wc * D * (32 + 27), 4 * hc * wc * (27 * D + D + 1)
      img2 = torch.rand(2, 3, H, W, device=dev)
      c0 = fnet.downsample[0]
      fc_ms, _ = time_kernel(lambda: ops.conv5x5s2_c3(img2, c0.weight, c0.bias), 20, flush, stream)
      fc_flops = 2 * 2 * 75 * 32 * ((H - 1) // 2 + 1) * ((W - 1) // 2 + 1)
      ref = snet.edge_aware_refinements[0]
      cz = torch.rand(1, hc, wc, device=dev) * 20
      rconv = ref.conv2d_feature[0][0]
      ri_old_ms, _ = time_kernel(lambda: ops.refine_in_conv(cz, img2[:1], rconv.weight, rconv.bias.detach(), lrelu=True), 20, flush, stream)
      rwimg = ops.refine_in_weights_ws(rconv.weight)
      ri_ms, _ = time_kernel(lambda: ops.refine_in_conv_ws(cz, img2[:1], rwimg, rconv.bias.detach(), lrelu=True), 20, flush, stream)
      ri_bytes = 4 * H * W * (32 + 3 + 1)

    def hbm(ms, nbytes):
      return {"bound": "hbm", "ms": ms, "achieved": nbytes / ms / 1e6, "peak": pk["hbm"], "unit": "GB/s", "frac": nbytes / ms / 1e6 / pk["hbm"],
              "frac_of_nominal_8TBs": nbytes / ms / 1e6 / 8000.0, "algorithmic_bytes": nbytes}

    def tens(ms, flops):
      return {"bound": "tensor", "ms": ms, "achieved": flops / ms / 1e9, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": flops / ms / 1e9 / pk["tensor"],
              "algorithmic_flops": flops}
    kernels = {
      "cost_volume": hbm(cv_ms, cv_bytes),
      "cost_volume_back_to_back": dict(hbm(cvr_ms, cv_bytes), note=f"{nrot} rotating 22.5 MB outputs (> 2x L2), launches back to back as inside the forward"),
      "cost_volume_batch8": hbm(cv8_ms, 8 * cv_bytes),
      "filter_conv3d_32x32": tens(f3_ms, f3_flops),
      "refine_conv2d_32x32_dil4": tens(r2_ms, r2_flops),
      "head_taps27_tensor_core": dict(hbm(tp_ms, tp_bytes), note="inference head, kernel 1 of 2: conv3d_alone as a 32 -> 27-tap contraction on the tensor cores"),
      "head_tapsum_softargmin": dict(hbm(ts_ms, ts_bytes), note="inference head, kernel 2 of 2: 27-tap gather + softmax + expectation + cost volume"),
      "head_fused_one_kernel": dict(hbm(hd_ms, hd_bytes), note="training path: conv3d_alone + softmax + expectation + cost + FCS in ONE CUDA-core kernel"),
      "first_conv5x5s2_2images": tens(fc_ms, fc_flops),
      "refine_in_conv": dict(hbm(ri_ms, ri_bytes), note="inference: snb_refine_pack_input + snb_conv_c4_ws (two launches)"),
      "refine_in_conv_im2col_training_path": hbm(ri_old_ms, ri_bytes),
    }
    # dominant kernel of the step = the 32->32 convolution (4 x 3-D filter + 6 x refinement launches per pair)
    dom_name = "filter_conv3d_32x32" if 4 * f3_ms >= 6 * r2_ms else "refine_conv2d_32x32_dil4"
    dom = kernels[dom_name]
    # DRAM traffic and tensor-pipe activity of the same kernel: NOT measured in this run, read from the committed `ncu --set full`
    # capture of the same kernel (profiles/r2_ncu_summary.json)
    ncu = {}
    try:
      ncu = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_summary.json")))
    except Exception:
      pass
    ncu_k = ncu.get("conv3d_ws" if dom_name == "filter_conv3d_32x32" else "conv2d_ws_dil4", {})
    roofline = {"kernel": dom_name, "bound": dom["bound"], "achieved": dom["achieved"], "peak": dom["peak"], "unit": dom["unit"],
                "frac": dom["frac"], "traffic": ncu_k.get("dram_bytes"),
                "traffic_source": "profiles/r2_ncu_summary.json (ncu --set full capture of this kernel; not re-measured in this run)",
                "peak_source": pk["src"] + " (bf16 cuBLAS burst; kernel timed alone)",
                "note": "achieved = algorithmic fp32 conv FLOPs / time; the kernel runs 3 fp16 MMA products per algorithmic product "
                        "(error-compensated split, fp32-grade parity), so 1/3 of the bf16 peak is the ceiling of this formulation",
                "frac_of_3xf16_ceiling": dom["achieved"] / (pk["tensor"] / 3.0),
                "ncu_tensor_pipe_active_pct": ncu_k.get("tensor_pipe_active_pct")}
    del flush

    cpu = cpu_reference(steps=args.cpu_steps, warmup=1, budget_s=25.0) if world == 1 and not args.skip_cpu else None

    in_bytes = 2 * left.numel() * 4
    out_bytes = out_pin.numel() * 4
    result = {
      "metric": METRIC, "value": world * steps_dev / (ms_dev / 1e3), "unit": "pairs/s", "n_gpus": world,
      "steps": steps_dev, "steps_requested": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / steps_dev, "higher_is_better": True,
      "scaling": "weak", "vs_baseline": None, "dtype": "f32",
      "data": "synthetic (textured left, right = left warped by a known disparity ramp; seeded random-init weights)",
      "config": {"workload": WORKLOAD, "pairs_per_gpu_per_step": 1, "k": K_DOWN, "maxdisp": MAXDISP,
                 "l2": "per-step working set ~0.7 GB of intermediates >> 126 MB L2; per-kernel numbers flush L2 before every launch",
                 "cuda_graph": not args.no_graph, "parallelism": f"independent pairs per GPU x{world}, no collective",
                 "min_timed_seconds": args.min_seconds,
                 "arithmetic": "fp32 I/O; 32->32 convolutions as error-compensated fp16-split tcgen05 MMAs (3 products, fp32 accumulate)"},
      "e2e": {"value": world * steps_e2e / (ms_e2e / 1e3), "unit": "pairs/s", "ms_per_step": ms_e2e / steps_e2e, "steps": steps_e2e,
              "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": out_bytes,
              "api": "stereonet_b200.runtime.StereoEngine.infer_host_async (pinned host images -> host disparity, every frame; "
                     "copies of neighbouring frames overlap the forward on separate streams)",
              "blocking_call_ms": ms_seq / steps_seq},
      "gpu_launches": launches * steps_dev,
      "launches_per_step": launches,
      "roofline": roofline, "kernels": kernels, "clocks": clocks,
    }
    if timing:
      result["timing_configs"] = timing
  # entries measured on every rank
  if rank == 0:
    if sf is not None:
      result["sceneflow_b32"] = sf
    if adapt is not None:
      result["adapt"] = adapt
    if cpu is not None:
      result["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
      if adapt is not None and not args.skip_cpu_adapt:
        result["adapt"]["cpu_baseline"] = cpu_reference_adapt(steps=2)
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()
  return result


def main():
  if os.environ.get("SNB_BENCH_DUMP_AFTER"):        # debugging aid: dump all Python stacks and exit if the run stalls
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ["SNB_BENCH_DUMP_AFTER"]), exit=True)
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=50)
  ap.add_argument("--warmup", type=int, default=5)
  ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
  ap.add_argument("--min-seconds", type=float, default=0.0,
                  help="> 0: every timed region runs at least this long (and at least its number of steps); 0: exactly its number of steps")
  ap.add_argument("--dump-outputs", metavar="DIR",
                  help="after the timed steps, write the outputs of the last step of the `value` region as DIR/<name>.npy (float32)")
  ap.add_argument("--no-graph", action="store_true")
  ap.add_argument("--skip-cpu", action="store_true")
  ap.add_argument("--cpu-steps", type=int, default=12)
  ap.add_argument("--skip-adapt", action="store_true")
  ap.add_argument("--skip-cpu-adapt", action="store_true")
  ap.add_argument("--skip-sceneflow", action="store_true")
  ap.add_argument("--skip-timing-configs", action="store_true")
  ap.add_argument("--adapt-single-stream", action="store_true", help="A/B: both feature passes of the adaptation step on one stream")
  args = ap.parse_args()

  rank = int(os.environ.get("RANK", "0"))
  if args.impl == "reference":
    if args.dump_outputs:
      ap.error("--dump-outputs applies to --impl b200 (the reference arm runs other seeded weights)")
    if rank != 0:
      return
    c = cpu_reference(steps=args.steps, warmup=min(args.warmup, 2), budget_s=float("inf"))
    line = {"impl": "reference", "metric": METRIC, "value": c["value"], "unit": "pairs/s", "n_gpus": args.gpus, "steps": c["steps"],
            "warmup": min(args.warmup, 2), "ms_per_step": c["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD},
            "cpu_baseline": {k: c[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": c["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return
  res = gpu_arm(args)
  if res is not None:
    print(json.dumps(res))


if __name__ == "__main__":
  main()
