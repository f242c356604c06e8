"""Shared-model data-parallel adaptation through the C-ABI: examples/stereonet_adapt_dp.cpp (one process, G devices, NCCL all-reduce of
the state's dp_flat piece between the captured forward + backward graph and the captured apply graph) at KITTI size (B = RB = 1,
376x1248, k = 3, maxdisp 192, clip on, one replay sample per rank and step, er_weight 0.05), at G = 1, 2, 4, 8 up to the number of
devices present.  Each G runs ROUNDS times; `step_us` is the example's device-event time per step over the steps after the first.
Next to it the Python DP step of the same workload, bench.py --gpus N (its keyed entry `adapt`: `ms_per_step` of the DP step with
replay at N > 1, `with_replay.ms_per_step` at N = 1), unless --no-python.  The native step runs its passes one after another; the
Python step overlaps them on several streams.
Usage: python scripts/bench_native_adapt_dp.py [--no-python] [out.json]"""
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "adaptive-stereo-icra-2021_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "scripts")]
import numpy as np
import torch

import stereonet_oracle as O
import stereonet_b200 as S
from stereonet_b200 import native
from bench_native import card

B, RB, H, W, K, MAXDISP = 1, 1, 376, 1248, 3, 192
F, NREP, STEPS, ROUNDS = 4, 8, 41, 3           # distinct frames per rank, stored replay samples, steps per run (the first untimed)


def build_example(tmp):
  import importlib.util
  spec = importlib.util.spec_from_file_location("snb200_build", os.path.join(ROOT, "adaptive-stereo-icra-2021_b200", "build.py"))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  return mod.build_example(os.path.join(tmp, "stereonet_adapt_dp"), "stereonet_adapt_dp")


def python_dp(n):
  """bench.py's DP adaptation step at N GPUs (ms per step), or the reason it is missing."""
  args = ["--gpus", str(n), "--steps", "50", "--warmup", "5", "--skip-cpu", "--skip-cpu-adapt", "--skip-sceneflow",
          "--skip-timing-configs"]
  cmd = ([sys.executable, os.path.join(ROOT, "bench.py")] if n == 1 else
         [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc_per_node={n}", os.path.join(ROOT, "bench.py")])
  r = subprocess.run(cmd + args, capture_output=True, text=True, timeout=1800, cwd=ROOT)
  lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
  if r.returncode != 0 or not lines:
    return dict(error=f"bench.py exit {r.returncode}: {(r.stdout + r.stderr)[-400:]}")
  adapt = json.loads(lines[-1]).get("adapt") or {}
  entry = adapt.get("with_replay", {}) if n == 1 else adapt
  return dict(step_us=entry.get("ms_per_step", float("nan")) * 1e3, source="bench.py --gpus %d: adapt%s" %
              (n, ".with_replay" if n == 1 else ""), parallelism=adapt.get("parallelism"))


def main():
  argv = [a for a in sys.argv[1:] if a != "--no-python"]
  with_python = "--no-python" not in sys.argv[1:]
  ndev = torch.cuda.device_count()
  if ndev < 1:
    raise SystemExit("bench_native_adapt_dp: no CUDA device")
  gs = [g for g in (1, 2, 4, 8) if g <= ndev]
  res = dict(card=card(), devices=ndev, shape=dict(B=B, RB=RB, H=H, W=W, k=K, maxdisp=MAXDISP, clip=True, er_weight=0.05),
             rounds=ROUNDS, timed_steps_per_round=STEPS - 1, distinct_frames_per_rank=F, replay_samples=NREP, native={}, python={})
  with tempfile.TemporaryDirectory() as tmp:
    exe = build_example(tmp)
    f = S.FeatureExtractorNetwork(K)
    n = S.StereoNet(K, 1, 0, maxdisp=MAXDISP)
    f.load_state_dict(O.make_feature_state(K, 11)); n.load_state_dict(O.make_stereo_state(22, sharpen=40.0))
    native.export_weights(f, n, os.path.join(tmp, "w.bin"))
    rng = np.random.default_rng(5)
    rimg = rng.random((NREP, 2, RB, 3, H, W), dtype=np.float32)
    gt = rng.random((NREP, RB, H, W), dtype=np.float32) * 40.0 + 0.5
    gt[..., :W // 4] = 0.0
    rimg.tofile(os.path.join(tmp, "rimg.bin")); gt.tofile(os.path.join(tmp, "rgt.bin"))
    for g in gs:
      rng.random((F, g, 2, B, 3, H, W), dtype=np.float32).tofile(os.path.join(tmp, "img.bin"))
      rows = []
      for _ in range(ROUNDS):
        r = subprocess.run([exe, str(g), os.path.join(tmp, "w.bin"), os.path.join(tmp, "img.bin"), str(B), str(H), str(W), str(STEPS),
                            os.path.join(tmp, "out.bin"), "5e-5", os.path.join(tmp, "rimg.bin"), os.path.join(tmp, "rgt.bin"), str(RB),
                            str(NREP)], capture_output=True, text=True, timeout=1800)
        m = re.search(r"([\d.]+) us per step", r.stdout)
        if r.returncode != 0 or not m or f"{g} replicas identical" not in r.stdout:
          raise SystemExit(f"stereonet_adapt_dp G = {g} failed:\n{(r.stdout + r.stderr)[-3000:]}")
        rows.append(float(m.group(1)))
      res["native"][str(g)] = dict(step_us_median=statistics.median(rows), step_us_min=min(rows), step_us_max=max(rows),
                                   steps_per_s_all_ranks=g * 1e6 / statistics.median(rows))
      print(g, res["native"][str(g)], flush=True)
  if with_python:
    for g in gs:
      res["python"][str(g)] = python_dp(g)
      print(g, res["python"][str(g)], flush=True)
  print(json.dumps(res, indent=1))
  if argv:
    os.makedirs(os.path.dirname(os.path.abspath(argv[0])), exist_ok=True)
    with open(argv[0], "w") as fh:
      json.dump(res, fh, indent=1)


if __name__ == "__main__":
  main()
