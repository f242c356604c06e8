"""Whole-model C-ABI (snb_stereonet_forward) against the Python eval path at KITTI size (B = 1, 376x1248, k = 3, maxdisp 192), in
one process with the two paths alternating round by round:
  graph   the native forward captured into a CUDA graph vs StereoEngine's captured forward (same kernels: device time should match);
  eager   one native call from the host vs the eager Python module forward (no_grad, eval), for the host launch cost per frame:
          `enqueue_us` is the host time to issue one frame, `frame_us` the event time of back-to-back frames.
Both produce the full-resolution and coarse disparity (no cost volume).  Usage: python scripts/bench_native.py [out.json]"""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "adaptive-stereo-icra-2021_b200"), os.path.join(ROOT, "oracle")]
import torch

import stereonet_oracle as O
import stereonet_b200 as S
from stereonet_b200 import _cabi, native
from stereonet_b200.runtime import StereoEngine

DEV = "cuda:0"
B, H, W, K, MAXDISP = 1, 376, 1248, 3, 192
ROUNDS, N = 7, 50


def card():
  info = dict(name=torch.cuda.get_device_name(0))
  try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30)
    info["power_limit_and_max_sm_clock"] = q.stdout.strip()
  except Exception as exc:      # the numbers are still worth having; say why the card data is missing
    info["power_limit_and_max_sm_clock"] = f"unavailable: {exc}"
  return info


def timed(fn, n, stream):
  """(event time per call, host enqueue time per call) over n back-to-back calls, microseconds."""
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  torch.cuda.synchronize()
  a.record(stream)
  t0 = time.perf_counter()
  for _ in range(n):
    fn()
  t1 = time.perf_counter()
  b.record(stream)
  torch.cuda.synchronize()
  return a.elapsed_time(b) * 1e3 / n, (t1 - t0) * 1e6 / n


def main():
  torch.backends.cudnn.benchmark = False
  f = S.FeatureExtractorNetwork(K).to(DEV).eval()
  n = S.StereoNet(K, 1, 0, maxdisp=MAXDISP).to(DEV).eval()
  f.load_state_dict(O.make_feature_state(K, 11)); n.load_state_dict(O.make_stereo_state(22, sharpen=40.0))
  g = torch.Generator(device=DEV).manual_seed(5)
  pair = torch.rand((2 * B, 3, H, W), device=DEV, generator=g)
  lib = _cabi.lib()
  stream = torch.cuda.current_stream()
  sp = C.c_void_p(stream.cuda_stream)

  weights = torch.empty((lib.snb_stereonet_weights_bytes(K),), device=DEV, dtype=torch.uint8)
  _cabi.check(lib.snb_stereonet_prepare(native.param_pointers(f, n), K, weights.data_ptr(), sp), "snb_stereonet_prepare")
  ws = torch.empty((lib.snb_stereonet_workspace_bytes(K, 0, MAXDISP, B, H, W),), device=DEV, dtype=torch.uint8)
  disp, coarse = torch.empty((B, H, W), device=DEV), torch.empty((B, H, W), device=DEV)
  args = (weights.data_ptr(), K, 0, MAXDISP, pair.data_ptr(), B, H, W, ws.data_ptr(), disp.data_ptr(), coarse.data_ptr(), None, None)

  def native_eager():
    lib.snb_stereonet_forward(*args, C.c_void_p(torch.cuda.current_stream().cuda_stream))

  native_eager()
  graph = torch.cuda.CUDAGraph()
  with torch.cuda.graph(graph):
    native_eager()

  eng = StereoEngine(f, n, output_cost_volume=False)
  eng(pair[:B], pair[B:])                                   # capture

  def python_eager():
    with torch.no_grad():
      eng._forward(pair)

  python_eager()
  graph.replay()
  out, _ = eng.run_static(tuple(pair[:B].shape), pair.device)
  torch.cuda.synchronize()
  same = torch.equal(disp, out["pred_disp_l/0"][:, 0]) and torch.equal(coarse, out["pred_disp_l/3"][:, 0])

  paths = {"graph_native": graph.replay, "graph_python": lambda: eng.run_static(tuple(pair[:B].shape), pair.device),
           "eager_native": native_eager, "eager_python": python_eager}
  for fn in paths.values():                                  # warm every path
    timed(fn, 5, stream)
  rows = {name: [] for name in paths}
  for _ in range(ROUNDS):
    for name, fn in paths.items():
      rows[name].append(timed(fn, N, stream))
  res = dict(card=card(), shape=dict(B=B, H=H, W=W, k=K, maxdisp=MAXDISP), rounds=ROUNDS, calls_per_round=N,
             outputs_bit_identical=same)
  for name, r in rows.items():
    res[name] = dict(frame_us_median=statistics.median(x[0] for x in r), frame_us_min=min(x[0] for x in r),
                     frame_us_max=max(x[0] for x in r), enqueue_us_median=statistics.median(x[1] for x in r))
  print(json.dumps(res, indent=1))
  if len(sys.argv) > 1:
    os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
    with open(sys.argv[1], "w") as fh:
      json.dump(res, fh, indent=1)


if __name__ == "__main__":
  main()
