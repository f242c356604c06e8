"""The opt-in reduced-precision forward (snb_stereonet_forward_f16) against the default fp32-grade one (snb_stereonet_forward) at
KITTI size (376x1248, k = 3, maxdisp 192), B = 1 and B = 8, in one process:
  forward  each forward captured into a CUDA graph; the two graphs alternate window by window (ROUNDS windows of N replays
           each, after WARMUP replays), so both see the same clocks and neighbours; the spread over the windows is reported;
  layers   one refinement block (dil 4, folded BN + LeakyReLU + residual) and one 3-D cost-filter layer (folded BN + LeakyReLU) on
           snb_conv_c32_ws vs snb_conv_c32_ws_f16, each launch alone with a 256 MB L2 flush before it (as bench.py's `kernels`).
The card name, power limit and max SM clock are read in the same run.  Usage: python scripts/bench_f16.py [out.json]"""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "adaptive-stereo-icra-2021_b200"), os.path.join(ROOT, "oracle")]
import torch

import stereonet_oracle as O
import stereonet_b200 as S
from stereonet_b200 import _cabi, native, ops
from stereonet_b200.autograd import fused

DEV = "cuda:0"
H, W, K, MAXDISP = 376, 1248, 3, 192
WARMUP, ROUNDS, N = 30, 8, 100


def card():
  info = dict(name=torch.cuda.get_device_name(0))
  try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30)
    info["power_limit_and_max_sm_clock"] = q.stdout.strip()
  except Exception as exc:
    info["power_limit_and_max_sm_clock"] = f"unavailable: {exc}"
  return info


def window_us(fn, n, stream):
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  a.record(stream)
  for _ in range(n):
    fn()
  b.record(stream)
  torch.cuda.synchronize()
  return a.elapsed_time(b) * 1e3 / n


def time_kernel_us(fn, iters, flush, stream):
  """Per-launch times (us) of fn() alone, L2 flushed before every launch, CUDA events on the launching stream."""
  for _ in range(3):
    fn()
  evs = []
  for _ in range(iters):
    flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream); fn(); b.record(stream)
    evs.append((a, b))
  torch.cuda.synchronize()
  return sorted(a.elapsed_time(b) * 1e3 for a, b in evs)


def summary(xs):
  return dict(median=statistics.median(xs), min=min(xs), max=max(xs))


def bench_forward(f, n, B, stream):
  lib = _cabi.lib()
  sp = C.c_void_p(stream.cuda_stream)
  weights = torch.empty((lib.snb_stereonet_weights_bytes(K),), device=DEV, dtype=torch.uint8)
  _cabi.check(lib.snb_stereonet_prepare(native.param_pointers(f, n), K, weights.data_ptr(), sp), "snb_stereonet_prepare")
  g = torch.Generator(device=DEV).manual_seed(5)
  pair = torch.rand((2, B, 3, H, W), device=DEV, generator=g)
  ws = torch.empty((lib.snb_stereonet_workspace_bytes(K, 0, MAXDISP, B, H, W),), device=DEV, dtype=torch.uint8)
  graphs, disps, bufs = {}, {}, []
  for name, fn in (("default", lib.snb_stereonet_forward), ("f16", lib.snb_stereonet_forward_f16)):
    disp, coarse = torch.empty((B, H, W), device=DEV), torch.empty((B, H, W), device=DEV)
    bufs.append(coarse)            # a captured graph writes it on every replay: it must outlive the graphs (the next capture frees cached blocks)
    args = (weights.data_ptr(), K, 0, MAXDISP, pair.data_ptr(), B, H, W, ws.data_ptr(), disp.data_ptr(), coarse.data_ptr(), None, None, sp)
    _cabi.check(fn(*args), name)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
      _cabi.check(fn(*args), name)
    graphs[name], disps[name] = graph, disp
  for graph in graphs.values():
    for _ in range(WARMUP):
      graph.replay()
  torch.cuda.synchronize()
  rows = {name: [] for name in graphs}
  for _ in range(ROUNDS):
    for name, graph in graphs.items():
      rows[name].append(window_us(graph.replay, N, stream))
  d = (disps["f16"] - disps["default"]).abs()
  res = {name: dict(summary(r), windows_us=r) for name, r in rows.items()}
  res["speedup_median"] = res["default"]["median"] / res["f16"]["median"]
  res["separated"] = res["f16"]["max"] < res["default"]["min"]            # every f16 window faster than every default window
  res["disp_abs_diff_vs_default"] = dict(max=d.max().item(), median=d.median().item())
  del graphs, bufs, ws, pair, weights
  return res


def bench_layers(n, stream):
  flush = torch.empty(256 * 1024 * 1024 // 4, device=DEV, dtype=torch.float32)
  hc, wc = (H + 7) // 8, (W + 7) // 8
  D = (MAXDISP + 1) // 2 ** K
  res = {}
  blk = n.edge_aware_refinements[0].residual_astrous_blocks[2]           # dilation 4
  conv, bn = blk.conv1[0][0], blk.conv1[0][1]
  x2 = torch.randn(1, H, W, 32, device=DEV)
  conv3, bn3 = n.filter[0][0][0], n.filter[0][0][1]
  x3 = torch.randn(1, D, hc, wc, 32, device=DEV)
  for tag, x, c, b, dil, resid in (("refine_block_dil4", x2, conv, bn, 4, True), ("filter3d_layer", x3, conv3, bn3, 1, False)):
    g = ops.geom(x.shape, 3, dil=dil)
    wimg = fused.wprep_tc(c)
    scale, shift = fused.bn_fold(b)
    kw = dict(bias=c.bias.detach(), scale=scale, shift=shift, residual=x if resid else None, lrelu=True)
    ts = {"default": [], "f16": []}
    for _ in range(4):                                                     # alternate the two kernels
      ts["default"] += time_kernel_us(lambda: ops.conv_c32_tc(x, wimg, g, fmt="ws", **kw), 10, flush, stream)
      ts["f16"] += time_kernel_us(lambda: ops.conv_c32_ws_f16(x, wimg, g, **kw), 10, flush, stream)
    out = {name: summary(v) for name, v in ts.items()}
    out["speedup_median"] = out["default"]["median"] / out["f16"]["median"]
    res[tag] = out
  del flush
  return res


def main():
  torch.backends.cudnn.benchmark = False
  f = S.FeatureExtractorNetwork(K).to(DEV).eval()
  n = S.StereoNet(K, 1, 0, maxdisp=MAXDISP).to(DEV).eval()
  f.load_state_dict(O.make_feature_state(K, 11)); n.load_state_dict(O.make_stereo_state(22, sharpen=40.0))
  stream = torch.cuda.Stream(device=DEV)
  res = dict(card=card(), shape=dict(H=H, W=W, k=K, maxdisp=MAXDISP), warmup_replays=WARMUP, windows=ROUNDS, replays_per_window=N)
  with torch.cuda.stream(stream), torch.no_grad():
    for B in (1, 8):
      res[f"forward_B{B}"] = bench_forward(f, n, B, stream)
      torch.cuda.empty_cache()
    res["layers"] = bench_layers(n, stream)
  res["card_after"] = card()
  print(json.dumps(res, indent=1))
  if len(sys.argv) > 1:
    os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
    with open(sys.argv[1], "w") as fh:
      json.dump(res, fh, indent=1)


if __name__ == "__main__":
  main()
