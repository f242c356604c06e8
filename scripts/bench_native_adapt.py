"""Single-pass adaptation step through the C-ABI (snb_stereonet_adapt_forward + _update, each captured into a CUDA graph) against
the Python step at KITTI size (B = 1, 376x1248, k = 3, maxdisp 192, clip on), in one process, the three variants alternating round
by round:
  native        the two native graphs replayed back to back (train-mode forward + loss, backward + clip + Adam);
  python_1s     AdaptStepper(make_optimizer(fused=True), two_streams=False, use_graph=True): the same kernels, one stream;
  python_2s     AdaptStepper(make_optimizer(fused=True), use_graph=True), the default: feature passes and weight gradients on
                side streams.
Each variant adapts its own copy of the same seeded model on the same frame; `frame_us` is event time of back-to-back steps.
--replay times the experience-replay step instead (snb_stereonet_adapt_forward_replay + _update_replay against
AdaptStepper.step(..., replay=(rl, rr, gt)), one stored sample, er_weight 0.05).  python_2s then runs the replay pass on a stream of
its own next to the stream pass; the native step and python_1s run the two passes one after the other.
Usage: python scripts/bench_native_adapt.py [--replay] [out.json]"""
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "adaptive-stereo-icra-2021_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "scripts")]
import torch

import stereonet_oracle as O
import stereonet_b200 as S
from stereonet_b200 import native
from stereonet_b200.adapt import AdaptStepper, make_optimizer
from bench_native import card, timed

DEV = "cuda:0"
B, H, W, K, MAXDISP = 1, 376, 1248, 3, 192
ROUNDS, N = 7, 20


def nets():
  f = S.FeatureExtractorNetwork(K).to(DEV)
  n = S.StereoNet(K, 1, 0, maxdisp=MAXDISP).to(DEV)
  f.load_state_dict(O.make_feature_state(K, 11)); n.load_state_dict(O.make_stereo_state(22, sharpen=40.0))
  return f, n


def main():
  argv = [a for a in sys.argv[1:] if a != "--replay"]
  replay = "--replay" in sys.argv[1:]
  g = torch.Generator(device=DEV).manual_seed(5)
  pair = torch.rand((2, B, 3, H, W), device=DEV, generator=g)
  rpair = torch.rand((2, B, 3, H, W), device=DEV, generator=g)
  gt = torch.rand((B, H, W), device=DEV, generator=g) * 40.0 + 0.5
  gt[:, :, :W // 4] = 0.0
  stream = torch.cuda.current_stream()

  nat = native.NativeAdapt(*nets(), lr=5e-5)
  loss = torch.empty((1 + B,), device=DEV)
  loss_replay = torch.empty((2,), device=DEV)
  nat.workspace(B, H, W, B if replay else 0)
  torch.cuda.synchronize()
  g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
  with torch.cuda.graph(g1):
    if replay:
      nat.forward(pair, loss, replay=(rpair, gt), loss_replay=loss_replay)
    else:
      nat.forward(pair, loss)
  with torch.cuda.graph(g2):
    nat.update()

  def native_step():
    g1.replay(); g2.replay()

  steppers = {}
  for name, two in (("python_1s", False), ("python_2s", True)):
    f, n = nets()
    steppers[name] = AdaptStepper(f, n, make_optimizer(f, n, lr=5e-5, fused=True), use_graph=True, two_streams=two)
  paths = {"native": native_step}
  for name, st in steppers.items():
    rep = (rpair[0], rpair[1], gt) if replay else None
    paths[name] = (lambda st=st, rep=rep: st.step(pair[0], pair[1], replay=rep))
  for fn in paths.values():                                  # capture / warm every path
    timed(fn, 3, stream)
  rows = {name: [] for name in paths}
  for _ in range(ROUNDS):
    for name, fn in paths.items():
      rows[name].append(timed(fn, N, stream)[0])
  shape = dict(B=B, H=H, W=W, k=K, maxdisp=MAXDISP, clip=True)
  if replay:
    shape.update(RB=B, er_weight=0.05)
  res = dict(card=card(), shape=shape, rounds=ROUNDS, steps_per_round=N, workspace_bytes=nat.workspace(B, H, W, B if replay else 0).numel())
  for name, r in rows.items():
    res[name] = dict(frame_us_median=statistics.median(r), frame_us_min=min(r), frame_us_max=max(r))
  print(json.dumps(res, indent=1))
  if argv:
    os.makedirs(os.path.dirname(os.path.abspath(argv[0])), exist_ok=True)
    with open(argv[0], "w") as fh:
      json.dump(res, fh, indent=1)


if __name__ == "__main__":
  main()
