"""AdaptStepper's data-parallel steps on a one-rank NCCL group against its plain step, eager and CUDA graph: with one rank the
all-reduce sums one term, and the 1 / world of the gradients and of the BatchNorm statistics is x 1.0, so the step must leave
exactly what the plain step leaves.  Both routes: dp_bucket (parallel.DPBucket + optim.FusedAdamClip) and dp_params
(parallel.used_parameters + torch.optim.Adam)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SNIPPET = r'''
import os, sys
import torch, torch.distributed as dist
ROOT = sys.argv[1]
for p in (ROOT, os.path.join(ROOT, "adaptive-stereo-icra-2021_b200"), os.path.join(ROOT, "oracle")):
  sys.path.insert(0, p)
import stereonet_oracle as O
import stereonet_b200 as S
from stereonet_b200 import parallel
from stereonet_b200.adapt import AdaptStepper, make_optimizer
torch.cuda.set_device(0)
dev = torch.device("cuda", 0)
dist.init_process_group("nccl", device_id=dev)
assert dist.get_world_size() == 1
H, W = 96, 256
frames = [O.make_stereo_pair(1, H, W, seed=1000 + i, max_disp_px=40.0) for i in range(3)]
samples = [O.make_stereo_pair(1, H, W, seed=5000 + i, max_disp_px=30.0) for i in range(3)]


def run(use_graph, fused, dp, replay):
  """Three steps from the same weights; returns the losses, the model state and the optimizer state."""
  f = S.FeatureExtractorNetwork(3).to(dev); s = S.StereoNet(3, 1, 0).to(dev)
  f.load_state_dict(O.make_feature_state(3, 11)); s.load_state_dict(O.make_stereo_state(22, sharpen=10.0))
  opt = make_optimizer(f, s, lr=5e-5, capturable=not fused, fused=fused)
  kw = {}
  if dp:
    kw = dict(dp_bucket=parallel.DPBucket(opt, s, f)) if fused else dict(dp_params=parallel.used_parameters(s, f))
  st = AdaptStepper(f, s, opt, H, W, use_graph=use_graph)
  losses = []
  for i in range(3):
    rep = tuple(t.to(dev) for t in samples[i]) if replay else None
    losses.append(st.step(frames[i][0].to(dev), frames[i][1].to(dev), replay=rep, **kw)[0].item())
  torch.cuda.synchronize()
  state = {"losses": torch.tensor(losses, dtype=torch.float64)}
  for tag, net in (("stereo_net.", s), ("feature_net.", f)):
    state.update({tag + n: v.detach().cpu().clone() for n, v in net.state_dict().items()})
  for idx, st_ in opt.state_dict()["state"].items():
    state.update({"optimizer.{}.{}".format(idx, n): torch.as_tensor(v).detach().cpu().clone() for n, v in st_.items()})
  return state


bad = []
for use_graph in (False, True):
  for fused in (True, False):
    for replay in (False, True):
      case = "use_graph={} {} replay={}".format(use_graph, "dp_bucket" if fused else "dp_params", replay)
      ref, got = run(use_graph, fused, False, replay), run(use_graph, fused, True, replay)
      assert ref.keys() == got.keys(), case
      assert not torch.equal(ref["stereo_net.filter.0.0.0.weight"], O.make_stereo_state(22, sharpen=10.0)["filter.0.0.0.weight"]), case
      assert int(ref["stereo_net.filter.0.0.1.num_batches_tracked"]) == 3 * (2 if replay else 1), case
      for n in ref:
        if not torch.equal(ref[n], got[n]):
          bad.append("{}: {} max|diff| = {}".format(case, n, float((ref[n].double() - got[n].double()).abs().max())))
dist.destroy_process_group()
print("\n".join(bad[:50]))
print("{} tensors differ".format(len(bad)))
assert not bad
print("DP1_OK")
'''


def test_world_one_dp_steps_equal_plain_step():
  """Three steps at 96x256 of each data-parallel route (dp_bucket with and without a replay sample, dp_params likewise), eager
  and CUDA graph, bit-identical to the plain step of the same optimizer: losses, parameters, buffers (num_batches_tracked
  included) and the optimizer's moments and step counts."""
  env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29575", WORLD_SIZE="1", RANK="0")
  p = subprocess.run([sys.executable, "-c", SNIPPET, ROOT], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                     timeout=900)
  assert p.returncode == 0 and "DP1_OK" in p.stdout, p.stdout[-6000:]
