"""The oracle (oracle/stereonet_oracle.py) against golden vectors produced by the reference module itself
(oracle/gen_golden.py, run in the build container).  CPU only."""
import os

import numpy as np
import pytest
import torch

import stereonet_oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TRAIN_SHARPEN_RATIO = 0.25      # oracle/gen_golden.py: milder conv3d_alone gain for the train-mode step
CASES = {
  "k3_small_dgtw": dict(B=1, H=64, W=128, k=3, s=0, sharpen=1.0, train=False),
  "k3_b2_sharp":   dict(B=2, H=96, W=256, k=3, s=0, sharpen=40.0, train=True),
  "k4_sharp":      dict(B=1, H=64, W=256, k=4, s=0, sharpen=40.0, train=False),
  "k3_ragged":     dict(B=1, H=68, W=120, k=3, s=0, sharpen=40.0, train=True),
  "k3_scale1":     dict(B=1, H=48, W=96,  k=3, s=1, sharpen=40.0, train=False),
}


def build(cfg):
  fsd = O.make_feature_state(cfg["k"], seed=11)
  ssd = O.make_stereo_state(seed=22, sharpen=cfg["sharpen"])
  left, right, gt = O.make_stereo_pair(cfg["B"], cfg["H"], cfg["W"], seed=1000, max_disp_px=min(60.0, cfg["W"] / 4))
  return fsd, ssd, left, right, gt


def summ(t):
  t = t.detach().double().flatten()
  return np.array([t.sum().item(), t.abs().sum().item(), (t * t).sum().sqrt().item()])


ADAM_LR = 5e-5


def zero_grad_bias(n):
  """Biases whose gradient in a train-mode step is mathematically zero: a convolution feeding a batch-statistics BatchNorm
  (convbn / convbn_3d: '<...>.0.0.bias', the BN removes the batch mean), conv3d_alone.bias (under the softmax: shift invariant) and
  conv_alone.bias (cancels in L - R).  What is computed for them is rounding noise whose value depends on the host CPU's
  summation order (its oneDNN kernels), and Adam's first step turns that noise into a move of up to lr per element.  They are
  held to zero up to rounding and to that lr bound instead of to the stored noise (as in tests/test_gpu_backward.py)."""
  return n.endswith(".0.0.bias") or n in ("conv3d_alone.bias", "conv_alone.bias")


def zero_up_to_rounding(grads, tag, n):
  """|gradient| <= 1e-3 x the largest gradient entry of the same convolution's weight (the noise measures below 5e-5 x)."""
  return grads[(tag, n)].abs().max().item() <= 1e-3 * grads[(tag, n[:-len("bias")] + "weight")].abs().max().item()


@pytest.mark.parametrize("name", list(CASES))
def test_inputs_regenerate(name):
  """Seeded weights/inputs must regenerate exactly, otherwise the fixtures do not apply."""
  cfg = CASES[name]
  g = np.load(os.path.join(GOLD, name + ".npz"))
  fsd, ssd, left, right, _ = build(cfg)
  np.testing.assert_allclose(summ(left), g["in_left_sum"], rtol=1e-12)
  np.testing.assert_allclose(summ(right), g["in_right_sum"], rtol=1e-12)
  np.testing.assert_allclose(summ(torch.cat([v.flatten().float() for v in fsd.values()])), g["w_feat_sum"], rtol=1e-12)
  np.testing.assert_allclose(summ(torch.cat([v.flatten().float() for v in ssd.values()])), g["w_stereo_sum"], rtol=1e-12)


@pytest.mark.parametrize("name", list(CASES))
def test_eval_forward_matches_reference(name):
  cfg = CASES[name]
  g = np.load(os.path.join(GOLD, name + ".npz"))
  fsd, ssd, left, right, gt = build(cfg)
  ex = {}
  with torch.no_grad():
    o = O.predict_disparity_left(fsd, ssd, left, right, cfg["k"], cfg["s"], training=False, extras=ex)
  np.testing.assert_allclose(ex["left_features"].numpy(), g["eval/left_features"], rtol=0, atol=2e-5)
  np.testing.assert_allclose(ex["right_features"].numpy(), g["eval/right_features"], rtol=0, atol=2e-5)
  for key, v in o.items():
    ref = g["eval/" + key]
    tol = 1e-3 if key.startswith("pred_disp") else 2e-4
    np.testing.assert_allclose(v.numpy(), ref, rtol=0, atol=tol, err_msg=key)
  s, k = cfg["s"], cfg["k"]
  assert abs(O.feature_contrast_mean(o[f"cost_volume_l/{s + k}"]).mean().item() - float(g["eval/fcs"])) < 1e-4
  assert abs(O.epe(o[f"pred_disp_l/{s}"], gt).item() - float(g["eval/epe"])) < 1e-3
  # the numpy literal-loop restatement of the cost volume is bit-identical to the differentiable one
  D = (192 + 1) // 2 ** (s + k)
  cv = O.cost_volume_numpy(ex["left_features"].numpy(), ex["right_features"].numpy(), D)
  assert np.array_equal(cv, ex["raw_cost_volume"].numpy())


@pytest.mark.parametrize("name", [n for n, c in CASES.items() if c["train"]])
def test_adapt_step_matches_reference(name):
  cfg = CASES[name]
  g = np.load(os.path.join(GOLD, name + ".npz"))
  fsd, ssd, left, right, _ = build(cfg)
  ssd = O.make_stereo_state(seed=22, sharpen=cfg["sharpen"] * TRAIN_SHARPEN_RATIO)
  fsd, ssd = O.clone_state(fsd, True), O.clone_state(ssd, True)
  adam = {}
  loss, outputs, grads = O.adapt_step(fsd, ssd, left, right, cfg["k"], adam, lr=ADAM_LR, input_scale=cfg["s"])
  assert abs(loss.item() - float(g["train/loss"])) < 2e-6
  for key, v in outputs.items():
    np.testing.assert_allclose(v.detach().numpy(), g["train/" + key], rtol=0, atol=2e-3, err_msg=key)
  # unclipped gradients were stored; recompute them from the clipped ones via the stored norm
  gn = float(g["train/grad_norm_stereo"])
  coef = min(1.0, 1.0 / (gn + 1e-6))
  checked = 0
  for key in g.files:
    if key.startswith("grad_sum/"):
      _, tag, n = key.split("/", 2)
      got = grads[(tag, n)] / (coef if tag == "s" else 1.0)
      ref = g[key]
      if zero_grad_bias(n):
        assert zero_up_to_rounding(grads, tag, n), key
      else:
        assert abs(summ(got)[2] - ref[2]) <= 2e-3 * ref[2] + 1e-7, (key, summ(got), ref)
      checked += 1
    elif key.startswith("grad_none/"):
      _, tag, n = key.split("/", 2)
      assert O.unused_param(n)
    elif key.startswith("grad/"):
      _, tag, n = key.split("/", 2)
      got = (grads[(tag, n)] / (coef if tag == "s" else 1.0)).numpy()
      ref = g[key]
      scale = np.abs(ref).max() + 1e-12
      assert zero_up_to_rounding(grads, tag, n) if zero_grad_bias(n) else np.abs(got - ref).max() <= 2e-3 * scale + 1e-7, key
  assert checked > 40
  for key in g.files:
    if key.startswith("post/"):
      _, tag, n = key.split("/", 2)
      sd = ssd if tag == "s" else fsd
      if zero_grad_bias(n):
        np.testing.assert_allclose(sd[n].detach().numpy(), g[key], rtol=0, atol=2 * ADAM_LR, err_msg=key)
      else:
        np.testing.assert_allclose(sd[n].detach().numpy(), g[key], rtol=1e-4, atol=1e-6, err_msg=key)
    elif key.startswith("post_sum/"):
      _, tag, n = key.split("/", 2)
      sd = ssd if tag == "s" else fsd
      if zero_grad_bias(n):
        np.testing.assert_allclose(summ(sd[n]), g[key], rtol=0, atol=2 * ADAM_LR * sd[n].numel(), err_msg=key)
      else:
        np.testing.assert_allclose(summ(sd[n]), g[key], rtol=1e-5, atol=1e-7, err_msg=key)


# ---- round 2: the reference's own test / timing configurations at full size (oracle/gen_golden.py BIG_CASES) and rows f3 / f4
BIG_CASES = {
  "T_320x960_k3": dict(B=1, H=320, W=960, k=3, s=0, sharpen=40.0),       # BASELINE.json configs[0], test/test_stereo_net.py:17-22
  "k4_320x960":   dict(B=1, H=320, W=960, k=4, s=0, sharpen=40.0),       # k = 4: every experiments/adaptation/*.sh
  "k3s1_160x480": dict(B=1, H=160, W=480, k=3, s=1, sharpen=40.0),       # input_scale = 1, test/test_stereo_net.py:60-72
}
SUB = 4


def check_big(name, o, fl, gt, g, cfg, disp_tol, cost_tol, feat_tol):
  """Shared by the CPU (oracle) and GPU (product) tests: outputs of one eval forward against the reference's golden tensors."""
  s, k = cfg["s"], cfg["k"]
  errs = {}
  errs["features"] = float(np.abs(fl[..., ::SUB, ::SUB] - g["eval/left_features_sub"]).max())
  errs["cost"] = float(np.abs(o[f"cost_volume_l/{s + k}"] - g[f"eval/cost_volume_l/{s + k}"]).max())
  errs["coarse"] = float(np.abs(o[f"pred_disp_l/{s + k}"][..., ::SUB, ::SUB] - g[f"eval/pred_disp_l/{s + k}_sub"]).max())
  errs["refined"] = float(np.abs(o[f"pred_disp_l/{s}"] - g[f"eval/pred_disp_l/{s}"]).max())
  print(f"[parity] {name}: " + "  ".join(f"{k_}={v:.3e}" for k_, v in errs.items()))
  assert errs["features"] <= feat_tol and errs["cost"] <= cost_tol and errs["coarse"] <= disp_tol and errs["refined"] <= disp_tol, errs
  pred = torch.from_numpy(np.asarray(o[f"pred_disp_l/{s}"]))
  m = O.eval_metrics(pred, gt)
  assert abs(m["EPE"] - float(g["eval/epe"])) <= 1e-3                         # north star: |dEPE| <= 1e-3 px
  for i, t in enumerate(O.D1_THRESHOLDS):
    assert abs(m[f"D1_all_{t}px"] - float(g["eval/d1_all"][i])) <= 1e-4
  return errs


@pytest.mark.parametrize("name", list(BIG_CASES))
def test_big_eval_forward_matches_reference(name):
  cfg = BIG_CASES[name]
  g = np.load(os.path.join(GOLD, name + ".npz"))
  fsd, ssd, left, right, gt = build(cfg)
  np.testing.assert_allclose(summ(left), g["in_left_sum"], rtol=1e-12)
  ex = {}
  with torch.no_grad():
    o = O.predict_disparity_left(fsd, ssd, left, right, cfg["k"], cfg["s"], training=False, extras=ex)
  check_big(name, {k_: v.numpy() for k_, v in o.items()}, ex["left_features"].numpy(), gt, g, cfg, disp_tol=1e-3, cost_tol=2e-4, feat_tol=2e-5)
  fcs = O.feature_contrast_mean(o[f"cost_volume_l/{cfg['s'] + cfg['k']}"]).mean().item()
  assert abs(fcs - float(g["eval/fcs"])) < 1e-4


def test_rows_f3_f4_oracle_matches_reference():
  """khamis_robust_loss, evaluate() metrics, the OVS validation loop and one two-pass ER Adam step of the oracle against the
  values the reference's own functions produced (oracle/gen_golden.py run_rows_case)."""
  g = np.load(os.path.join(GOLD, "rows_f3_f4.npz"))
  pred = torch.from_numpy(g["khamis/pred"]).requires_grad_(); gt = torch.from_numpy(g["khamis/gt"])
  loss = O.khamis_robust_loss(pred, gt)
  loss.backward()
  assert abs(loss.item() - float(g["khamis/loss"])) < 1e-6
  np.testing.assert_allclose(pred.grad.numpy(), g["khamis/dpred"], rtol=1e-5, atol=1e-9)
  H, W, k = 96, 256, 3
  fsd, ssd = O.make_feature_state(k, 11), O.make_stereo_state(22, sharpen=10.0)
  # evaluate(): 3 batches of 2 pairs
  epe, d1, fcs = [], [], []
  with torch.no_grad():
    for i in range(3):
      l, r, gtd = O.make_stereo_pair(2, H, W, seed=3000 + i, max_disp_px=40.0)
      o = O.predict_disparity_left(fsd, ssd, l, r, k)
      m = O.eval_metrics(o["pred_disp_l/0"], gtd, o["cost_volume_l/3"])
      epe.append(m["EPE"]); fcs.append(m["FCS"]); d1.append([m[f"D1_all_{t}px"] for t in O.D1_THRESHOLDS])
  assert abs(np.mean(epe) - float(g["evaluate/EPE"])) < 1e-4
  assert abs(np.mean(fcs) - float(g["evaluate/FCS"])) < 1e-4
  np.testing.assert_allclose(np.mean(np.array(d1), axis=0), g["evaluate/D1_all"], atol=3e-5)
  # StateMachine.validate loop
  pairs = [O.make_stereo_pair(1, H, W, seed=2000 + i, max_disp_px=40.0)[:2] for i in range(5)]
  np.testing.assert_allclose(np.array(O.validate_ovs(fsd, ssd, pairs, k)), g["validate/losses"], atol=2e-6)
  # one ER step (two train-mode passes)
  f2, s2 = O.clone_state(fsd, True), O.clone_state(ssd, True)
  l, r, _ = O.make_stereo_pair(1, H, W, seed=1000, max_disp_px=40.0)
  rl, rr, rgt = O.make_stereo_pair(1, H, W, seed=1001, max_disp_px=40.0)
  loss, _, grads = O.adapt_step(f2, s2, l, r, k, {}, lr=ADAM_LR, replay=(rl, rr, rgt))
  assert abs(loss.item() - float(g["er/loss"])) < 2e-5
  for key in g.files:
    if key.startswith("er/post/") and ("running_" in key or "num_batches" in key):
      _, _, tag, n = key.split("/", 3)
      np.testing.assert_allclose((s2 if tag == "s" else f2)[n].detach().numpy(), g[key], rtol=1e-4, atol=1e-6, err_msg=key)
    elif key.startswith("er/post_sum/"):
      _, _, tag, n = key.split("/", 3)
      t = (s2 if tag == "s" else f2)[n]
      if zero_grad_bias(n):
        assert zero_up_to_rounding(grads, tag, n), key
        np.testing.assert_allclose(summ(t), g[key], rtol=0, atol=2 * ADAM_LR * t.numel(), err_msg=key)
      else:
        np.testing.assert_allclose(summ(t), g[key], rtol=1e-5, atol=1e-7, err_msg=key)
