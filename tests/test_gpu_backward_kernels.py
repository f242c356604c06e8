"""Backward kernels of the adaptation step, one wrapper at a time, against plain high-precision references at the shapes the
KITTI step runs (k = 3: 188x624, 94x312 and 47x156 features, a 24x47x156 cost volume, 376x1248 refinement; B = 1 and 2), at
375x1242 (ragged upsampling ratio) and at tiny / degenerate sizes.

Exact data wherever the kernel allows it: small integers for activations and gradients, dyadic weights (k/16, k/256),
power-of-two invstd with integer mean.  Every product and partial sum is then exact in fp32 (and in the fp16 / TF32 operand
splits), so the kernel must equal the float64 reference bit for bit whatever its summation order: a dropped, duplicated or
mis-indexed row or tap cannot hide behind a tolerance.  Each kernel also gets a random-float case against float64, with the
bound and its reason written beside it.  Where a LeakyReLU / ReLU kink makes rounding matter, inputs sit at least 1e-3 (or,
for integer-grid data, a checked margin) away from it, so no tolerance has to absorb a flipped mask.

The composite tests at the end run the autograd Functions of the adaptation step at the sizes the step runs, on the product
"ws" convolution back end and on "tc3" as a cross-check, in the pattern of test_gpu_backward.test_conv_bn_lrelu_backward."""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import stereonet_oracle as O
from stereonet_b200 import ops
from stereonet_b200.autograd import functions as Fn, fused
from test_gpu_kernels import cl, uncl, rnd, close, DEV

pytestmark = pytest.mark.gpu

BN_EPS = 1e-5
LRELU = 0.2


def gen(seed):
  return torch.Generator().manual_seed(seed)


def ints(shape, lo, hi, seed):
  """Integers in [lo, hi] as fp32."""
  return torch.randint(lo, hi + 1, tuple(shape), generator=gen(seed)).float()


def dyadic(shape, k, den, seed):
  """Multiples of 1/den in [-k/den, k/den]: exact in fp32, in the fp16 split and in TF32."""
  return ints(shape, -k, k, seed) / den


def exact(got, ref, what):
  """Bit-exact up to the sign of zero (a zero sum may come out +0 or -0 depending on order); NaN never passes."""
  got = got.detach().cpu().float()
  ref = ref.detach().cpu().to(torch.float32)
  assert tuple(got.shape) == tuple(ref.shape), f"{what}: shape {tuple(got.shape)} vs {tuple(ref.shape)}"
  bad = got != ref
  n = int(bad.sum())
  if n:
    i = int(bad.flatten().nonzero()[0])
    raise AssertionError(f"{what}: {n} of {bad.numel()} entries differ, first at flat index {i}: "
                         f"{got.flatten()[i].item()!r} vs {ref.flatten()[i].item()!r}")


def bounded(got, ref, bound, what):
  """|got - ref| <= bound, elementwise (bound: a tensor broadcastable to ref, or a scalar)."""
  got = got.detach().cpu().double()
  ref = ref.detach().cpu().double()
  assert tuple(got.shape) == tuple(ref.shape), f"{what}: shape {tuple(got.shape)} vs {tuple(ref.shape)}"
  err = (got - ref).abs()
  excess = err - bound
  assert bool(torch.isfinite(got).all()), f"{what}: non-finite output"
  worst = int(excess.flatten().argmax())
  assert float(excess.flatten()[worst]) <= 0.0, (
      f"{what}: error {err.flatten()[worst].item():.3e} exceeds its bound "
      f"{(bound if isinstance(bound, float) else torch.as_tensor(bound).expand_as(err).flatten()[worst].item()):.3e} at flat index {worst}")


# ------------------------------------------------------------------------------------------------ reduce_partials
N_ROWS = [1, 7, 63, 64, 65, 255, 256, 257, 592, 940, 1376, 3666]
LENS = [1, 32, 64, 289, 512, 513, 865, 1152, 2400]


@pytest.mark.parametrize("n", N_ROWS)
def test_reduce_partials_exact(n):
  """[n, len] integer partials -> mul * column sums.  Reference: closed form (float64 sum, one rounding of sum * fp32(mul)).
  Bit-exact.  n >= 64 with len <= 512 takes reduce_partials_narrow_kernel (4-way unrolled main loop over 256-row steps and a
  64-row remainder loop; n = 64, 65, 255, 256, 257 sit on its boundaries), everything else reduce_partials_kernel.  The n of
  the KITTI step: 592 (grid-capped BN / bias partials), 940 (refine_in tiles), 1376 and 3666 (32->1 conv partial rows)."""
  for ln in LENS:
    part = ints((n, ln), -1000, 1000, seed=n * 10007 + ln)
    pd = part.to(DEV)
    s = part.double().sum(0)
    kern = "reduce_partials_narrow_kernel" if (n >= 64 and ln <= 512) else "reduce_partials_kernel"
    for mul in (1.0, 0.1, -0.375):
      exact(ops.reduce_partials(pd, mul), s * float(np.float32(mul)), f"{kern} n={n} len={ln} mul={mul}")


@pytest.mark.parametrize("taps", [9, 27])
@pytest.mark.parametrize("n", [1, 63, 257, 592])
def test_reduce_wgrad_partials_layout(n, taps):
  """[n][taps][32 ci][32 co] integer partials -> weight gradient in PyTorch's [co][ci][(kd,)kh,kw] layout.  Reference: float64
  sum + permute (closed form).  Bit-exact."""
  part = ints((n, taps * 1024), -1000, 1000, seed=31 * n + taps)
  wshape = (32, 32, 3, 3) if taps == 9 else (32, 32, 3, 3, 3)
  ref = part.double().sum(0).view(taps, 32, 32).permute(2, 1, 0).reshape(wshape)
  exact(ops.reduce_wgrad_partials(part.to(DEV), taps, wshape), ref, f"reduce_partials_kernel (wgrad layout) n={n} taps={taps}")


# ------------------------------------------------------------------------------------------------ BatchNorm + LeakyReLU backward
# npos: 1; 986 (fewer than 64 partial rows); 16320; 18944 = 592 blocks x 256 threads / 8 float4 per position (the grid cap)
# and 18945, one past it; two 94x78 halves; the 24x47x156 cost volume; the 376x1248 refinement (25 grid-stride iterations).
BN_NPOS = [1, 986, 16320, 18944, 18945, 2 * 7332, 24 * 47 * 156, 376 * 1248]


def bn_lrelu_bwd_closed_form(z, dy, scale, shift, mean, invstd, train, lrelu):
  """float64: du = dy * LeakyReLU'(z*scale + shift); zhat = (z - mean) * invstd;
  dz = scale * (du - train * (mean(du) + zhat * mean(du * zhat))).  Returns dz, dgamma, dbeta, dbias and the sums of
  |terms| of the three reductions."""
  z, dy = z.double(), dy.double()
  u = z * scale.double() + shift.double()
  du = torch.where((u <= 0) & lrelu, dy * LRELU, dy)
  zhat = (z - mean.double()) * invstd.double()
  dbeta, dgamma = du.sum(0), (du * zhat).sum(0)
  n = z.shape[0]
  dz = scale.double() * ((du - dbeta / n - zhat * (dgamma / n)) if train else du)
  return dz, dgamma, dbeta, dz.sum(0), (du * zhat).abs().sum(0), du.abs().sum(0), dz.abs().sum(0)


# fp32 summation bound of the reductions: each thread adds <= 25 grid-stride terms, then 32 thread sums are added serially, all
# in fp32 (the partial rows are then summed in double): |error| <= (25 + 31) * 2^-24 * sum|terms| = 3.4e-6 * sum|terms|.
SUM_RTOL = 1e-5


@pytest.mark.parametrize("lrelu", [False, True])
@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("npos", BN_NPOS)
def test_bn_lrelu_bwd_exact(npos, train, lrelu):
  """Integer z / dy, integer mean, power-of-two invstd, dyadic scale and an odd multiple of 1/32 as shift (so z*scale + shift
  is never 0: every LeakyReLU mask is unambiguous).  Reference: closed form in float64.
  LeakyReLU off: dgamma and dbeta are bit-exact; so are dz and dbias in eval mode.  In train mode dz uses fp32(1/npos): bound
  1e-5 of max|dz| (a few ulps of the largest term), dbias as a sum of those dz by SUM_RTOL.  LeakyReLU on: dy * 0.2f rounds,
  so dz gets 1e-5 of max|dz| and the sums SUM_RTOL."""
  s = npos % 9973
  z, dy = ints((npos, 32), -8, 8, s + 1), ints((npos, 32), -4, 4, s + 2)
  mean = ints((32,), -2, 2, s + 3)
  invstd = 2.0 ** ints((32,), -2, 1, s + 4)
  scale = ints((32,), 1, 16, s + 5) / 16 * torch.where(ints((32,), 0, 1, s + 6) > 0, 1.0, -1.0)
  shift = (2 * ints((32,), -16, 15, s + 7) + 1) / 32
  dz_r, dg_r, db_r, dbias_r, dg_abs, db_abs, dbias_abs = bn_lrelu_bwd_closed_form(z, dy, scale, shift, mean, invstd, train, lrelu)
  dz, dgamma, dbeta, dbias = ops.bn_lrelu_bwd(z.to(DEV), dy.to(DEV), scale.to(DEV), shift.to(DEV), mean.to(DEV), invstd.to(DEV),
                                              train, lrelu=lrelu)
  what = f"bn_lrelu_bwd npos={npos} train={train} lrelu={lrelu}"
  if not lrelu:
    exact(dgamma, dg_r, f"{what}: dgamma (bn_lrelu_bwd_reduce_kernel)")
    exact(dbeta, db_r, f"{what}: dbeta (bn_lrelu_bwd_reduce_kernel)")
  else:
    bounded(dgamma, dg_r, SUM_RTOL * dg_abs, f"{what}: dgamma (bn_lrelu_bwd_reduce_kernel)")
    bounded(dbeta, db_r, SUM_RTOL * db_abs, f"{what}: dbeta (bn_lrelu_bwd_reduce_kernel)")
  if not lrelu and not train:
    exact(dz, dz_r, f"{what}: dz (bn_lrelu_bwd_apply_kernel)")
    exact(dbias, dbias_r, f"{what}: dbias (bn_lrelu_bwd_apply_kernel)")
  else:
    bounded(dz, dz_r, 1e-5 * dz_r.abs().max().item(), f"{what}: dz (bn_lrelu_bwd_apply_kernel)")
    bounded(dbias, dbias_r, SUM_RTOL * dbias_abs, f"{what}: dbias (bn_lrelu_bwd_apply_kernel)")


@pytest.mark.parametrize("lrelu", [False, True])
@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("npos", BN_NPOS)
def test_bn_lrelu_bwd_vs_autograd(npos, train, lrelu):
  """Random floats against float64 autograd of leaky_relu(batch_norm(z)): in train mode the batch statistics stay in the graph,
  in eval mode the running statistics are constants.  The kernel gets fp32 roundings of the same statistics.  z is pushed at
  least 1e-3 away from the kink first.  Bounds: dz 1e-5 of max|dz| (fp32 arithmetic on O(1) terms); dgamma, dbeta, dbias
  SUM_RTOL of the sum of |terms| (see SUM_RTOL)."""
  s = npos % 7919
  gamma = (rnd(32, seed=s + 3).abs() + 0.5) * torch.where(rnd(32, seed=s + 4) > -0.5, 1.0, -1.0)
  beta = rnd(32, seed=s + 5) * 0.5
  beta = torch.where(beta.abs() < 0.05, beta + 0.1, beta)              # npos = 1 in train mode: u = beta exactly
  rm, rv = rnd(32, seed=s + 6) * 0.3, rnd(32, seed=s + 7).abs() + 0.5
  dy = rnd(npos, 32, seed=s + 2)
  z = rnd(npos, 32, seed=s + 1) * 1.5 + 0.25

  def stats(z):
    z64 = z.double()
    if train:
      mu, var = z64.mean(0), ((z64 - z64.mean(0)) ** 2).mean(0)
    else:
      mu, var = rm.double(), rv.double()
    return mu, 1.0 / torch.sqrt(var + BN_EPS)

  mu, inv = stats(z)
  sc = gamma.double() * inv
  u = (z.double() - mu) * sc + beta.double()
  away = torch.where(u >= 0, 1.0, -1.0) * torch.sign(sc) * 2e-3 / sc.abs()
  z = torch.where(u.abs() < 1e-3, z.double() + away, z.double()).float()
  mu, inv = stats(z)
  sc = gamma.double() * inv
  u = (z.double() - mu) * sc + beta.double()
  assert u.abs().min().item() >= 5e-4, "test setup: activation too close to the LeakyReLU kink"

  z64 = z.double().requires_grad_()
  g64, b64 = gamma.double().requires_grad_(), beta.double().requires_grad_()
  if train:
    m = z64.mean(0)
    y = (z64 - m) / torch.sqrt(((z64 - m) ** 2).mean(0) + BN_EPS) * g64 + b64
  else:
    y = (z64 - rm.double()) / torch.sqrt(rv.double() + BN_EPS) * g64 + b64
  if lrelu:
    y = F.leaky_relu(y, LRELU)
  y.backward(dy.double())
  du = dy.double() * torch.where((u <= 0) & lrelu, LRELU, 1.0)
  zhat = (z.double() - mu) * inv
  f32 = lambda t: t.float().to(DEV)
  dz, dgamma, dbeta, dbias = ops.bn_lrelu_bwd(f32(z), f32(dy), f32(sc), f32(beta.double() - mu * sc), f32(mu), f32(inv), train,
                                              lrelu=lrelu)
  what = f"bn_lrelu_bwd (random) npos={npos} train={train} lrelu={lrelu}"
  bounded(dz, z64.grad, 1e-5 * z64.grad.abs().max().item(), f"{what}: dz (bn_lrelu_bwd_apply_kernel)")
  bounded(dgamma, g64.grad, SUM_RTOL * (du * zhat).abs().sum(0), f"{what}: dgamma (bn_lrelu_bwd_reduce_kernel)")
  bounded(dbeta, b64.grad, SUM_RTOL * du.abs().sum(0), f"{what}: dbeta (bn_lrelu_bwd_reduce_kernel)")
  bounded(dbias, z64.grad.sum(0), SUM_RTOL * z64.grad.abs().sum(0) + 1e-6 * z64.grad.abs().max().item(),
          f"{what}: dbias (bn_lrelu_bwd_apply_kernel)")


# ------------------------------------------------------------------------------------------------ channel_sum
@pytest.mark.parametrize("B,D,H,W", [(1, 1, 188, 624), (2, 1, 188, 624), (1, 1, 94, 312), (2, 1, 94, 312), (1, 1, 47, 156),
                                     (2, 1, 47, 156), (2, 24, 47, 156), (1, 1, 376, 1248), (2, 1, 376, 1248), (1, 1, 1, 1),
                                     (1, 1, 3, 5)])
def test_channel_sum_exact(B, D, H, W):
  """Per-channel sums of a channels-last [B,(D),H,W,32] tensor (the bias gradients of the plain convolutions).  Integer data;
  reference: float64 sum.  Bit-exact."""
  x = ints((B, D, H, W, 32), -8, 8, seed=B * 7 + H * 3 + W)
  if D == 1:
    x = x[:, 0]
  exact(ops.channel_sum(x.contiguous().to(DEV)), x.double().reshape(-1, 32).sum(0), f"channel_sum_kernel {B}x{D}x{H}x{W}")


# ------------------------------------------------------------------------------------------------ 32->1 conv backward (tap form)
def conv32to1_ref(x, w, g, ntaps):
  """float64 autograd of F.conv3d / F.conv2d(32 -> 1, pad 1): (dx [B,32,(D),H,W], dw [1,32,*k], db [1])."""
  x64, w64 = x.double().requires_grad_(), w.double().requires_grad_()
  b64 = torch.zeros(1, dtype=torch.float64, requires_grad=True)
  out = (F.conv3d if ntaps == 27 else F.conv2d)(x64, w64, b64, padding=1).squeeze(1)
  out.backward(g.double())
  return x64.grad, w64.grad, b64.grad


TAPS_BWD_CASES = [  # ntaps, B, D, H, W: the head at 1 and 2 x 24x47x156, the refine tail at 376x1248, H = 1, W = 1, npos = 1,
                    # npos not a multiple of 128
  (27, 1, 24, 47, 156), (27, 2, 24, 47, 156), (27, 1, 24, 1, 156), (27, 1, 6, 5, 1), (27, 1, 1, 1, 1), (27, 1, 5, 7, 11),
  (9, 1, 1, 376, 1248), (9, 2, 1, 1, 130), (9, 1, 1, 67, 1), (9, 1, 1, 1, 1), (9, 2, 1, 13, 17),
]


def taps_bwd_inputs(ntaps, B, D, H, W, exact_data, seed):
  xs = (B, 32, D, H, W) if ntaps == 27 else (B, 32, H, W)
  gs = (B, D, H, W) if ntaps == 27 else (B, H, W)
  ws = (1, 32, 3, 3, 3) if ntaps == 27 else (1, 32, 3, 3)
  if exact_data:
    return ints(xs, -2, 2, seed), dyadic(ws, 8, 16, seed + 1), ints(gs, -4, 4, seed + 2)
  return rnd(*xs, seed=seed), rnd(*ws, seed=seed + 1, scale=0.2), rnd(*gs, seed=seed + 2)


@pytest.mark.parametrize("ntaps,B,D,H,W", TAPS_BWD_CASES)
def test_conv_c32_taps_bwd_exact(ntaps, B, D, H, W):
  """dx, dw, db of the 32->1 convolution from its output gradient (conv3d_alone, refinement conv2d_out).  Integer x and g,
  weights k/16.  Reference: float64 autograd of F.conv3d / F.conv2d.  Bit-exact."""
  x, w, g = taps_bwd_inputs(ntaps, B, D, H, W, True, seed=ntaps * 100 + H)
  dx_r, dw_r, db_r = conv32to1_ref(x, w, g, ntaps)
  dx, dw, db = ops.conv_c32_taps_bwd(cl(x), w.to(DEV), g.to(DEV), ntaps)
  what = f"conv_c32_taps_bwd_kernel<{ntaps}> {B}x{D}x{H}x{W}"
  exact(uncl(dx), dx_r, what + ": dx")
  exact(dw, dw_r, what + ": dw")
  exact(db, db_r, what + ": db")


@pytest.mark.parametrize("ntaps,B,D,H,W", [(27, 1, 24, 47, 156), (9, 1, 1, 376, 1248)])
def test_conv_c32_taps_bwd_random(ntaps, B, D, H, W):
  """Random floats.  Reference: float64 autograd; the same computation on |x|, |w|, |g| gives each output's sum of |terms|.
  Bound 1e-5 of that: dx is an ntaps-term fp32 FMA chain (<= 27 * 2^-24), dw a 128-term fp32 FMA chain per block summed in
  double (<= 128 * 2^-24 = 7.6e-6), db a 128-lane fp32 tree."""
  x, w, g = taps_bwd_inputs(ntaps, B, D, H, W, False, seed=7)
  dx_r, dw_r, db_r = conv32to1_ref(x, w, g, ntaps)
  dx_a, dw_a, db_a = conv32to1_ref(x.abs(), w.abs(), g.abs(), ntaps)
  dx, dw, db = ops.conv_c32_taps_bwd(cl(x), w.to(DEV), g.to(DEV), ntaps)
  what = f"conv_c32_taps_bwd_kernel<{ntaps}> (random) {B}x{D}x{H}x{W}"
  bounded(uncl(dx), dx_r, 1e-5 * dx_a, what + ": dx")
  bounded(dw, dw_r, 1e-5 * dw_a, what + ": dw")
  bounded(db, db_r, 1e-5 * db_a, what + ": db")


# ------------------------------------------------------------------------------------------------ soft-argmin backward
@pytest.mark.parametrize("grads", ["dpred", "dpred+extra", "extra"])
@pytest.mark.parametrize("spread", [1.0, 40.0, 200.0])
@pytest.mark.parametrize("D", [1, 6, 24, 48])
def test_softargmin_bwd(D, spread, grads):
  """dcost of pred = sum_d d * softmax(cost)_d (+ dcost_extra, the gradient arriving on the cost volume itself), given the
  `pred` of the training forward kernel (snb_conv3d_out_softargmin, fed a cost volume through an identity 32->1 tap).
  Costs uniform in [0, spread): spread 1 is soft, 40 and 200 are sharp (most exp terms tiny or underflowing).  Reference:
  float64 autograd of the softmax expectation.  Bound 1e-5 of max|dcost|: fp32 exp / division / product on O(1) terms."""
  B, H, W = 2, 13, 37
  cost = torch.rand(B, D, H, W, generator=gen(D * 13 + int(spread))) * spread
  x = torch.zeros(B, D, H, W, 32)
  x[..., 0] = cost
  wid = torch.zeros(1, 32, 3, 3, 3)
  wid[0, 0, 1, 1, 1] = 1.0
  cost_k, pred_k, _ = ops.conv3d_out_softargmin(x.to(DEV), wid.to(DEV), torch.zeros(1, device=DEV), want_cost=True)
  exact(cost_k, cost, "conv3d_out_softargmin identity tap: cost")
  dpred = rnd(B, H, W, seed=3) if "dpred" in grads else None
  extra = rnd(B, D, H, W, seed=4) * 0.1 if "extra" in grads else None
  c64 = cost.double().requires_grad_()
  pred64 = (F.softmax(c64, 1) * torch.arange(D, dtype=torch.float64).view(1, D, 1, 1)).sum(1)
  loss = torch.zeros((), dtype=torch.float64)
  if dpred is not None:
    loss = loss + (pred64 * dpred.double()).sum()
  if extra is not None:
    loss = loss + (c64 * extra.double()).sum()
  loss.backward()
  ref = c64.grad
  got = ops.softargmin_bwd(cost_k, pred_k, None if dpred is None else dpred.to(DEV), None if extra is None else extra.to(DEV))
  bounded(got, ref, 1e-5 * ref.abs().max().item() + 1e-30, f"softargmin_bwd_kernel D={D} spread={spread} {grads}")


# ------------------------------------------------------------------------------------------------ ReLU backward
@pytest.mark.parametrize("n", [1, 1000, 2 * 188 * 621, 376 * 1248])
def test_relu_bwd_bit_exact(n):
  """dres = dout where out > 0, else +0 (refinement output ReLU).  Outputs exactly +0, -0, a positive subnormal and negative
  values; dout with -0 entries.  Reference: torch.where.  Bit-exact including the sign of zero."""
  out = rnd(n, seed=n)
  out[::7] = 0.0
  out[3::11] = -0.0
  out[5::13] = 1e-40
  dout = rnd(n, seed=n + 1)
  dout[2::5] = -0.0
  got = ops.relu_bwd(out.to(DEV), dout.to(DEV)).cpu()
  ref = torch.where(out > 0, dout, torch.zeros_like(dout))
  assert torch.equal(got.view(torch.int32), ref.view(torch.int32)), f"relu_bwd_kernel n={n}: bits differ"


# ------------------------------------------------------------------------------------------------ first-layer weight gradients
def conv5x5s2_c3_dw_ref(img, dy):
  """float64 autograd of F.conv2d(img [B,3,H,W], w [32,3,5,5], stride 2, pad 2) given dy [B,OH,OW,32] -> dw [32,3,5,5]."""
  w64 = torch.zeros(32, 3, 5, 5, dtype=torch.float64, requires_grad=True)
  F.conv2d(img.double(), w64, None, stride=2, padding=2).backward(dy.double().permute(0, 3, 1, 2))
  return w64.grad


@pytest.mark.parametrize("B,H,W", [(1, 376, 1248), (2, 376, 1248), (1, 375, 1242), (1, 1, 1), (1, 2, 2), (1, 3, 5), (1, 17, 130),
                                   (1, 130, 17)])
def test_conv5x5s2_c3_wgrad_exact(B, H, W):
  """Weight gradient of downsample[0] (3 -> 32, 5x5, stride 2, pad 2).  Image k/256, integer dy: every per-tile fp32 sum is
  exact, the partial rows are summed in double and rounded once.  Reference: float64 autograd.  Bit-exact.  17x130 (9x65
  output) has partial 8x64 tiles in both axes, 130x17 (65x9) is taller than wide; 376x1248 runs 240 tiles per image."""
  img = ints((B, 3, H, W), 0, 255, seed=H + W) / 256
  OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
  dy = ints((B, OH, OW, 32), -4, 4, seed=H * W)
  exact(ops.conv5x5s2_c3_wgrad(img.to(DEV), dy.to(DEV)), conv5x5s2_c3_dw_ref(img, dy), f"conv_small_wgrad_kernel<3,5,2> {B}x{H}x{W}")


def test_conv5x5s2_c3_wgrad_random():
  """Random image and dy at 375x1242.  Reference: float64 autograd.  Bound 1e-5 of max|dw|: 512-term fp32 FMA chains per
  tile, summed in double."""
  img = torch.rand(1, 3, 375, 1242, generator=gen(1))
  dy = rnd(1, 188, 621, 32, seed=2)
  ref = conv5x5s2_c3_dw_ref(img, dy)
  close(ops.conv5x5s2_c3_wgrad(img.to(DEV), dy.to(DEV)).cpu().double(), ref, 1e-5, "conv_small_wgrad_kernel<3,5,2> (random)")


@pytest.mark.parametrize("B,h,w,H,W", [(1, 47, 156, 376, 1248), (2, 47, 156, 376, 1248), (1, 47, 156, 375, 1242), (1, 1, 1, 3, 5)])
def test_refine_in_wgrad(B, h, w, H, W):
  """Weight gradient of the refinement's Conv2d(4 -> 32) over [W/w * bilinear(coarse), rgb].  Reference: float64, upsampling
  included (bilinear_matrix: at 376x1248 these are the exact weights, at the ragged 375x1242 the fp32 source coordinates of
  the forward).  Bound 1e-5 of max|dw|: 512-term fp32 FMA chains per tile, summed in double.  Checked per input channel (the
  disparity channel is ~100x larger than the colour channels)."""
  coarse = torch.rand(B, h, w, generator=gen(1)) * 20
  rgb = torch.rand(B, 3, H, W, generator=gen(2))
  dz = rnd(B, H, W, 32, seed=3)
  mul = float(np.float32(W) / np.float32(w))
  up = (mul * torch.einsum("yi,bij,xj->byx", bilinear_matrix(H, h), coarse.double(), bilinear_matrix(W, w))).unsqueeze(1)
  w64 = torch.zeros(32, 4, 3, 3, dtype=torch.float64, requires_grad=True)
  F.conv2d(torch.cat([up, rgb.double()], 1), w64, None, padding=1).backward(dz.double().permute(0, 3, 1, 2))
  got = ops.refine_in_wgrad(coarse.to(DEV), rgb.to(DEV), dz.to(DEV)).cpu().double()
  for c in range(4):
    close(got[:, c], w64.grad[:, c], 1e-5, f"conv_small_wgrad_kernel<4,3,1> {B}x{h}x{w}->{H}x{W} input channel {c}")


# ------------------------------------------------------------------------------------------------ polyphase split / merge
PHASE_SHAPES = [(1, 1, 1), (1, 1, 2), (1, 2, 1), (2, 3, 5), (1, 4, 6), (1, 7, 8), (2, 188, 624), (1, 188, 621), (1, 187, 623)]


@pytest.mark.parametrize("B,H,W", PHASE_SHAPES)
def test_phase_split_merge_exact(B, H, W):
  """phase_split: phase a*2+b = x[:, a::2, b::2] zero padded to ceil(H/2) x ceil(W/2); phase_merge: its inverse (the data
  gradient of the 5x5 stride-2 layers).  Reference: slicing.  Bit-exact."""
  OH, OW = (H + 1) // 2, (W + 1) // 2
  x = rnd(B, H, W, 32, seed=H * W)
  ref = torch.zeros(4, B, OH, OW, 32)
  for a in (0, 1):
    for b in (0, 1):
      s = x[:, a::2, b::2]
      ref[a * 2 + b, :, :s.shape[1], :s.shape[2]] = s
  exact(ops.phase_split(x.to(DEV)), ref, f"phase_split_kernel {B}x{H}x{W}")
  ph = rnd(4, B, OH, OW, 32, seed=H * W + 1)
  ref = torch.empty(B, H, W, 32)
  for a in (0, 1):
    for b in (0, 1):
      na, nb = len(range(a, H, 2)), len(range(b, W, 2))
      ref[:, a::2, b::2] = ph[a * 2 + b, :, :na, :nb]
  exact(ops.phase_merge(ph.to(DEV), H, W), ref, f"phase_merge_kernel {B}x{H}x{W}")


@pytest.mark.parametrize("B,H,W", [(1, 376, 1248), (2, 376, 1248), (1, 375, 1247), (1, 4, 8), (2, 36, 100)])
def test_conv5x5s2_c3_phases_exact(B, H, W):
  """downsample[0] written straight into polyphase form (the KITTI inference path: its 188x624 output is even) against
  phase_split of the plain layer's output.  Same arithmetic, other addressing: bit-exact."""
  img = torch.rand(B, 3, H, W, generator=gen(1))
  w, b = rnd(32, 3, 5, 5, seed=2, scale=0.2).to(DEV), rnd(32, seed=3).to(DEV)
  ref = ops.phase_split(ops.conv5x5s2_c3(img.to(DEV), w, b))
  exact(ops.conv5x5s2_c3_phases(img.to(DEV), w, b), ref, f"snb_conv5x5s2_c3_phases {B}x{H}x{W}")


# ------------------------------------------------------------------------------------------------ cost volume / upsampling adjoints
@pytest.mark.parametrize("B", [1, 2])
def test_cost_volume_bwd_exact(B):
  """Adjoint of the difference cost volume at the KITTI size (32 x 47x156, D = 24).  Integer gradients; reference: float64
  autograd of the oracle's cost volume.  Bit-exact."""
  H, W, D = 47, 156, 24
  L = torch.zeros(B, 32, H, W, dtype=torch.float64, requires_grad=True)
  R = torch.zeros(B, 32, H, W, dtype=torch.float64, requires_grad=True)
  g = ints((B, 32, D, H, W), -4, 4, seed=B)
  O.cost_volume(L, R, D).backward(g.double())
  dl, dr = ops.cost_volume_bwd(cl(g))
  exact(uncl(dl), L.grad, f"cost_volume_bwd_kernel B={B}: dleft")
  exact(uncl(dr), R.grad, f"cost_volume_bwd_kernel B={B}: dright")


def upsample_adjoint_ref(g, h, w, mul):
  x = torch.zeros(g.shape[0], 1, h, w, dtype=torch.float64, requires_grad=True)
  (mul * F.interpolate(x, size=tuple(g.shape[-2:]), mode="bilinear", align_corners=False)).squeeze(1).backward(g.double())
  return x.grad.squeeze(1)


def bilinear_matrix(n_out, n_in):
  """float64 [n_out, n_in] bilinear weights (align_corners=False) at the fp32 source coordinates of PyTorch's float kernels
  and of this library: s = fp32(n_in / n_out) * (d + 0.5) - 0.5 rounded once to fp32 (one FMA), clamped at 0.  At a
  non-integer ratio these coordinates are a few ulps of s (s up to 156) away from the exact ones, which moves an
  upsampled value by ~1e-5 of its magnitude: a property of fp32 bilinear upsampling, not of a kernel."""
  sc = float(np.float32(n_in) / np.float32(n_out))
  s = (sc * (torch.arange(n_out, dtype=torch.float64) + 0.5) - 0.5).float().clamp(min=0)
  i0 = s.long().clamp(max=n_in - 1)
  i1 = torch.where(i0 < n_in - 1, i0 + 1, i0)
  lam = s - i0.float()
  A = torch.zeros(n_out, n_in, dtype=torch.float64)
  rows = torch.arange(n_out)
  A.index_put_((rows, i0), (1 - lam).double(), accumulate=True)
  A.index_put_((rows, i1), lam.double(), accumulate=True)
  return A


def test_upsample_bilinear_bwd_kitti_exact():
  """Adjoint of the x8 upsampling 47x156 -> 376x1248 (ratio exactly 1/8: every bilinear weight is a multiple of 1/16).
  Integer gradients; reference: float64 autograd of F.interpolate.  Bit-exact."""
  g = ints((2, 376, 1248), -4, 4, seed=5)
  exact(ops.upsample_bilinear_bwd(g.to(DEV), 47, 156, 8.0), upsample_adjoint_ref(g, 47, 156, 8.0),
        "upsample_bilinear_bwd_kernel 47x156 <- 376x1248")


def test_upsample_bilinear_bwd_ragged():
  """47x156 -> 375x1242, the ragged ratio.  Reference: the float64 adjoint Ay^T g Ax of bilinear_matrix (fp32 source
  coordinates, as the forward upsampling uses them).  Bound 1e-5 of max|din|: each weight product is rounded once in fp32 and
  a coarse pixel sums ~60 fine-pixel terms in fp32."""
  g = rnd(2, 375, 1242, seed=6)
  mul = float(np.float32(1242 / 156))
  ref = mul * torch.einsum("yi,byx,xj->bij", bilinear_matrix(375, 47), g.double(), bilinear_matrix(1242, 156))
  close(ops.upsample_bilinear_bwd(g.to(DEV), 47, 156, mul).cpu().double(), ref, 1e-5, "upsample_bilinear_bwd_kernel 47x156 <- 375x1242")


# ------------------------------------------------------------------------------------------------ composite layers (autograd Functions)
def with_backend(name, fn):
  old = fused.CONV_BACKEND
  fused.set_conv_backend(name)
  try:
    return fn()
  finally:
    fused.set_conv_backend(old)


def randomize_bn(bn, seed):
  with torch.no_grad():
    bn.weight.copy_(rnd(32, seed=seed).abs() + 0.5); bn.bias.copy_(rnd(32, seed=seed + 1))
    bn.running_mean.copy_(rnd(32, seed=seed + 2) * 0.1); bn.running_var.copy_(rnd(32, seed=seed + 3).abs() + 0.5)


# shape, dil, residual: the refinement's dilated residual blocks at 376x1248, a feature block at B = 2 x 47x156, a cost filter
# layer at 24x47x156
CBL_CASES = [((1, 32, 376, 1248), 1, True), ((1, 32, 376, 1248), 2, True), ((1, 32, 376, 1248), 4, True),
             ((1, 32, 376, 1248), 8, True), ((2, 32, 47, 156), 1, True), ((1, 32, 24, 47, 156), 1, False)]


@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("shape,dil,residual", CBL_CASES)
def test_conv_bn_lrelu_backward_kitti(shape, dil, residual, training):
  """ConvBnLrelu (conv + BN + LeakyReLU [+ x]) forward and backward on the product "ws" back end and on "tc3".  Integer x and
  weights k/16 make every convolution sum exact, so z is bit-identical on CPU and GPU; the BN pre-activation is checked to sit
  >= 1e-5 from the kink (a flipped mask there would be a legitimate O(1) difference).  Reference: float64 CPU autograd, one per
  case, shared by both back ends (an fp32 CPU reference is itself ~2e-5 off in dW at 376x1248, where every entry sums 470k
  products); bounds as test_gpu_backward.test_conv_bn_lrelu_backward."""
  three_d = len(shape) == 5
  x = ints(shape, -2, 2, seed=1)
  torch.manual_seed(5)
  conv = (torch.nn.Conv3d(32, 32, 3, padding=1) if three_d else torch.nn.Conv2d(32, 32, 3, padding=dil, dilation=dil))
  with torch.no_grad():
    conv.weight.copy_(dyadic(conv.weight.shape, 2, 16, seed=3))
    conv.bias.copy_(dyadic((32,), 4, 8, seed=4))
  bn = torch.nn.BatchNorm3d(32) if three_d else torch.nn.BatchNorm2d(32)
  randomize_bn(bn, 7 + dil)
  gconv0, gbn0 = copy.deepcopy(conv), copy.deepcopy(bn)
  conv, bn = conv.double(), bn.double()
  conv.train(training); bn.train(training)
  x64 = x.double().requires_grad_()
  u = bn(conv(x64))
  assert u.detach().abs().min().item() >= 1e-5, "test setup: BN output too close to the LeakyReLU kink"
  y = F.leaky_relu(u, LRELU)
  if residual:
    y = x64 + y
  gy = rnd(*shape, seed=2)
  y.backward(gy.double())
  for backend in ("ws", "tc3"):
    gconv, gbn = copy.deepcopy(gconv0).to(DEV), copy.deepcopy(gbn0).to(DEV)
    gbn.train(training)
    xg = cl(x).requires_grad_()

    def run():
      yg = Fn.conv_bn_lrelu_autograd(xg, gconv, gbn, dil, residual, training)
      yg.backward(cl(gy))
      return yg
    yg = with_backend(backend, run)
    what = f"ConvBnLrelu {backend} {tuple(shape)} dil={dil} train={training}"
    close(uncl(yg.detach()), y.detach(), 1e-5, what + ": forward")
    close(uncl(xg.grad), x64.grad, 2e-5, what + ": dx")
    close(gconv.weight.grad.cpu(), conv.weight.grad, 2e-5, what + ": dW")
    close(gbn.weight.grad.cpu(), bn.weight.grad, 2e-5, what + ": dgamma")
    close(gbn.bias.grad.cpu(), bn.bias.grad, 2e-5, what + ": dbeta")
    if training:   # the conv-bias gradient under batch-stat BN is mathematically zero: compare absolutely
      assert gconv.bias.grad.abs().max().item() <= 1e-3 * (conv.weight.grad.abs().max().item() + 1.0), what + ": dbias"
    else:
      close(gconv.bias.grad.cpu(), conv.bias.grad, 2e-5, what + ": dbias")


@pytest.mark.parametrize("H,W", [(188, 624), (188, 621)])
def test_conv5x5s2_c32_backward_exact(H, W):
  """ConvC32 5x5 stride 2 (downsample[1]) from 188x624 and the odd 188x621.  On "ws" the data gradient is four polyphase 3x3
  convolutions + phase_merge; on "tc3" the same through the 3xTF32 kernels.  Integer x and dy, weights k/16: every product and
  sum is exact in fp32 and in both operand splits.  Reference: float64 autograd.  Bit-exact (forward, dx, dW, dbias)."""
  x = ints((1, 32, H, W), -2, 2, seed=H + W)
  w, b = dyadic((32, 32, 5, 5), 2, 16, seed=3), dyadic((32,), 4, 8, seed=4)
  OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
  dy = ints((1, 32, OH, OW), -2, 2, seed=5)
  x64, w64, b64 = x.double().requires_grad_(), w.double().requires_grad_(), b.double().requires_grad_()
  y64 = F.conv2d(x64, w64, b64, stride=2, padding=2)
  y64.backward(dy.double())
  for backend in ("ws", "tc3"):
    conv = torch.nn.Conv2d(32, 32, 5, stride=2, padding=2).to(DEV)
    with torch.no_grad():
      conv.weight.copy_(w); conv.bias.copy_(b)
    xg = cl(x).requires_grad_()

    def run():
      yg = Fn.ConvC32.apply(xg, conv.weight, conv.bias, conv, 5, 2)
      yg.backward(cl(dy))
      return yg
    yg = with_backend(backend, run)
    what = f"ConvC32 5x5s2 {backend} 1x{H}x{W}"
    exact(uncl(yg.detach()), y64.detach(), what + ": forward")
    exact(uncl(xg.grad), x64.grad, what + ": dx (polyphase dgrad + phase_merge)")
    exact(conv.weight.grad, w64.grad, what + ": dW")
    exact(conv.bias.grad, b64.grad, what + ": dbias (channel_sum)")


def test_conv3d_out_softargmin_backward_kitti():
  """Conv3dOutSoftargmin (conv3d_alone 32 -> 1 + softmax + expectation) at 2 x 24x47x156: softargmin_bwd + conv_c32_taps_bwd
  through the autograd Function.  Reference: float64 CPU autograd.  dx and dw: 3e-5 of their magnitude, as
  test_gpu_backward.test_head_backward.  db sums 352k entries of dcost whose soft-argmin parts cancel per pixel, so it is
  bounded by SUM_RTOL of sum|dcost| (fp32 dcost, 128-position fp32 block sums, then double)."""
  B, D, H, W = 2, 24, 47, 156
  x = rnd(B, 32, D, H, W, seed=1)
  torch.manual_seed(5)
  conv = torch.nn.Conv3d(32, 1, 3, padding=1)
  with torch.no_grad():
    conv.weight.mul_(10.0)
  gconv = copy.deepcopy(conv).to(DEV)
  conv = conv.double()
  x64 = x.double().requires_grad_()
  cost = conv(x64).squeeze(1)
  cost.retain_grad()
  pred = O.soft_argmin(cost)
  gp, gc = rnd(B, H, W, seed=2), rnd(B, D, H, W, seed=3) * 0.1
  ((pred * gp.double()).sum() + (cost * gc.double()).sum()).backward()
  xg = cl(x).requires_grad_()
  cg, pg, _fcs = Fn.Conv3dOutSoftargmin.apply(xg, gconv.weight, gconv.bias)
  ((pg * gp.to(DEV)).sum() + (cg * gc.to(DEV)).sum()).backward()
  close(uncl(xg.grad), x64.grad, 3e-5, "Conv3dOutSoftargmin 2x24x47x156: dx")
  close(gconv.weight.grad.cpu(), conv.weight.grad, 3e-5, "Conv3dOutSoftargmin 2x24x47x156: dw")
  bounded(gconv.bias.grad, conv.bias.grad, SUM_RTOL * cost.grad.abs().sum().item(), "Conv3dOutSoftargmin 2x24x47x156: db")


@pytest.fixture(scope="module")
def kitti_refine_inputs():
  """Coarse 47x156 disparity and 376x1248 guidance image shared by the refinement tests."""
  coarse = torch.rand(1, 47, 156, generator=gen(1)) * 20
  rgb = torch.rand(1, 3, 376, 1248, generator=gen(2))
  return coarse, rgb


@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("bn_bias", [60.0, -60.0])
def test_refine_head_backward_kitti(kitti_refine_inputs, training, bn_bias):
  """RefineHead (upsample + concat + conv 4 -> 32 + BN + LeakyReLU) at 47x156 -> 376x1248 with the BN shift at +-60, so every
  mask is unambiguous.  Reference: float64 CPU autograd.  Forward, dcoarse, dgamma, dbeta: bounds as
  test_gpu_backward.test_refine_head_backward_exact_side_of_kink.  dW: the disparity channel (~90 on average) meets a dz that
  sums to zero per channel in train mode, so dW cancels; its bound is 5e-5 of sum|input * dz| (512-term fp32 FMA chains per
  tile, <= 3.1e-5 of that sum, on an fp32 dz)."""
  coarse0, rgb = kitti_refine_inputs
  B, h, w, H, W = 1, 47, 156, 376, 1248
  torch.manual_seed(5)
  conv = torch.nn.Conv2d(4, 32, 3, padding=1); bn = torch.nn.BatchNorm2d(32)
  randomize_bn(bn, 7)
  with torch.no_grad():
    bn.bias.fill_(bn_bias)
    if not training:
      bn.running_var.fill_(400.0)
  gconv, gbn = copy.deepcopy(conv).to(DEV), copy.deepcopy(bn).to(DEV)
  conv, bn = conv.double(), bn.double()
  bn.train(training); gbn.train(training)
  coarse = coarse0.double().requires_grad_()
  up = F.interpolate(coarse.unsqueeze(1), size=(H, W), mode="bilinear", align_corners=False) * (W / w)
  inp = torch.cat([up, rgb.double()], 1)
  z = conv(inp)
  z.retain_grad()
  y = F.leaky_relu(bn(z), LRELU)
  gy, gu = rnd(B, 32, H, W, seed=3), rnd(B, H, W, seed=4)
  ((y * gy.double()).sum() + (up.squeeze(1) * gu.double()).sum()).backward()
  dw_abs = torch.nn.grad.conv2d_weight(inp.detach().abs(), conv.weight.shape, z.grad.abs(), padding=1)
  cg = coarse0.to(DEV).requires_grad_()
  upg, yg = Fn.refine_head_autograd(cg, rgb.to(DEV), gconv, gbn, training)
  ((yg * cl(gy)).sum() + (upg * gu.to(DEV)).sum()).backward()
  what = f"RefineHead 376x1248 shift={bn_bias} train={training}"
  close(uncl(yg.detach()), y.detach(), 1e-5, what + ": forward")
  close(cg.grad.cpu(), coarse.grad, 3e-5, what + ": dcoarse")
  bounded(gconv.weight.grad, conv.weight.grad, 5e-5 * dw_abs, what + ": dW")
  close(gbn.weight.grad.cpu(), bn.weight.grad, 3e-5, what + ": dgamma")
  close(gbn.bias.grad.cpu(), bn.bias.grad, 3e-5, what + ": dbeta")


def test_refine_tail_backward_kitti():
  """RefineTail (conv 32 -> 1 + upsampled disparity + ReLU) at 376x1248: relu_bwd + conv_c32_taps_bwd<9> through the autograd
  Function.  The upsampled disparity is pushed so that every pre-activation sits >= 1e-3 from the ReLU kink.  Reference: fp32
  CPU autograd; bounds as test_gpu_backward.test_refine_tail_backward."""
  B, H, W = 1, 376, 1248
  x = rnd(B, 32, H, W, seed=1).requires_grad_()
  torch.manual_seed(5)
  conv = torch.nn.Conv2d(32, 1, 3, padding=1)
  gconv = copy.deepcopy(conv).to(DEV)
  up = rnd(B, H, W, seed=2) * 2
  with torch.no_grad():
    pre = up + conv(x).squeeze(1)
    up = up + torch.where(pre.abs() < 1e-3, torch.where(pre >= 0, 2e-3, -2e-3), 0.0)
    assert (up + conv(x).squeeze(1)).abs().min().item() >= 5e-4, "test setup: pre-activation too close to the ReLU kink"
  up.requires_grad_()
  out = F.relu(up.unsqueeze(1) + conv(x)).squeeze(1)
  g = rnd(B, H, W, seed=3)
  out.backward(g)
  xg, ug = cl(x.detach()).requires_grad_(), up.detach().to(DEV).requires_grad_()
  og = Fn.refine_tail_autograd(xg, gconv, ug)
  og.backward(g.to(DEV))
  close(og.detach().cpu(), out.detach(), 1e-5, "RefineTail 376x1248: forward")
  close(ug.grad.cpu(), up.grad, 1e-5, "RefineTail 376x1248: dup")
  close(uncl(xg.grad), x.grad, 1e-4, "RefineTail 376x1248: dx")
  close(gconv.weight.grad.cpu(), conv.weight.grad, 1e-4, "RefineTail 376x1248: dw")
  close(gconv.bias.grad.cpu(), conv.bias.grad, 1e-4, "RefineTail 376x1248: db")
