"""Forward kernels of the inference and train-mode forward, one wrapper at a time, against plain high-precision references at
the shapes the product path launches: KITTI k = 3 (376x1248 -> 188x624 -> 94x312 -> 47x156, a 24x47x156 cost volume,
376x1248 refinement), the ragged 375x1242 and the SceneFlow 540x960 (540 -> 270 -> 135 -> 68, a 24x68x120 cost volume),
with the batch sizes the bench and a sharded SceneFlow batch run (B = 1, 2, 4, 8, 32).

Method as test_gpu_backward_kernels: small integers for activations, dyadic weights, scales and shifts (k/16, k/256).  Every
product and partial sum is then exact in fp32 and in the fp16 operand split (the low half of every operand is 0 and the
weight image's 2^-s scaling is exact), so the kernel must equal the reference bit for bit: a dropped, duplicated or
mis-indexed tap, row, tile or sample cannot hide behind a tolerance.  The reference is a float64 convolution on the GPU, cast
to fp32 (exact), followed by the kernel's own epilogue rounding sequence in fp32 torch ops.  Each kernel also gets a
random-float case against float64 with its bound and the reason beside it; the batched random cases also check that each
sample equals a B = 1 call on that sample bit for bit (these kernels tile per sample and row and never reduce across
samples; BatchNorm statistics, which do, are excluded)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import stereonet_oracle as O
from stereonet_b200 import ops
from test_gpu_backward_kernels import bilinear_matrix, bounded as bounded_cpu, dyadic, exact, ints
from test_gpu_kernels import DEV, rnd

pytestmark = pytest.mark.gpu

SLOPE = torch.tensor(0.2, dtype=torch.float32)          # SNB_LRELU_SLOPE (0.2f): the fp32 constant the kernels multiply by
U = 2.0 ** -24                                          # unit roundoff of fp32
GRID_LIMIT = 2 ** 24                                    # fp32 sums of values on a grid g are exact below 2^24 g


def bounded(got, ref, bound, what):
  """test_gpu_backward_kernels.bounded with a bound that may live on the GPU."""
  bounded_cpu(got, ref, bound.detach().cpu() if isinstance(bound, torch.Tensor) else float(bound), what)


def dints(shape, lo, hi, seed):
  """Integers in [lo, hi] as fp32, generated on the GPU (the B = 32 and full-resolution cases)."""
  g = torch.Generator(DEV).manual_seed(seed)
  return torch.randint(lo, hi + 1, tuple(shape), generator=g, device=DEV).float()


def drnd(shape, seed, scale=1.0):
  g = torch.Generator(DEV).manual_seed(seed)
  return torch.randn(tuple(shape), generator=g, device=DEV) * scale


def to_nc(x):      # channels-last [B,(D),H,W,C] -> [B,C,(D),H,W]
  return x.permute(0, 4, 1, 2, 3) if x.dim() == 5 else x.permute(0, 3, 1, 2)


def to_cl(x):      # [B,C,(D),H,W] -> channels-last
  return (x.permute(0, 2, 3, 4, 1) if x.dim() == 5 else x.permute(0, 2, 3, 1)).contiguous()


def conv64(x_cl, w, dil=1, stride=1, pad=None):
  """float64 convolution of a channels-last activation on the GPU, result channels-last, no bias."""
  x = to_nc(x_cl).to(DEV, torch.float64)
  w = w.to(DEV, torch.float64)
  if x.dim() == 5:
    return to_cl(F.conv3d(x, w, padding=1))
  k = w.shape[-1]
  return to_cl(F.conv2d(x, w, stride=stride, padding=dil * (k - 1) // 2 if pad is None else pad, dilation=dil))


def walk_epilogue(conv, bias=None, scale=None, shift=None, lrelu=False, residual=None):
  """The walk kernel's epilogue (conv_c32_ws.cu, epilogue warps) in fp32 on its accumulator `conv` (float64, exact or rounded
  once to fp32 here).  Host side of the kernel (sPar): alpha = scale * 2^-s, beta = fmaf(scale, bias, shift) (scale 1 and
  shift 0 without a BatchNorm fold) -- 2^-s undoes the weight image's power-of-two scaling exactly, so alpha * acc equals
  scale * conv.  Then o = fmaf(acc, alpha, beta); o > 0 ? o : o * 0.2f; o + residual.  The fmafs round once: float64
  evaluation of an exact fp32 product plus an fp32 addend, rounded to fp32, gives the same value whenever the sum is
  representable (the exact-data cases) and is within one fp32 rounding otherwise."""
  acc = conv.float()
  dev = acc.device
  sc = (torch.ones(32) if scale is None else scale).to(dev)
  b = (torch.zeros(32) if bias is None else bias).to(dev)
  sh = (torch.zeros(32) if shift is None else shift).to(dev)
  beta = (sc.double() * b.double() + sh.double()).float()
  o = (acc.double() * sc.double() + beta.double()).float()
  if lrelu:
    o = torch.where(o > 0, o, o * SLOPE.to(dev))
  if residual is not None:
    o = o + residual
  return o


def walk_bound(conv_abs, scale=None, bias=None, shift=None):
  """Bound of a random-float walk-kernel output against float64: the fp16 split keeps 22 bits of each operand (<= 2^-21 of
  each product), and each output collects ~40 fp32 roundings (18-54 K = 16 slices into the accumulator, the in-slice sums, the
  epilogue fmaf and residual add), <= 40 * 2^-24 of the sum of |terms|.  Together < 1e-5 of sum|terms|."""
  sc = (torch.ones(32) if scale is None else scale.abs()).to(conv_abs.device).double()
  beta = ((torch.zeros(32) if bias is None else bias.abs()).to(conv_abs.device).double() * sc
          + (torch.zeros(32) if shift is None else shift.abs()).to(conv_abs.device).double())
  return 1e-5 * (conv_abs * sc + beta)


def per_sample(fn, batched_out, *inputs, what):
  """Batch invariance: output sample i of the batched call equals the B = 1 call on sample i, bit for bit."""
  outs = batched_out if isinstance(batched_out, (tuple, list)) else (batched_out,)
  for i in range(inputs[0].shape[0]):
    one = fn(*[t[i:i + 1].contiguous() if isinstance(t, torch.Tensor) and t.dim() > 1 else t for t in inputs])
    one = one if isinstance(one, (tuple, list)) else (one,)
    for k, (a, b) in enumerate(zip(outs, one)):
      if a is None:
        continue
      assert torch.equal(a[i:i + 1], b), f"{what}: output {k} of sample {i} differs from the B = 1 call"


def assert_exact_sums(v, grid, what):
  """The test's own data keeps these partial sums exact in fp32: every |sum| below 2^24 grid units."""
  m = float(v.abs().max())
  assert m < GRID_LIMIT * grid, f"test setup ({what}): a partial sum {m:.4g} reaches 2^24 grid units of {grid}"


# ================================================================================================ 1. 5x5 stride-2 layers
C3_SHAPES = [(1, 376, 1248), (2, 376, 1248), (1, 375, 1242), (2, 375, 1242), (4, 540, 960)]


@pytest.mark.parametrize("B,H,W", C3_SHAPES)
def test_conv5x5s2_c3_exact(B, H, W):
  """downsample[0] (3 -> 32, 5x5 stride 2): snb_conv5x5s2_c3_phases where its output is even (376x1248 -> 188x624,
  540x960 -> 270x480: the inference path), snb_conv5x5s2_c3 where it is not (375x1242 -> 188x621).  Image k/256, weights
  k/16, bias k/16: 75 products on the 2^-12 grid, |y| < 10.  Reference: float64 conv.  Bit-exact."""
  img = dints((B, 3, H, W), 0, 255, seed=H + W) / 256
  w, b = dyadic((32, 3, 5, 5), 2, 16, seed=1), dyadic((32,), 16, 16, seed=2)
  ref = to_cl(F.conv2d(img.double(), w.to(DEV, torch.float64), b.to(DEV, torch.float64), stride=2, padding=2)).float()
  OH, OW = ref.shape[1:3]
  if OH % 2 == 0 and OW % 2 == 0:
    got = ops.conv5x5s2_c3_phases(img, w.to(DEV), b.to(DEV))
    exact(got, torch.stack([ref[:, a::2, c::2] for a in (0, 1) for c in (0, 1)]), f"snb_conv5x5s2_c3_phases {B}x{H}x{W}")
  exact(ops.conv5x5s2_c3(img, w.to(DEV), b.to(DEV)), ref, f"snb_conv5x5s2_c3 {B}x{H}x{W}")


# input of downsample[1] / [2]: 188x624 and 94x312 (KITTI), 188x621 and 94x311 (375x1242), 270x480 and the odd 135x240 -> 68x120
C32_5X5_SHAPES = [(1, 188, 624), (2, 188, 624), (1, 94, 312), (2, 94, 312), (1, 188, 621), (2, 188, 621), (1, 94, 311),
                  (4, 270, 480), (4, 135, 240)]


@pytest.mark.parametrize("B,H,W", C32_5X5_SHAPES)
def test_conv5x5s2_c32_ws_exact(B, H, W):
  """downsample[1:] (32 -> 32, 5x5 stride 2, pad 2) on the walk kernel: snb_conv5x5s2_c32_ws over the polyphase images and
  snb_conv5x5s2_c32_ws_x over strided views of the un-split input.  Integer x in [-2, 2], weights and bias k/16: 800 products
  on the 1/16 grid, |y| <= 202.  Reference: float64 conv.  Both bit-exact, and the _x path identical to the phases path."""
  x = dints((B, H, W, 32), -2, 2, seed=H * 7 + W)
  w, b = dyadic((32, 32, 5, 5), 2, 16, seed=3), dyadic((32,), 16, 16, seed=4)
  ref = walk_epilogue(conv64(x, w, stride=2, pad=2), bias=b)
  wimg = ops.prep_conv5x5s2_weights_ws(w.to(DEV))
  y = ops.conv5x5s2_c32_ws(ops.phase_split(x), wimg, bias=b.to(DEV))
  exact(y, ref, f"snb_conv5x5s2_c32_ws (phases) {B}x{H}x{W}")
  y2 = ops.conv5x5s2_c32_ws_x(x, wimg, bias=b.to(DEV))
  assert torch.equal(y2, y), f"snb_conv5x5s2_c32_ws_x {B}x{H}x{W}: differs from the phases path"


@pytest.mark.parametrize("B,IH,IW", [(2, 375, 1242), (4, 270, 480)])
def test_conv5x5s2_random(B, IH, IW):
  """Random floats: downsample[0] from a 375x1242 / 270x480 image and downsample[1:] on its output size (188x621, 135x240).
  Bounds against float64: the first layer is a 75-term fp32 FMA chain (<= 75 * 2^-24 < 5e-6 of sum|terms|); the 32-channel
  layer walk_bound.  Each sample equals a B = 1 call."""
  H, W = (IH + 1) // 2, (IW + 1) // 2
  img = torch.rand(B, 3, IH, IW, generator=torch.Generator().manual_seed(IH)).to(DEV)
  w0, b0 = rnd(32, 3, 5, 5, seed=1, scale=0.2), rnd(32, seed=2)
  ref0 = to_cl(F.conv2d(img.double(), w0.to(DEV, torch.float64), b0.to(DEV, torch.float64), stride=2, padding=2))
  abs0 = to_cl(F.conv2d(img.double(), w0.abs().to(DEV, torch.float64), b0.abs().to(DEV, torch.float64), stride=2, padding=2))
  y0 = ops.conv5x5s2_c3(img, w0.to(DEV), b0.to(DEV))
  bounded(y0, ref0, 5e-6 * abs0, f"snb_conv5x5s2_c3 (random) {tuple(img.shape)}")
  per_sample(lambda i: ops.conv5x5s2_c3(i, w0.to(DEV), b0.to(DEV)), y0, img, what="snb_conv5x5s2_c3 batch invariance")
  x = drnd((B, H, W, 32), seed=5)
  w, b = rnd(32, 32, 5, 5, seed=6, scale=0.05), rnd(32, seed=7)
  wimg = ops.prep_conv5x5s2_weights_ws(w.to(DEV))
  y = ops.conv5x5s2_c32_ws(ops.phase_split(x), wimg, bias=b.to(DEV))
  bounded(y, conv64(x, w, stride=2, pad=2) + b.to(DEV).double(), walk_bound(conv64(x.abs(), w.abs(), stride=2, pad=2), bias=b),
          f"snb_conv5x5s2_c32_ws (random) {B}x{H}x{W}")
  assert torch.equal(ops.conv5x5s2_c32_ws_x(x, wimg, bias=b.to(DEV)), y), f"snb_conv5x5s2_c32_ws_x (random) {B}x{H}x{W}"
  per_sample(lambda t: ops.conv5x5s2_c32_ws(ops.phase_split(t), wimg, bias=b.to(DEV)), y, x,
             what=f"snb_conv5x5s2_c32_ws batch invariance {B}x{H}x{W}")


# ================================================================================================ 2./3. walk kernel, eval epilogue
def bn_fold_data(seed):
  """Exact folded-BN data: scale k/16 (either sign, nonzero), shift k/256, conv bias k/16."""
  sc = ints((32,), 1, 32, seed) / 16 * torch.where(ints((32,), 0, 1, seed + 1) > 0, 1.0, -1.0)
  return dyadic((32,), 16, 16, seed + 2), sc, dyadic((32,), 512, 256, seed + 3)


# (B, H, W, dil): feature residual blocks at 47x156 and 68x120; refinement blocks at 376x1248, 375x1242 and 540x960, one case
# per distinct dilation of the six (1, 2, 4, 8, 1, 1)
WALK2D_CASES = [(1, 47, 156, 1), (2, 47, 156, 1), (4, 47, 156, 1), (1, 68, 120, 1), (2, 68, 120, 1), (4, 68, 120, 1)] + \
               [(B, 376, 1248, d) for B in (1, 2) for d in (1, 2, 4, 8)] + [(1, 375, 1242, d) for d in (1, 2, 4, 8)] + \
               [(2, 540, 960, d) for d in (1, 2, 4, 8)]


@pytest.mark.parametrize("B,H,W,dil", WALK2D_CASES)
def test_walk2d_residual_block_exact(B, H, W, dil):
  """A residual block in eval mode: y = x + LeakyReLU(scale * (conv(x) + bias) + shift), the residual read on chip from the
  input (res_mode 1), as BasicBlock.forward_cl runs it.  At full resolution each CTA walks ~25 tiles, so the staging and
  residual rings and their barrier phases wrap many times.  Integer x in [-2, 2], weights k/16: |conv| <= 72 on the 1/16 grid,
  o on the 1/256 grid.  Reference: float64 conv + walk_epilogue.  Bit-exact."""
  x = dints((B, H, W, 32), -2, 2, seed=H + W + dil)
  w = dyadic((32, 32, 3, 3), 2, 16, seed=dil)
  bias, sc, sh = bn_fold_data(10 + dil)
  ref = walk_epilogue(conv64(x, w, dil), bias, sc, sh, lrelu=True, residual=x)
  g = ops.geom((B, H, W, 32), 3, dil=dil)
  y, _ = ops.conv_c32_tc(x, ops.prep_conv_weights_tc(w.to(DEV)), g, bias=bias.to(DEV), scale=sc.to(DEV), shift=sh.to(DEV),
                         residual=x, lrelu=True)
  exact(y, ref, f"snb_conv_c32_ws 2-D eval epilogue + in-place residual {B}x{H}x{W} dil={dil}")


@pytest.mark.parametrize("B,H,W", [(1, 47, 156), (2, 47, 156), (4, 68, 120), (1, 376, 1248)])
def test_walk2d_bias_only_exact(B, H, W):
  """conv_alone (bias only, no BatchNorm, no activation) and a bias-only layer at full resolution.  Bit-exact."""
  x = dints((B, H, W, 32), -2, 2, seed=H * W)
  w, b = dyadic((32, 32, 3, 3), 2, 16, seed=21), dyadic((32,), 16, 16, seed=22)
  y, _ = ops.conv_c32_tc(x, ops.prep_conv_weights_tc(w.to(DEV)), ops.geom((B, H, W, 32), 3), bias=b.to(DEV))
  exact(y, walk_epilogue(conv64(x, w), bias=b), f"snb_conv_c32_ws 2-D bias only {B}x{H}x{W}")


@pytest.mark.parametrize("B,H,W,dil", [(2, 376, 1248, 8), (2, 540, 960, 2), (4, 68, 120, 1)])
def test_walk2d_random(B, H, W, dil):
  """Random floats, eval epilogue with the in-place residual.  Bound: walk_bound (LeakyReLU scales the error by <= 1) plus one
  rounding of the residual add.  Each sample equals a B = 1 call."""
  x = drnd((B, H, W, 32), seed=dil)
  w, bias = rnd(32, 32, 3, 3, seed=1, scale=0.1), rnd(32, seed=2)
  sc, sh = rnd(32, seed=3).abs() + 0.5, rnd(32, seed=4)
  c = conv64(x, w, dil)
  u = (c + bias.to(DEV).double()) * sc.to(DEV).double() + sh.to(DEV).double()
  ref = torch.where(u > 0, u, 0.2 * u) + x.double()
  wimg = ops.prep_conv_weights_tc(w.to(DEV))
  run = lambda t: ops.conv_c32_tc(t, wimg, ops.geom(tuple(t.shape), 3, dil=dil), bias=bias.to(DEV), scale=sc.to(DEV),
                                  shift=sh.to(DEV), residual=t, lrelu=True)[0]
  y = run(x)
  bounded(y, ref, walk_bound(conv64(x.abs(), w.abs(), dil), sc, bias, sh) + U * ref.abs(),
          f"snb_conv_c32_ws 2-D (random) {B}x{H}x{W} dil={dil}")
  per_sample(run, y, x, what=f"snb_conv_c32_ws 2-D batch invariance {B}x{H}x{W} dil={dil}")


WALK3D_CASES = [(1, 24, 47, 156), (2, 24, 47, 156), (4, 24, 68, 120), (1, 12, 24, 78)]


@pytest.mark.parametrize("B,D,H,W", WALK3D_CASES)
def test_walk3d_eval_exact(B, D, H, W):
  """A cost-filter layer in eval mode: LeakyReLU(scale * (conv3d(x) + bias) + shift), no residual; the 3-D walk kernel with its
  two accumulator rings, acc = fmaf(D2, 2^-11, D1) (D2 = 0 here: the low operand halves are 0).  Integer x in [-2, 2], weights
  k/16: |conv| <= 216 on the 1/16 grid.  Includes D' = 12 (k = 4, 24x78).  Reference: float64 conv3d + walk_epilogue.
  Bit-exact."""
  x = dints((B, D, H, W, 32), -2, 2, seed=D * H + W)
  w = dyadic((32, 32, 3, 3, 3), 2, 16, seed=31)
  bias, sc, sh = bn_fold_data(32)
  y, _ = ops.conv_c32_tc(x, ops.prep_conv_weights_tc(w.to(DEV)), ops.geom((B, D, H, W, 32), 3), bias=bias.to(DEV),
                         scale=sc.to(DEV), shift=sh.to(DEV), lrelu=True)
  exact(y, walk_epilogue(conv64(x, w), bias, sc, sh, lrelu=True), f"snb_conv_c32_ws 3-D eval epilogue {B}x{D}x{H}x{W}")


def test_walk3d_random():
  """Random floats at 4 x 24x68x120.  Bound: walk_bound (864 products per output).  Each sample equals a B = 1 call."""
  B, D, H, W = 4, 24, 68, 120
  x = drnd((B, D, H, W, 32), seed=41)
  w, bias = rnd(32, 32, 3, 3, 3, seed=42, scale=0.05), rnd(32, seed=43)
  sc, sh = rnd(32, seed=44).abs() + 0.5, rnd(32, seed=45)
  u = (conv64(x, w) + bias.to(DEV).double()) * sc.to(DEV).double() + sh.to(DEV).double()
  ref = torch.where(u > 0, u, 0.2 * u)
  wimg = ops.prep_conv_weights_tc(w.to(DEV))
  run = lambda t: ops.conv_c32_tc(t, wimg, ops.geom(tuple(t.shape), 3), bias=bias.to(DEV), scale=sc.to(DEV), shift=sh.to(DEV),
                                  lrelu=True)[0]
  y = run(x)
  bounded(y, ref, walk_bound(conv64(x.abs(), w.abs()), sc, bias, sh), f"snb_conv_c32_ws 3-D (random) {B}x{D}x{H}x{W}")
  per_sample(run, y, x, what=f"snb_conv_c32_ws 3-D batch invariance {B}x{D}x{H}x{W}")


# ================================================================================================ 4. cost volume
@pytest.mark.parametrize("B,H,W", [(1, 47, 156), (2, 47, 156), (4, 68, 120), (32, 68, 120), (1, 24, 78)])
def test_cost_volume_exact(B, H, W):
  """Difference cost volume (D = 24; D' = 12 at 24x78).  4 x 24x68x120 (100 MB) and 32 x 24x68x120 (800 MB) are over 64 MB and
  take the TMA-staged kernel.  One fp32 subtraction per element: bit-exact against O.cost_volume_numpy.  Each sample equals a
  B = 1 call."""
  D = 12 if H == 24 else 24
  L, R = drnd((B, H, W, 32), seed=1), drnd((B, H, W, 32), seed=2)
  got = ops.cost_volume(L, R, D)
  ref = O.cost_volume_numpy(to_nc(L).cpu().numpy(), to_nc(R).cpu().numpy(), D)
  assert np.array_equal(to_nc(got).cpu().numpy(), ref), f"snb_cost_volume_fwd {B}x{D}x{H}x{W}: differs from cost_volume_numpy"
  if B > 1:
    per_sample(lambda l, r: ops.cost_volume(l, r, D), got, L, R, what=f"snb_cost_volume_fwd batch invariance B={B}")


# ================================================================================================ 5. stereo heads
def pred_bound(D):
  """|pred - float64 soft-argmin of the same costs|: pred = sum_d d p_d, so a relative error delta in each exp term moves it by
  <= 2 (D - 1) delta.  __expf / expf of c - m <= 0: <= 2^-21 + |c - m| 2^-24 relative, and terms with c - m < -30 weigh
  < 1e-13, so delta <= 2^-21 + 30 * 2^-24; the D-term sums and the division add (D + 2) 2^-24 of (D - 1)."""
  return (D - 1) * (2 * (2.0 ** -21 + 30 * U) + (D + 2) * U)


def fcs_bound(cost):
  """|fcs - reference| <= (2D + 4) 2^-24 max_d |cost| per pixel: a D-term fp32 sum of the costs, a division and two
  subtractions, each partial bounded by D max|cost|."""
  D = cost.shape[1]
  return (2 * D + 4) * U * cost.abs().amax(1)


def softargmin64(cost):
  c = cost.double()
  return (torch.softmax(c, 1) * torch.arange(c.shape[1], dtype=torch.float64, device=c.device).view(1, -1, 1, 1)).sum(1)


def fcs64(cost):
  s = torch.sort(cost.double(), dim=1, descending=True)[0]
  return s[:, 0] - s[:, 2:].mean(1)


HEAD_CASES = [(1, 24, 47, 156), (2, 24, 47, 156), (4, 24, 68, 120), (32, 24, 68, 120), (1, 12, 24, 78)]


@pytest.mark.parametrize("B,D,H,W", HEAD_CASES)
def test_heads_exact_cost(B, D, H, W):
  """conv3d_alone (32 -> 1) + soft-argmin: the inference head (snb_conv_c32_taps with 27 taps + snb_tapsum_softargmin) and the
  training head (snb_conv3d_out_softargmin: cost, pred, FCS).  Integer x in [-2, 2], weights and bias k/16: the cost is
  bit-exact against the float64 conv3d; pred against the float64 soft-argmin of that cost within pred_bound(D), FCS against
  sorted_desc[0] - mean(sorted_desc[2:]) within fcs_bound.  The three outputs of the inference head with and without the cost
  are identical."""
  x = dints((B, D, H, W, 32), -2, 2, seed=B + D * H)
  w, b = dyadic((1, 32, 3, 3, 3), 2, 16, seed=51), dyadic((1,), 16, 16, seed=52)
  cost_ref = (to_nc(conv64(x, w)).squeeze(1) + b.item()).float()
  what = f"{B}x{D}x{H}x{W}"
  taps = ops.conv_c32_taps(x, w.to(DEV), 27)
  cost, pred = ops.tapsum_softargmin(taps, b.to(DEV), True)
  exact(cost, cost_ref, f"snb_conv_c32_taps<27> + snb_tapsum_softargmin {what}: cost")
  bounded(pred, softargmin64(cost_ref), pred_bound(D), f"snb_tapsum_softargmin {what}: pred")
  _, pred2 = ops.tapsum_softargmin(taps, b.to(DEV), False)
  assert torch.equal(pred, pred2), f"snb_tapsum_softargmin {what}: pred depends on want_cost"
  cost_f, pred_f, fcs = ops.conv3d_out_softargmin(x, w.to(DEV), b.to(DEV), want_cost=True, want_fcs=True)
  exact(cost_f, cost_ref, f"snb_conv3d_out_softargmin {what}: cost")
  bounded(pred_f, softargmin64(cost_ref), pred_bound(D), f"snb_conv3d_out_softargmin {what}: pred")
  bounded(fcs, fcs64(cost_ref), fcs_bound(cost_ref), f"snb_conv3d_out_softargmin {what}: fcs")


def identity_tap_input(cost):
  """x [B,D,H,W,32] with x[..., 0] = cost and a weight that passes channel 0 of the centre tap: the head sees `cost` itself."""
  x = torch.zeros(tuple(cost.shape) + (32,), device=DEV)
  x[..., 0] = cost
  w = torch.zeros(1, 32, 3, 3, 3, device=DEV)
  w[0, 0, 1, 1, 1] = 1.0
  return x, w


@pytest.mark.parametrize("case", ["equal", "spread1e3", "plus1e4", "minus1e4"])
@pytest.mark.parametrize("D", [12, 24])
def test_heads_soft_argmin_edges(case, D):
  """Soft-argmin edges through both heads, fed through an identity tap: all-equal costs (pred = (D - 1) / 2), a spread of 1e3
  (all but the top terms underflow in exp) and costs around +-1e4 (exp overflows without the max subtraction).  Costs sit on a
  1/64 grid with <= 20 significant bits, so they pass the fp16 split exactly (checked).  Bounds: pred_bound(D), fcs_bound."""
  B, H, W = 2, 9, 70
  g = torch.Generator(DEV).manual_seed(D * 7 + len(case))
  if case == "equal":
    cost = torch.full((B, D, H, W), 3.25, device=DEV)
  elif case == "spread1e3":
    cost = torch.randint(0, 64000, (B, D, H, W), generator=g, device=DEV).float() / 64
  else:
    cost = torch.randint(0, 512, (B, D, H, W), generator=g, device=DEV).float() / 64 + (1e4 if case == "plus1e4" else -1e4)
  x, w = identity_tap_input(cost)
  zero = torch.zeros(1, device=DEV)
  c1, p1 = ops.tapsum_softargmin(ops.conv_c32_taps(x, w, 27), zero, True)
  c2, p2, fcs = ops.conv3d_out_softargmin(x, w, zero, want_cost=True, want_fcs=True)
  ref = softargmin64(cost)
  what = f"D={D} {case}"
  exact(c1, cost, f"snb_conv_c32_taps<27> identity tap {what}: cost")
  exact(c2, cost, f"snb_conv3d_out_softargmin identity tap {what}: cost")
  if case == "equal":
    assert float((ref - (D - 1) / 2).abs().max()) < 1e-12
  bounded(p1, ref, pred_bound(D), f"snb_tapsum_softargmin {what}: pred")
  bounded(p2, ref, pred_bound(D), f"snb_conv3d_out_softargmin {what}: pred")
  bounded(fcs, fcs64(cost), fcs_bound(cost), f"snb_conv3d_out_softargmin {what}: fcs")


def test_heads_random():
  """Random floats at 4 x 24x68x120.  Cost bound 1e-5 of the sum of |terms| (fp16-split taps: walk_bound's reasoning, 864
  products); pred: pred_bound(D) plus 2 (D - 1) times the largest cost error; FCS: fcs_bound plus 2x the largest cost error.
  Each sample equals a B = 1 call in both heads."""
  B, D, H, W = 4, 24, 68, 120
  x = drnd((B, D, H, W, 32), seed=61)
  w, b = rnd(1, 32, 3, 3, 3, seed=62, scale=0.5), rnd(1, seed=63)
  c64 = to_nc(conv64(x, w)).squeeze(1) + b.item()
  cb = 1e-5 * (to_nc(conv64(x.abs(), w.abs())).squeeze(1) + abs(b.item()))
  emax = float(cb.max())
  taps_run = lambda t: ops.tapsum_softargmin(ops.conv_c32_taps(t, w.to(DEV), 27), b.to(DEV), True)
  cost, pred = taps_run(x)
  bounded(cost, c64, cb, "snb_conv_c32_taps<27> + snb_tapsum_softargmin (random): cost")
  bounded(pred, softargmin64(c64), pred_bound(D) + 2 * (D - 1) * emax, "snb_tapsum_softargmin (random): pred")
  per_sample(taps_run, (cost, pred), x, what="inference head batch invariance")
  fused_run = lambda t: ops.conv3d_out_softargmin(t, w.to(DEV), b.to(DEV), want_cost=True, want_fcs=True)
  cf, pf, ff = fused_run(x)
  bounded(cf, c64, cb, "snb_conv3d_out_softargmin (random): cost")
  bounded(pf, softargmin64(c64), pred_bound(D) + 2 * (D - 1) * emax, "snb_conv3d_out_softargmin (random): pred")
  bounded(ff, fcs64(c64), fcs_bound(c64) + 2 * emax, "snb_conv3d_out_softargmin (random): fcs")
  per_sample(fused_run, (cf, pf, ff), x, what="training head batch invariance")


# ================================================================================================ 6. refinement input layer
def up_ref64(coarse, H, W):
  """float64 mul * bilinear(coarse) at the fp32 source coordinates (bilinear_matrix), mul = fp32(W) / fp32(w) as ops passes it."""
  B, h, w = coarse.shape
  mul = float(np.float32(float(W) / float(w)))
  Ay, Ax = bilinear_matrix(H, h).to(DEV), bilinear_matrix(W, w).to(DEV)
  return mul * torch.einsum("yi,bij,xj->byx", Ay, coarse.double(), Ax)


def refine_in_ref(coarse, rgb, w, H, W):
  """(up, float64 conv of [up, rgb] without bias [B,H,W,32], the same conv of |inputs|, |w|)."""
  up = up_ref64(coarse, H, W)
  inp = torch.cat([up.unsqueeze(1), rgb.double()], 1)
  w64 = w.to(DEV, torch.float64)
  return up, to_cl(F.conv2d(inp, w64, padding=1)), to_cl(F.conv2d(inp.abs(), w64.abs(), padding=1))


REFINE_IN_CASES = [(1, 47, 156, 376, 1248), (2, 47, 156, 376, 1248), (1, 47, 156, 375, 1242), (1, 68, 120, 540, 960),
                   (2, 68, 120, 540, 960)]


@pytest.mark.parametrize("B,h,w,H,W", REFINE_IN_CASES)
def test_refine_in(B, h, w, H, W):
  """The refinement's input layer: upsample x W/w + concat with the image + Conv2d(4 -> 32).  Eval: snb_refine_pack_input +
  snb_conv_c4_ws (walk kernel) with the folded-BN epilogue; train: snb_refine_in_conv with bias only and its statistics.
  At 376x1248 the ratio is exactly 8: every 1-D bilinear weight is a multiple of 1/16, so with coarse integers in [0, 40], the
  image k/16 and weights k/16, up (1/32 grid, <= 320), z (1/512 grid, |z| < 400) and the eval output (2^-13 grid, < 800) are
  exact: bit-exact against the float64 reference.  The statistics' tile sums of z^2 (512 positions on a 2^-16 grid) are not exact: their
  column totals get 512 * 2^-24 of sum z^2 (the longest fp32 chain of a tile), and sum z as much of sum |z|.
  Ragged ratios (375x1242, and 540/68 in y at 540x960): up within 16 ulps of max|up| (a few fp32 roundings at the same fp32
  source coordinates as bilinear_matrix), z and the eval output within 2e-5 of sum|terms| (walk_bound, doubled for the error
  carried by up)."""
  coarse = dints((B, h, w), 0, 40, seed=H + B)
  rgb = dints((B, 3, H, W), 0, 15, seed=W + B) / 16
  wt = dyadic((32, 4, 3, 3), 2, 16, seed=71)
  bias, sc, sh = bn_fold_data(72)
  up64, c64, cabs = refine_in_ref(coarse, rgb, wt, H, W)
  ragged = (H % h != 0) or (W % w != 0) or (H // h != W // w)
  what = f"{B}x{h}x{w}->{H}x{W}"
  wimg = ops.refine_in_weights_ws(wt.to(DEV))
  up, y, _ = ops.refine_in_conv_ws(coarse, rgb, wimg, bias.to(DEV), scale=sc.to(DEV), shift=sh.to(DEV), lrelu=True)
  up_t, z, stats = ops.refine_in_conv(coarse, rgb, wt.to(DEV), bias.to(DEV), want_stats=True)
  zref = c64 + bias.to(DEV).double()
  s_ref = torch.stack([zref.sum((0, 1, 2)), (zref ** 2).sum((0, 1, 2))])
  s_got = stats.double().sum(0)
  s_bound = 512 * U * torch.stack([zref.abs().sum((0, 1, 2)), (zref ** 2).sum((0, 1, 2))])
  zb = 2e-5 * (cabs + bias.abs().to(DEV).double())
  if ragged:        # plus what z's own error (zb) contributes to the totals
    s_bound = s_bound + torch.stack([zb.sum((0, 1, 2)), (2 * zref.abs() * zb + zb * zb).sum((0, 1, 2))])
  bounded(s_got, s_ref, s_bound, f"snb_refine_in_conv {what}: statistics column totals")
  if not ragged:
    exact(up, up64, f"snb_refine_pack_input {what}: up")
    exact(up_t, up64, f"snb_refine_in_conv {what}: up")
    exact(y, walk_epilogue(c64, bias, sc, sh, lrelu=True), f"snb_conv_c4_ws eval epilogue {what}")
    exact(z, zref, f"snb_refine_in_conv {what}: z")
    return
  up_b = 16 * 2 * U * float(up64.abs().max())
  bounded(up, up64, up_b, f"snb_refine_pack_input {what}: up")
  bounded(up_t, up64, up_b, f"snb_refine_in_conv {what}: up")
  u = zref * sc.to(DEV).double() + sh.to(DEV).double()
  bounded(y, torch.where(u > 0, u, 0.2 * u), zb * sc.abs().to(DEV).double() + 2 * U * u.abs(), f"snb_conv_c4_ws eval epilogue {what}")
  bounded(z, zref, zb, f"snb_refine_in_conv {what}: z")


def test_refine_in_random():
  """Random floats at 2 x 47x156 -> 376x1248 (coarse disparities in [0, 20), random image, weights and BN fold).  Bounds: up 16
  ulps of max|up|; the eval output of the walk kernel 2e-5 of sum|terms| (as test_refine_in).  Each sample equals a B = 1 call."""
  B, h, w, H, W = 2, 47, 156, 376, 1248
  coarse = torch.rand(B, h, w, generator=torch.Generator().manual_seed(1)).to(DEV) * 20
  rgb = torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(2)).to(DEV)
  wt, bias = rnd(32, 4, 3, 3, seed=3, scale=0.2), rnd(32, seed=4)
  sc, sh = rnd(32, seed=5).abs() + 0.5, rnd(32, seed=6)
  up64, c64, cabs = refine_in_ref(coarse, rgb, wt, H, W)
  wimg = ops.refine_in_weights_ws(wt.to(DEV))
  run = lambda c, r: ops.refine_in_conv_ws(c, r, wimg, bias.to(DEV), scale=sc.to(DEV), shift=sh.to(DEV), lrelu=True)[:2]
  up, y = run(coarse, rgb)
  bounded(up, up64, 16 * 2 * U * float(up64.abs().max()), "snb_refine_pack_input (random): up")
  u = (c64 + bias.to(DEV).double()) * sc.to(DEV).double() + sh.to(DEV).double()
  bounded(y, torch.where(u > 0, u, 0.2 * u), 2e-5 * ((cabs + bias.abs().to(DEV).double()) * sc.to(DEV).double() + sh.abs().to(DEV).double()),
          "snb_conv_c4_ws (random) eval epilogue")
  per_sample(run, (up, y), coarse, rgb, what="refinement input batch invariance")


# ================================================================================================ 7. refinement output layer
@pytest.mark.parametrize("B,H,W", [(1, 376, 1248), (2, 376, 1248), (2, 540, 960)])
def test_refine_out_exact(B, H, W):
  """conv2d_out (32 -> 1, 9 taps) + upsampled disparity + ReLU: snb_conv_c32_taps<9> + snb_tapsum_refine_out.  Integer x in
  [-2, 2], weights and bias k/16, up on the 1/2 grid in [0, 160]: the 9 taps, their sum, + bias + up are exact.  Reference:
  ReLU of the float64 sum.  Bit-exact."""
  x = dints((B, H, W, 32), -2, 2, seed=H + B)
  w, b = dyadic((1, 32, 3, 3), 2, 16, seed=81), dyadic((1,), 16, 16, seed=82)
  up = dints((B, H, W), 0, 320, seed=W + B) / 2
  ref = torch.relu(to_nc(conv64(x, w)).squeeze(1) + b.item() + up.double())
  out = ops.tapsum_refine_out(ops.conv_c32_taps(x, w.to(DEV), 9), b.to(DEV), up)
  exact(out, ref, f"snb_conv_c32_taps<9> + snb_tapsum_refine_out {B}x{H}x{W}")


def test_refine_out_random():
  """Random floats at 2 x 376x1248, up pushed so that every ReLU input sits >= 1e-3 from 0 (no flipped mask).  Bound: 1e-5 of
  the sum of |terms| (fp16-split taps, 288 products; then 11 fp32 additions).  Each sample equals a B = 1 call."""
  B, H, W = 2, 376, 1248
  x = drnd((B, H, W, 32), seed=91)
  w, b = rnd(1, 32, 3, 3, seed=92, scale=0.1), rnd(1, seed=93)
  c = to_nc(conv64(x, w)).squeeze(1) + b.item()
  up = drnd((B, H, W), seed=94) * 2
  pre = c + up.double()
  up = (up.double() + torch.where(pre.abs() < 1e-3, torch.where(pre >= 0, 2e-3, -2e-3), 0.0)).float()
  pre = c + up.double()
  assert float(pre.abs().min()) >= 5e-4, "test setup: ReLU input too close to 0"
  bound = 1e-5 * (to_nc(conv64(x.abs(), w.abs())).squeeze(1) + abs(b.item()) + up.abs().double())
  run = lambda t, u: ops.tapsum_refine_out(ops.conv_c32_taps(t, w.to(DEV), 9), b.to(DEV), u)
  out = run(x, up)
  bounded(out, torch.relu(pre), bound, "snb_conv_c32_taps<9> + snb_tapsum_refine_out (random) 2x376x1248")
  per_sample(run, out, x, up, what="refinement output batch invariance")


# ================================================================================================ 8. train-mode BatchNorm pieces
def tile_rows(z):
  """float64 per-tile (sum, sumsq) rows of the walk kernel's statistics: 2-D z [B,H,W,32] -> row (b*H + h) * ncb + cb over the
  128-pixel column blocks of a row; 3-D z [B,D,H,W,32] -> row (b*D + d) * ncb + cb over 128-position blocks of a flat slice."""
  if z.dim() == 5:
    z = z.reshape(z.shape[0], z.shape[1], -1, 32)
  B, R, L, _ = z.shape
  ncb = (L + 127) // 128
  zp = F.pad(z, (0, 0, 0, ncb * 128 - L)).view(B, R, ncb, 128, 32)
  return torch.stack([zp.sum(3), (zp * zp).sum(3)], 3).reshape(-1, 2, 32), torch.stack([zp.abs().sum(3), (zp * zp).sum(3)], 3)


@pytest.mark.parametrize("B,D,H,W,dil", [(2, 1, 376, 1248, 1), (2, 1, 376, 1248, 4), (2, 1, 47, 156, 1), (2, 24, 47, 156, 1)])
def test_walk_stats_rows_exact(B, D, H, W, dil):
  """The walk kernel's train-mode call (conv + bias, want_stats): z and every per-tile (sum, sumsq) row.  Integer x in
  [-1, 1], weights and bias k/16: z on the 1/16 grid, z^2 on the 1/256 grid; the test asserts that every tile's sum of |z|
  and of z^2 stays below 2^24 grid units, so the fp32 tile sums are exact in any order.  Reference: float64 per-tile sums.
  Bit-exact, rows of both samples included."""
  shape = (B, H, W, 32) if D == 1 else (B, D, H, W, 32)
  x = dints(shape, -1, 1, seed=H + D + dil)
  w = dyadic((32, 32, 3, 3) if D == 1 else (32, 32, 3, 3, 3), 1, 16, seed=101)
  b = dyadic((32,), 16, 16, seed=102)
  zref = conv64(x, w, dil) + b.to(DEV).double()
  rows, absrows = tile_rows(zref)
  assert_exact_sums(absrows[..., 0, :], 1 / 16, "tile sums of |z|")
  assert_exact_sums(absrows[..., 1, :], 1 / 256, "tile sums of z^2")
  g = ops.geom(shape, 3, dil=dil)
  z, stats = ops.conv_c32_tc(x, ops.prep_conv_weights_tc(w.to(DEV)), g, bias=b.to(DEV), want_stats=True)
  what = f"snb_conv_c32_ws {'3-D' if D > 1 else '2-D'} statistics {B}x{D}x{H}x{W} dil={dil}"
  exact(z, zref, what + ": z")
  exact(stats, rows, what + ": per-tile rows")


def bn_reference(s1, s2, count, gamma, beta, rm, rv):
  """snb_bn_finalize_ws in float64 on exact totals: mean = S1 / n, var = S2 / n - mean^2, invstd = 1 / sqrt(var + eps),
  running stats with the unbiased variance and momentum fp32(0.1); scale = gamma * fp32(invstd) in fp32."""
  eps, mom = float(np.float32(ops.BN_EPS)), float(np.float32(ops.BN_MOMENTUM))
  mean = s1 / count
  var = (s2 / count - mean * mean).clamp(min=0)
  invstd = 1.0 / torch.sqrt(var + eps)
  unb = var * count / (count - 1) if count > 1 else var
  rm_new = ((1 - mom) * rm.double() + mom * mean).float()
  rv_new = ((1 - mom) * rv.double() + mom * unb).float()
  scale = gamma * invstd.float()
  shift = beta.double() - mean.float().double() * scale.double()
  return mean.float(), invstd.float(), scale, shift, rm_new, rv_new


@pytest.mark.parametrize("nrows", [1, 256, 257, 1392, 3760])
def test_bn_finalize_exact(nrows):
  """snb_bn_finalize_ws: one stage up to 256 rows, the 64-CTA pre-reduce + finalize above (1392 rows: a 3-D filter layer at
  KITTI, 3760: a refinement block).  Rows are the (sum, sumsq) of 16 integer values per channel (offsets up to +-3), so every
  row, chunk and total is exact.  mean, invstd, scale, running_mean, running_var bit-exact against the float64 formula;
  shift = beta - mean * scale within one rounding of its terms; num_batches_tracked += 1."""
  zz = ints((nrows, 16, 32), -8, 8, seed=nrows) + ints((32,), -3, 3, seed=nrows + 1)
  stats = torch.stack([zz.sum(1), (zz * zz).sum(1)], 1)
  count = nrows * 16
  bn = torch.nn.BatchNorm2d(32)
  with torch.no_grad():
    bn.weight.copy_(rnd(32, seed=3).abs() + 0.5); bn.bias.copy_(rnd(32, seed=4))
    bn.running_mean.copy_(rnd(32, seed=5)); bn.running_var.copy_(rnd(32, seed=6).abs() + 0.5)
  ref = bn_reference(zz.double().sum((0, 1)), (zz.double() ** 2).sum((0, 1)), count, bn.weight.detach(), bn.bias.detach(),
                     bn.running_mean, bn.running_var)
  beta = bn.bias.detach().clone()
  gbn = bn.to(DEV)
  nbt0 = int(gbn.num_batches_tracked)
  scale, shift, mean, invstd = ops.bn_finalize(stats.to(DEV), count, gbn)
  what = f"snb_bn_finalize_ws rows={nrows}"
  exact(mean, ref[0], what + ": mean")
  exact(invstd, ref[1], what + ": invstd")
  exact(scale, ref[2], what + ": scale")
  bounded(shift, ref[3], 2 * U * (beta.abs().double() + (ref[0].double() * ref[2].double()).abs()), what + ": shift")
  exact(gbn.running_mean, ref[4], what + ": running_mean")
  exact(gbn.running_var, ref[5], what + ": running_var")
  assert int(gbn.num_batches_tracked) == nbt0 + 1, what + ": num_batches_tracked"


RATIOS = (0.0, 7.0, 100.0, 1000.0)


def invstd_limit(r):
  """Relative invstd error of the train-mode statistics at mean/std = r.  var = E[z^2] - mean^2 cancels, so an error of
  e * mean^2 in the sums of z^2 becomes e * r^2 of var.  The pre-reduce keeps its chunk sums in fp64; what is left is the
  fp32 per-tile (sum, sumsq) rows of the walk kernel.  Measured on a B200 (this test, 3760 tile rows): 1.34e-5 at r = 100 and
  1.49e-3 at r = 1000, i.e. 1.3e-9 to 1.5e-9 * r^2 (with fp32 chunk sums: 5.3e-5 and 4.4e-3).  Limit: about twice that,
  max(1e-5, 3e-9 * r^2): 1e-5 up to r ~ 58, eight times the largest ratio of the model's synthetic states (6.8)."""
  return max(1e-5, 3e-9 * r * r)


def test_bn_stats_precision():
  """The train-mode statistics pipeline at a refinement-block shape (376x1248: 3760 tile rows, both finalize stages): the walk
  kernel's statistics call on an identity 3x3 kernel with bias = mean gives z = x + mean per channel, random N(0, 1) x, eight
  channels each at mean/std 0, 7, 100 and 1000; then ops.bn_finalize.  Reference: float64 two-pass mean and variance of the z
  the kernel wrote.  invstd within invstd_limit(r) relative; mean within 2^-20 (|mean| + std).  The error by ratio is printed."""
  B, H, W = 1, 376, 1248
  r = torch.tensor(RATIOS).repeat_interleave(8)
  x = drnd((B, H, W, 32), seed=111)
  w = torch.zeros(32, 32, 3, 3)
  w[range(32), range(32), 1, 1] = 1.0
  z, stats = ops.conv_c32_tc(x, ops.prep_conv_weights_tc(w.to(DEV)), ops.geom((B, H, W, 32), 3), bias=r.to(DEV), want_stats=True)
  z64 = z.double().reshape(-1, 32)
  m64 = z64.mean(0)
  v64 = ((z64 - m64) ** 2).mean(0)
  inv64 = 1.0 / torch.sqrt(v64 + float(np.float32(ops.BN_EPS)))
  bn = torch.nn.BatchNorm2d(32).to(DEV)
  _, _, mean, invstd = ops.bn_finalize(stats, B * H * W, bn)
  rel = ((invstd.double() - inv64).abs() / inv64).cpu()
  print("[bn stats] relative invstd error by mean/std: " +
        ", ".join(f"{q:g}: {float(rel[r == q].max()):.2e}" for q in RATIOS))
  for q in RATIOS:
    sel = r == q
    bounded(invstd.cpu()[sel], inv64.cpu()[sel], invstd_limit(q) * inv64.cpu()[sel],
            f"bn_stats_prereduce_kernel + bn_finalize_kernel 376x1248 mean/std={q:g}: invstd")
  bounded(mean, m64, 2.0 ** -20 * (m64.abs() + v64.sqrt()), "bn_finalize_kernel 376x1248: mean")


@pytest.mark.parametrize("residual", [False, True])
def test_bn_apply_exact(residual):
  """snb_bn_apply at 2 x 376x1248: y = [r +] LeakyReLU(fmaf(z, scale, shift)).  Integer z and residual, scale k/16, shift an
  odd multiple of 1/32: the fmaf is exact, the LeakyReLU product rounds as in fp32 torch.  Bit-exact."""
  z = dints((2, 376, 1248, 32), -8, 8, seed=121)
  sc = (ints((32,), 1, 16, 122) / 16 * torch.where(ints((32,), 0, 1, 123) > 0, 1.0, -1.0)).to(DEV)
  sh = ((2 * ints((32,), -16, 15, 124) + 1) / 32).to(DEV)
  res = dints(z.shape, -4, 4, seed=125) if residual else None
  o = (z.double() * sc.double() + sh.double()).float()
  o = torch.where(o > 0, o, o * SLOPE.to(DEV))
  if residual:
    o = o + res
  exact(ops.bn_apply(z, sc, sh, residual=res, lrelu=True), o, f"bn_apply_kernel 2x376x1248 residual={residual}")


# ================================================================================================ 10. whole model, bench batch shapes
@pytest.mark.parametrize("B,H,W", [(32, 540, 960), (8, 376, 1248)])
def test_engine_batch_equals_single(B, H, W):
  """StereoEngine (CUDA graph, output_cost_volume=False, as bench.py's SceneFlow arm) at 540x960 with B = 32 and at KITTI with
  B = 8: every sample's disparity equals a B = 1 run of that sample, bit for bit (torch.equal).  Eval mode never mixes samples:
  BatchNorm uses its running statistics and every kernel tiles per sample."""
  import stereonet_b200 as S
  from stereonet_b200.runtime import StereoEngine
  torch.manual_seed(123)
  f, s = S.FeatureExtractorNetwork(3).to(DEV), S.StereoNet(3, 1, 0, maxdisp=192).to(DEV)
  f.eval(); s.eval()
  g = torch.Generator(DEV).manual_seed(B)
  left = torch.rand((B, 3, H, W), generator=g, device=DEV)
  right = torch.roll(left, shifts=-12, dims=3) * 0.9 + 0.1 * torch.rand((B, 3, H, W), generator=g, device=DEV)
  eng = StereoEngine(f, s, output_cost_volume=False)
  outs = eng(left, right)
  key = "pred_disp_l/0"
  batched = outs[key].clone()
  assert bool(torch.isfinite(batched).all()), f"StereoEngine {B}x{H}x{W}: non-finite disparity"
  for i in range(B):
    one = eng(left[i:i + 1].contiguous(), right[i:i + 1].contiguous())[key]
    assert torch.equal(batched[i:i + 1], one), (
        f"StereoEngine {B}x{H}x{W}: sample {i} differs from its B = 1 run, max |diff| {(batched[i:i + 1] - one).abs().max().item():.3e}")
