"""Loss and metric kernels of the adaptation step against plain float64 references: snb_photo_loss (photo_loss.cu, where every
backward pass of the step starts), snb_khamis_loss and snb_eval_metrics (metrics.cu), at the KITTI (376x1248, 375x1242) and
SceneFlow (540x960) shapes, at the edges of the photometric kernel's 16x64 tiles, and at the warp's edge cases.

snb_photo_loss.  The reference restates O.monodepth_single_loss in float64 and takes d loss / d disp by float64 autograd.
The one part kept in fp32 is the sample coordinate (gx, gy, the valid mask, ix, iy, their clamping): the reference computes it
in fp32 and the kernel follows it (warp_coord), so it is recomputed here in fp32 op by op and carried into float64 with a
straight-through derivative.  With those shared, the sample cell and every mask decision are identical on both sides.  The
data keep every other kink away by construction, each checked by an assertion on the test setup:
  - left image in [0.75, 1], right image in [0, 0.25]: L - I^ > 0 at every pixel (no L1 sign flip), and the 3x3 means keep
    mu_L >= 3 mu_I, so the luminance factor 2 mu_L mu_I / (mu_L^2 + mu_I^2) <= 0.6.  Since |contrast-structure| <= 1, the SSIM
    argument (1 - n/d) / 2 stays within [0.2, 0.8], far from the clamp.  (L in (0.5, 1] and I^ in [0, 0.5) would not do: two
    means just either side of 0.5 give a luminance factor near 1.)
  - neighbouring disparities differ by at least 1/8 px, or by exactly 0 (no smoothness sign flip).
Every bounded check has its bound and the reason beside it; no check uses an outlier fraction or a cosine similarity."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from stereonet_b200 import ops
from stereonet_b200.losses import monodepth_single_loss
from test_gpu_backward_kernels import bounded as bounded_cpu, dyadic, exact, gen, ints
from test_gpu_kernels import DEV, rnd

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                      # unit roundoff of fp32
C1, C2 = 0.01 ** 2, 0.03 ** 2       # SSIM constants (loss_functions.py)


def bounded(got, ref, bound, what):
  """test_gpu_backward_kernels.bounded with a bound that may live on the GPU."""
  bounded_cpu(got, ref, bound.detach().cpu() if isinstance(bound, torch.Tensor) else float(bound), what)


# ================================================================================================ 1. snb_photo_loss
def warp_coords(disp):
  """fp32 sample coordinates of photo_loss.cu warp_coord (linear_warping.py's grid + grid_sample's unnormalize and border
  clip, align_corners=False), op by op on the CPU: gx = (2 (col - d)) / W - 1, gy likewise, valid = both in [-1, 1],
  ix = ((gx + 1) W - 1) / 2 clamped to [0, W - 1], iy likewise.  The kernel evaluates (gx + 1) W - 1 as one fused
  multiply-add (FFMA in its SASS); the product of an fp32 value and W is exact in float64, so rounding (gx + 1) W - 1 once
  to fp32 reproduces it.  Returns valid, ix, iy (fp32, clamped) and `clamped` (ix clamped: zero x gradient)."""
  B, H, W = disp.shape
  d = disp.detach().cpu().float()
  col = torch.arange(W, dtype=torch.float32).view(1, 1, W)
  row = torch.arange(H, dtype=torch.float32).view(1, H, 1)
  gx = (2.0 * (col - d)) / W - 1.0
  gy = ((2.0 * row) / H - 1.0).expand(B, H, W)
  valid = (gx >= -1.0) & (gx <= 1.0) & (gy >= -1.0) & (gy <= 1.0)
  ix = ((gx + 1.0).double() * W - 1.0).float() * 0.5
  iy = ((gy + 1.0).double() * H - 1.0).float() * 0.5
  clamped = (ix <= 0) | (ix >= W - 1)
  return valid, ix.clamp(0, W - 1), iy.clamp(0, H - 1), clamped, gx


def sum3x3(x):
  """3x3 sum with zero padding ([B,C,H,W])."""
  return F.avg_pool2d(x, 3, 1, 1, count_include_pad=True) * 9


def photo_ref(left, right, disp, smooth_w):
  """float64 restatement of O.monodepth_single_loss(left, right, disp[:, None], smooth_w) on DEV, its gradient by float64
  autograd, and the per-pixel / per-loss error bounds of the fp32 kernel (see photo_bound_terms).  Coordinates: warp_coords,
  carried into float64 as ix64 = ix32 + gmul (d.detach() - d), so d ix / d d = -gmul (0 where ix was clamped)."""
  B, _, H, W = left.shape
  valid, ix32, iy32, clamped, gx = warp_coords(disp)
  f64 = lambda t: t.to(DEV, torch.float64)
  L, R = f64(left), f64(right)
  d = f64(disp).requires_grad_()
  gmul = f64(~clamped)
  x0, y0 = ix32.floor(), iy32.floor()
  wx = f64(ix32 - x0) + gmul * (d.detach() - d)
  wy = f64(iy32 - y0)
  x0, y0 = x0.long().to(DEV), y0.long().to(DEV)
  x1ok, y1ok = x0 + 1 <= W - 1, y0 + 1 <= H - 1          # out-of-image corners weigh 0 (grid_sample)
  x1, y1 = torch.where(x1ok, x0 + 1, x0), torch.where(y1ok, y0 + 1, y0)
  wxb, wyb = torch.where(x1ok, wx, torch.zeros_like(wx)), torch.where(y1ok, wy, torch.zeros_like(wy))
  Rf = R.reshape(B, 3, H * W)

  def at(yy, xx):
    return Rf.gather(2, (yy * W + xx).reshape(B, 1, H * W).expand(B, 3, H * W)).view(B, 3, H, W)
  r00, r01, r10, r11 = at(y0, x0), at(y0, x1), at(y1, x0), at(y1, x1)
  u1 = lambda t: t.unsqueeze(1)
  I = (u1((1 - wx) * (1 - wy)) * r00 + u1(wxb * (1 - wy)) * r01 + u1((1 - wx) * wyb) * r10 + u1(wxb * wyb) * r11)

  pool = lambda t: F.avg_pool2d(t, 3, 1, 1)
  mx, my = pool(L), pool(I)
  sLL, sII = pool(L * L), pool(I * I)
  sx, sy, sxy = sLL - mx * mx, sII - my * my, pool(L * I) - mx * my
  a, bb = 2 * mx * my + C1, 2 * sxy + C2
  cc, e = mx * mx + my * my + C1, sx + sy + C2
  raw = (1 - a * bb / (cc * e)) / 2
  ssim = raw.clamp(0, 1).mean(1)
  l1 = (L - I).abs().mean(1)
  m = d.mean((1, 2), keepdim=True) + 1e-7
  dn = d / m
  ex = torch.exp(-(L[..., :-1] - L[..., 1:]).abs().mean(1))
  ey = torch.exp(-(L[..., :-1, :] - L[..., 1:, :]).abs().mean(1))
  sdx = F.pad((dn[..., :-1] - dn[..., 1:]).abs() * ex, (0, 1))
  sdy = F.pad((dn[..., :-1, :] - dn[..., 1:, :]).abs() * ey, (0, 0, 0, 1))
  total = 0.85 * ssim + 0.15 * l1 + smooth_w * (sdx + sdy)
  mask = valid.to(DEV)
  loss = total[mask].mean()
  per = torch.stack([total[b][mask[b]].mean() for b in range(B)])
  loss.backward()

  with torch.no_grad():
    cnt = mask.double().sum((1, 2))
    dd = d.detach()
    exsum = F.pad(ex, (0, 1)) + F.pad(ex, (1, 0)) + F.pad(ey, (0, 0, 0, 1)) + F.pad(ey, (0, 0, 1, 0))
    dimag = u1(gmul) * (u1(1 - wy) * (r00.abs() + r01.abs()) + u1(wy) * (r10.abs() + r11.abs()))
    P, V = photo_bound_terms(L, I.detach(), mask, mx, my, sLL, sII, a, bb.detach(), cc, e.detach(), dimag)
    mb = m.detach()
    Hm = smooth_w * exsum / mb
    Cm = smooth_w * (exsum * dd.abs()).sum((1, 2), keepdim=True) / (mb * mb * H * W)
    tot_cnt = cnt.sum()
    # ddisp: PHOTO_GRAD_C u of the photometric magnitude P (photo_bound_terms); 16 u of the smoothness and coupling terms
    # (__expf within a few ulps for arguments in [-1, 0], h sums <= 4 terms, h * inv_m and the fp32 mean disparity + 1e-7
    # round once each; T sums fp32 products in double, block partials are rounded to fp32 once, coupling ~ 1 / m^2); all over
    # the batch count
    gbound = U * (PHOTO_GRAD_C * P + 16 * Hm + 16 * Cm) / tot_cnt
    # loss: PHOTO_VALUE_C u of each valid pixel's value magnitude (photo_bound_terms, plus the smoothness value |df| ex), plus
    # the rounding of the block partials to fp32 and of the final quotient (<= u |loss| each)
    sval = (sdx + sdy).detach()
    Vpix = mask.double() * (V + smooth_w * sval)
    lbound = U * PHOTO_VALUE_C * Vpix.sum() / tot_cnt + 2 * U * loss.detach().abs()
    pbound = U * PHOTO_VALUE_C * Vpix.sum((1, 2)) / cnt + 2 * U * per.detach().abs()
  return dict(loss=loss.detach(), per=per.detach(), ddisp=d.grad.detach(), gbound=gbound, lbound=lbound, pbound=pbound,
              raw=raw.detach(), LmI=(L - I).detach(), valid=valid, clamped=clamped, ix=ix32, gx=gx, cnt=cnt, m=mb.flatten())


# Constants of the photometric bounds, set from a B200 measurement (1000 W limit) over every snb_photo_loss case of this
# file: the largest ddisp error at smooth_w = 0 was 0.21 u P / count (1x2x63; <= 0.084 at the KITTI and SceneFlow shapes) and
# the largest loss error 0.14 u sum(V) / count beyond the final roundings (exact 2x16x512); each constant is about twice that.
# The operation count alone gives ~60 + 24 M / e roundings per term (photo_bound_terms), far above the measured error: the
# coefficient errors are correlated (they share the rounded moments) and largely cancel in k0 + k1 L + k2 I^.  At these
# constants the ddisp bound is ~1e-3 of |ddisp| at the median pixel (>= 6 % of it at ~1 % of pixels), and the loss bound
# ~2.6e-7 of the loss at 376x1248.
PHOTO_GRAD_C = 0.45
PHOTO_VALUE_C = 0.3


def photo_bound_terms(L, I, mask, mx, my, sLL, sII, a, bb, cc, e, dimag):
  """Float64 magnitudes of the photometric terms the kernel adds for each pixel's gradient (P [B,H,W]) and loss value
  (V [B,H,W]), each carrying the one factor (1 + M / e) by which the fp32 variances lose accuracy.

  Gradient: g = sum_c dI^_c/dd * (sum over the 3x3 centres q of k0_q + k1_q L + k2_q I^, + 0.05 sign(I^ - L)), with the
  analytic SSIM coefficients k0 = -(mu_L (b - a) / dn - n mu_I (e - c) / dn^2) / 9, k1 = -a / (9 dn), k2 = n c / (9 dn^2)
  (n = a b, dn = c e).  The variances are E[x^2] - mu^2 in fp32: their absolute error is a few u (E[L^2] + E[I^2]), which
  reaches e and b (both only >= C2) with the relative factor M / e = (E[L^2] + E[I^2]) / e.  P is the sum over channels of
  |dI^/dd| terms times (sum over centres of (|k0| + |k1 L| + |k2 I^|) (1 + M / e) + 0.05), with |k0| the sum of its two
  terms' magnitudes.  V: 0.85/3 (|n / dn| (1 + M / e) + 1) / 2 for the SSIM term, 0.15/3 (|L| + |I^|) for the L1 term."""
  w = u1c(mask) * (0.85 / 3)
  amp = 1 + (sLL + sII) / e.abs()           # e >= C2 > 0 in exact arithmetic; abs() only guards the factor
  dn = cc * e.abs()
  n = a * bb
  k0 = ((mx * (bb - a)).abs() / dn + (n * my * (e - cc)).abs() / (dn * dn)) / 9 * amp
  k1 = a.abs() / dn / 9 * amp
  k2 = (n * cc).abs() / (dn * dn) / 9 * amp
  kap = sum3x3(w * k0) + sum3x3(w * k1) * L.abs() + sum3x3(w * k2) * I.abs() + 0.05 * u1c(mask)
  P = (kap * dimag).sum(1)
  V = ((0.85 / 3) * 0.5 * ((n / dn).abs() * amp + 1) + (0.15 / 3) * (L.abs() + I.abs())).sum(1)
  return P, V


def u1c(mask):
  return mask.double().unsqueeze(1)


def photo_images(B, H, W, seed):
  """Left image in [0.75, 1], right image in [0, 0.25] (see the module docstring)."""
  g = gen(seed)
  return 0.75 + 0.25 * torch.rand(B, 3, H, W, generator=g), 0.25 * torch.rand(B, 3, H, W, generator=g)


def smooth_disp(B, H, W, seed, quarter=False):
  """A smooth field (slope <= 0.08 px per pixel in either direction) with a different mean per sample, plus ((x + 2y) mod 5)/4,
  whose steps are 1/4 or -1 along x and 1/2 or -3/4 along y: neighbours differ by >= 1/4 - 0.08 > 1/8.  quarter: the field
  rounded to multiples of 1/4, so every disparity is on a 1/4 grid (neighbours then differ by 0 or >= 1/4)."""
  g = gen(seed)
  y = torch.arange(H, dtype=torch.float64).view(1, H, 1)
  x = torch.arange(W, dtype=torch.float64).view(1, 1, W)
  ph = torch.rand(B, 2, generator=g, dtype=torch.float64) * 6.28
  base = (0.02 * W + 0.5) * (1 + 0.4 * torch.arange(B, dtype=torch.float64)).view(B, 1, 1)
  wave = torch.sin(0.05 * x + ph[:, 0].view(B, 1, 1)) * torch.cos(0.03 * y + ph[:, 1].view(B, 1, 1))
  field = base + 0.03 * x * (W > 64) + min(1.0, 0.1 * W) * wave        # W = 2: a small wave keeps the mean away from 0
  if quarter:
    field = torch.round(field * 4) / 4
  return (field + ((x + 2 * y) % 5) / 4).float()


def check_photo_setup(ref, disp, what, allow_equal=False, samples=None):
  """The data keep the kernel's kinks away: asserted, not assumed (for the given samples; default all)."""
  sel = slice(None) if samples is None else list(samples)
  raw, disp = ref["raw"][sel], disp[sel]
  assert float(raw.min()) >= 0.19 and float(raw.max()) <= 0.81, f"test setup ({what}): SSIM argument reaches the clamp"
  assert float(ref["LmI"][sel].min()) > 0, f"test setup ({what}): L - I^ <= 0 somewhere (L1 sign flip)"
  for dd in (disp[..., 1:] - disp[..., :-1], disp[..., 1:, :] - disp[..., :-1, :]):
    a = dd.abs()
    near = (a < 0.125) & ~(allow_equal & (a == 0))
    assert not bool(near.any()), f"test setup ({what}): neighbouring disparities closer than 1/8 px"
  assert float(ref["cnt"][sel].min()) > 0 and float(ref["m"][sel].min()) > 0.25, f"test setup ({what}): empty mask or tiny mean"


def run_photo(left, right, disp, smooth_w):
  loss, ddisp = ops.photo_loss(left.to(DEV), right.to(DEV), disp.to(DEV).contiguous(), smooth_w)
  return loss.cpu(), ddisp


def check_photo(left, right, disp, smooth_w, what, allow_equal=False):
  ref = photo_ref(left, right, disp, smooth_w)
  check_photo_setup(ref, disp, what, allow_equal)
  loss, ddisp = run_photo(left, right, disp, smooth_w)
  bounded(loss[0], ref["loss"], ref["lbound"], f"{what}: loss_out[0] (photo_loss_finalize_kernel)")
  bounded(loss[1:], ref["per"], ref["pbound"], f"{what}: loss_out[1 + b] (photo_loss_finalize_kernel)")
  bounded(ddisp, ref["ddisp"], ref["gbound"], f"{what}: ddisp (photo_loss_tile_kernel + finalize)")
  return ref, loss, ddisp


SMOOTH_W = [0.0, 1e-3, 1.0]     # photometric term alone; the product weight; smoothness and coupling as large as photometric
PHOTO_SHAPES = ([(1, 376, 1248), (2, 376, 1248), (1, 375, 1242), (2, 375, 1242), (4, 540, 960)]
                + [(1, h, w) for h in (2, 15, 16, 17) for w in (2, 63, 64, 65)])


@pytest.mark.parametrize("smooth_w", SMOOTH_W)
@pytest.mark.parametrize("B,H,W", PHOTO_SHAPES)
def test_photo_loss(B, H, W, smooth_w):
  """Loss, per-sample loss and ddisp at every pixel against the float64 reference.  KITTI 376x1248 (the last tile row is
  ragged) and 375x1242 (ragged both ways), SceneFlow 540x960 x 4, and H in {2, 15, 16, 17} x W in {2, 63, 64, 65} around the
  16x64 tile and its 2-pixel halo.  The disparities leave the left columns masked (col - d < 0) with some valid-but-clamped
  pixels (col - d in [0, 0.5)) next to them."""
  left, right = photo_images(B, H, W, seed=H * 131 + W)
  disp = smooth_disp(B, H, W, seed=H + 7 * W)
  check_photo(left, right, disp, smooth_w, f"snb_photo_loss {B}x{H}x{W} smooth_w={smooth_w}")


@pytest.mark.parametrize("smooth_w", SMOOTH_W)
@pytest.mark.parametrize("B,H,W", [(1, 64, 1024), (2, 16, 512)])
def test_photo_loss_exact_coordinates(B, H, W, smooth_w):
  """Power-of-two H and W with disparities on a 1/4 grid: every fp32 step of the coordinate pipeline is exact, so the
  reference is float64 throughout (no fp32 coordinate shared with the kernel).  ix = col - d - 1/2 lands on integers, so
  sample cells start exactly on pixel centres."""
  left, right = photo_images(B, H, W, seed=5 + W)
  disp = smooth_disp(B, H, W, seed=11 + H, quarter=True)
  ref = check_photo(left, right, disp, smooth_w, f"snb_photo_loss exact {B}x{H}x{W} smooth_w={smooth_w}", allow_equal=True)[0]
  col = torch.arange(W, dtype=torch.float64)
  ix_exact = (col - disp.double() - 0.5).clamp(0, W - 1)
  assert torch.equal(ref["ix"].double(), ix_exact), "test setup: the fp32 coordinate pipeline is not exact here"


def regime_disp(B, H, W, seed):
  """Disparities on a 1/4 grid covering every warp regime: masked and clamped (col - d < 0), valid but clamped (col - d in
  [0, 0.5): d = col - 1/4 and d = col, gx = -1 exactly), the right border (last column, d in (-1, -1/2]: valid, ix clamped to
  W - 1, the x + 1 corner outside the image; d = -1 gives gx = 1 exactly), and negative disparity masked by gx > 1 (last
  columns, d < col - W).  Elsewhere random multiples of 1/4 in [1, 12]."""
  g = gen(seed)
  d = ints((B, H, W), 4, 48, seed) / 4
  col = torch.arange(W, dtype=torch.float32)
  pick = torch.randint(0, 4, (B, H), generator=g)
  for b in range(B):
    for y in range(H):
      k = int(pick[b, y])
      c = (y % 6) + 1
      if c < W:
        d[b, y, c] = col[c] - (0.25 if k % 2 else 0.0)          # valid, clamped at the left border
      d[b, y, W - 1] = (-0.75, -1.0, -1.25, -0.5)[k]            # right border: clamped-valid, gx = 1, masked (gx > 1), clamped
      if W > 2:
        d[b, y, W - 2] = (-1.5, -0.75, -2.25, 3.0)[k]           # ix = W - 1 exactly; unclamped; masked (gx > 1); positive
  return d


@pytest.mark.parametrize("smooth_w", SMOOTH_W)
@pytest.mark.parametrize("B,H,W", [(2, 16, 64), (1, 17, 65), (1, 16, 128)])
def test_photo_loss_warp_regimes(B, H, W, smooth_w):
  """Every warp regime (regime_disp) against the same reference; each regime is asserted to occur."""
  left, right = photo_images(B, H, W, seed=3 * W)
  disp = regime_disp(B, H, W, seed=W + H)
  ref = check_photo(left, right, disp, smooth_w, f"snb_photo_loss regimes {B}x{H}x{W} smooth_w={smooth_w}", allow_equal=True)[0]
  v, c, ix, gx = ref["valid"], ref["clamped"], ref["ix"], ref["gx"]
  assert bool((~v & c & (gx < -1)).any()), "test setup: no masked-and-clamped pixel"
  assert bool((v & c & (ix == 0)).any()), "test setup: no valid-but-clamped pixel at the left border"
  assert bool((v & c & (ix == W - 1)).any()), "test setup: no valid pixel clamped at the right border"
  assert bool((~v & (gx > 1)).any()), "test setup: no negative disparity masked by gx > 1"


@pytest.mark.parametrize("smooth_w", SMOOTH_W)
def test_photo_loss_constant_region(smooth_w):
  """A region of constant disparity (rows 3-12, columns 20-90, across a tile boundary): there df == 0 exactly, and both
  implementations take the zero sub-gradient of |df|.  (Computed as d_a * inv_m - d_b * inv_m, the difference contracted to
  an FMA and left the rounding error of d_a * inv_m, of either sign: a smoothness gradient of +-exp(.) where the reference
  has 0.  The quarter-grid cases of test_photo_loss_exact_coordinates and test_photo_loss_warp_regimes have such ties too.)"""
  B, H, W = 1, 20, 130
  left, right = photo_images(B, H, W, seed=17)
  disp = smooth_disp(B, H, W, seed=19, quarter=True)
  disp[:, 3:13, 20:91] = 6.25
  check_photo(left, right, disp, smooth_w, f"snb_photo_loss constant region smooth_w={smooth_w}", allow_equal=True)


def test_photo_loss_empty_mask():
  """No valid pixel in the batch (every col - d < 0).  The reference's total[mask].mean() is NaN and its gradient all zeros;
  the kernel must give the same: loss_out all NaN, ddisp exactly 0 (not 0 * (1 / 0) = NaN)."""
  B, H, W = 2, 17, 65
  left, right = photo_images(B, H, W, seed=23)
  disp = W + 0.5 + ints((B, H, W), 0, 8, seed=29) / 4
  ref = photo_ref(left, right, disp, 1.0)
  assert math.isnan(float(ref["loss"])) and bool(torch.isnan(ref["per"]).all()), "reference: the loss over an empty mask is NaN"
  assert float(ref["ddisp"].abs().max()) == 0.0, "reference: the gradient over an empty mask is 0"
  for smooth_w in SMOOTH_W:
    loss, ddisp = run_photo(left, right, disp, smooth_w)
    assert bool(torch.isnan(loss).all()), f"empty mask smooth_w={smooth_w}: loss_out {loss.tolist()} should be NaN"
    exact(ddisp, torch.zeros(B, H, W), f"empty mask smooth_w={smooth_w}: ddisp (photo_loss_finalize_kernel)")


@pytest.mark.parametrize("smooth_w", SMOOTH_W)
def test_photo_loss_one_sample_masked(smooth_w):
  """B = 3 with sample 1 fully masked: loss_out[1 + b] per sample (NaN for sample 1, as the reference's one-pair loss) and
  loss_out[0] over the batch count; sample 1's ddisp is exactly 0, the others against the reference."""
  B, H, W = 3, 40, 150
  left, right = photo_images(B, H, W, seed=31)
  disp = smooth_disp(B, H, W, seed=37)
  disp[1] = W + 1.0 + ints((H, W), 0, 8, seed=41) / 4
  ref = photo_ref(left, right, disp, smooth_w)
  assert float(ref["cnt"][1]) == 0 and math.isnan(float(ref["per"][1])), "test setup: sample 1 is not fully masked"
  what = f"snb_photo_loss one sample masked smooth_w={smooth_w}"
  keep = [0, 2]
  check_photo_setup(ref, disp, what, samples=keep)
  loss, ddisp = run_photo(left, right, disp, smooth_w)
  bounded(loss[0], ref["loss"], ref["lbound"], f"{what}: loss_out[0]")
  assert math.isnan(float(loss[2])), f"{what}: loss_out[2] = {float(loss[2])} (sample 1 has no valid pixel: NaN)"
  bounded(loss[1:][keep], ref["per"][keep], ref["pbound"][keep], f"{what}: loss_out[1 + b], b = 0, 2")
  exact(ddisp[1], torch.zeros(H, W), f"{what}: ddisp of the masked sample")
  bounded(ddisp, ref["ddisp"], ref["gbound"], f"{what}: ddisp")


def test_photo_loss_scales_by_incoming_gradient():
  """losses.monodepth_single_loss: backward with grad_output 2.0 gives exactly twice snb_photo_loss's ddisp."""
  B, H, W = 2, 376, 1248
  left, right = photo_images(B, H, W, seed=43)
  disp = smooth_disp(B, H, W, seed=47).to(DEV)
  l, r = left.to(DEV), right.to(DEV)
  _, ddisp = ops.photo_loss(l, r, disp, 1e-3)
  d = disp.unsqueeze(1).clone().requires_grad_()
  monodepth_single_loss(l, r, {"pred_disp_l/0": d}, 0).backward(torch.tensor(2.0, device=DEV))
  exact(d.grad.squeeze(1), 2.0 * ddisp, "monodepth_single_loss backward(2.0)")


# ================================================================================================ 2. snb_khamis_loss
def khamis_ref(pred, gt):
  """float64: loss = sum_{gt > 0} (sqrt((gt - pred)^2 + 4) / 2 - 1) / max(#valid, 1), and the kernel's dpred rounded once per
  step in its order, fl(fl(fl(-0.5 d) / fl(sqrt(d^2 + 4))) * fl(1 / nv)).  With integer d, d^2 + 4 is exact; float64 sqrt
  and division rounded to fp32 are the correctly rounded fp32 results (53 >= 2 * 24 + 2), as are sqrtf and '/' in a build
  without --use_fast_math (test_khamis_build_flags)."""
  p, g = pred.double().flatten(), gt.double().flatten()
  valid = g > 0
  d = (g - p).float().double()
  nv = max(int(valid.sum()), 1)
  r32 = torch.sqrt(d * d + 4).float().double()
  gr = ((-0.5 * d).float().double() / r32).float().double()
  dpred = torch.where(valid, (gr * float(np.float32(1.0 / nv))).float().double(), torch.zeros_like(d))
  terms = torch.where(valid, torch.sqrt(d * d + 4) / 2 - 1, torch.zeros_like(d))
  mags = torch.where(valid, torch.sqrt(d * d + 4) / 2 + 1, torch.zeros_like(d))
  return terms.sum() / nv, dpred.view(pred.shape), mags.sum() / nv


def khamis_blocks(n):
  return int(min(max((n + 1023) // 1024, 1), 592))


def test_khamis_build_flags():
  """dpred is held bit-exact to correctly rounded sqrt and division: the library must not be built with fast math."""
  import importlib.util
  import os
  spec = importlib.util.spec_from_file_location(
      "snb200_build_flags", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                         "adaptive-stereo-icra-2021_b200", "build.py"))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  flags = " ".join(mod.FLAGS)
  for f in ("fast_math", "fast-math", "prec-div=false", "prec_div=false", "prec-sqrt=false", "prec_sqrt=false", "ftz=true"):
    assert f not in flags, f"build.py passes {f}: sqrtf / division would no longer be correctly rounded"


# n: one element; the KITTI frame at B = 1; 592 * 1024 (the last n before the block count caps at 592) and one past it;
# KITTI at B = 2 (938 496 elements: 592 blocks, each thread's grid-stride loop runs 7 times)
KHAMIS_SHAPES = [(1,), (1, 376, 1248), (592 * 1024,), (592 * 1024 + 1,), (2, 376, 1248)]


@pytest.mark.parametrize("shape", KHAMIS_SHAPES)
def test_khamis_loss(shape):
  """Integer gt - pred (gt in [-20, 200], about 10 % invalid: gt <= 0), so dpred is bit-exact (khamis_ref).  The loss sums
  fp32 terms: each thread adds k = ceil(n / (blocks * 256)) grid-stride terms, the warp tree 5 levels, the block 8 warp sums;
  the block partials are summed in double.  Each term 0.5 r - 1 is one fmaf on a correctly rounded r.  Bound:
  (k + 16) u of sum(0.5 r + 1) / nv, + u |loss| for the final rounding."""
  n = int(np.prod(shape))
  g = ints(shape, -20, 200, seed=n % 9973)
  pred = g - ints(shape, -300, 300, seed=n % 9973 + 1)
  loss_ref, dpred_ref, mag = khamis_ref(pred, g)
  loss, dpred = ops.khamis_loss(pred.to(DEV), g.to(DEV))
  what = f"snb_khamis_loss n={n}"
  exact(dpred, dpred_ref, what + ": dpred (khamis_partial_kernel + finalize)")
  k = -(-n // (khamis_blocks(n) * 256))
  bounded(loss.cpu()[0], loss_ref, (k + 16) * U * float(mag) + U * abs(float(loss_ref)), what + ": loss")


def test_khamis_loss_single_valid_and_all_invalid():
  """One valid pixel in a KITTI frame (nv = 1), a single-element input, and a frame with no valid pixel: loss 0 and dpred 0
  (sum over nothing / max(0, 1))."""
  H, W = 376, 1248
  pred = ints((1, H, W), -50, 50, seed=3)
  gt = torch.zeros(1, H, W)
  gt[0, 200, 777] = 37.0
  for p, g, what in ((pred, gt, "one valid pixel"), (pred[:, :1, :1].contiguous(), gt[:, 200:201, 777:778].contiguous(), "n = 1"),
                     (pred, -ints((1, H, W), 0, 5, seed=4), "all invalid")):
    loss_ref, dpred_ref, mag = khamis_ref(p, g)
    loss, dpred = ops.khamis_loss(p.to(DEV), g.to(DEV))
    exact(dpred, dpred_ref, f"snb_khamis_loss {what}: dpred")
    bounded(loss.cpu()[0], loss_ref, 17 * U * float(mag) + U * abs(float(loss_ref)), f"snb_khamis_loss {what}: loss")


def test_khamis_loss_random():
  """Random floats at KITTI B = 2.  dpred within 6 u of its float64 value: gt - pred rounds once (d / r is no more sensitive
  to d than d itself: 4 / r^2 <= 1), fmaf + sqrtf 1.5 u, the division 1 u, fp32(1 / nv) and the product 2 u.  The loss as in
  test_khamis_loss."""
  shape = (2, 376, 1248)
  g = torch.rand(shape, generator=gen(5)) * 80 + 0.5
  g[torch.rand(shape, generator=gen(6)) < 0.3] = 0.0
  pred = g + 5.0 * rnd(*shape, seed=7)
  p64, g64 = pred.double(), g.double()
  valid = g64 > 0
  nv = int(valid.sum())
  d = g64 - p64
  r = torch.sqrt(d * d + 4)
  dref = torch.where(valid, -0.5 * d / r / nv, torch.zeros_like(d))
  lref = torch.where(valid, r / 2 - 1, torch.zeros_like(d)).sum() / nv
  loss, dpred = ops.khamis_loss(pred.to(DEV), g.to(DEV))
  bounded(dpred, dref, 5 * U * dref.abs() + U * (0.5 * d.abs() / r / nv), "snb_khamis_loss (random): dpred")
  k = -(-shape[0] * shape[1] * shape[2] // (592 * 256))
  bounded(loss.cpu()[0], lref, (k + 16) * U * float(torch.where(valid, r / 2 + 1, torch.zeros_like(r)).sum() / nv)
          + U * abs(float(lref)), "snb_khamis_loss (random): loss")


# ================================================================================================ 3. snb_eval_metrics
THRESH = (2.0, 3.0, 4.0, 5.0)
# |pred - gt| values: exactly on each threshold (not counted: the test is strictly greater), 1/64 either side, 0, and far off
ERRS = torch.tensor([0.0, 0.5, 2.0, 2 - 1 / 64, 2 + 1 / 64, 3.0, 3 - 1 / 64, 3 + 1 / 64, 4.0, 4 - 1 / 64, 4 + 1 / 64, 5.0,
                     5 - 1 / 64, 5 + 1 / 64, 7.25, 40.0])


def metrics_ref(pred, gt):
  """[B, 6] float64: sum |fl(pred - gt)| over gt > 0, #valid, #(|e| > t) for t = 2, 3, 4, 5."""
  B = pred.shape[0]
  e = (pred - gt).abs().double().view(B, -1)
  v = (gt > 0).view(B, -1)
  cols = [torch.where(v, e, torch.zeros_like(e)).sum(1), v.sum(1).double()]
  cols += [(v & (e > t)).sum(1).double() for t in THRESH]
  return torch.stack(cols, 1)


@pytest.mark.parametrize("B,H,W", [(1, 376, 1248), (8, 376, 1248), (4, 540, 960)])
def test_eval_metrics_exact(B, H, W):
  """gt multiples of 1/4 in [-190, 190] (gt <= 0 invalid) and pred = gt +- an error from ERRS: every difference and its
  absolute value are exact in fp32, so the counts, including errors exactly on 2, 3, 4 and 5 px, must be exact, and the
  double accumulation of sum |e| is exact (multiples of 1/64 far below 2^53 / 64), rounded once to fp32."""
  gt = dyadic((B, H, W), 760, 4, seed=B * 7 + H)
  pick = torch.randint(0, len(ERRS), (B, H, W), generator=gen(B + W))
  sign = torch.where(torch.rand(B, H, W, generator=gen(H)) < 0.5, -1.0, 1.0)
  pred = gt + sign * ERRS[pick]
  assert bool(((pred - gt).abs() == ERRS[pick]).all()), "test setup: pred - gt is not exact in fp32"
  ref = metrics_ref(pred, gt)
  assert bool((ref[:, 1] < 2 ** 24).all())
  got = ops.eval_metrics(pred.to(DEV), gt.to(DEV))
  exact(got, ref.float(), f"snb_eval_metrics {B}x{H}x{W}")


@pytest.mark.parametrize("B,H,W", [(1, 376, 1248), (8, 376, 1248), (4, 540, 960)])
def test_eval_metrics_random(B, H, W):
  """Random floats.  Counts exact against float64 comparisons of the same fp32 differences.  sum |e| against a float64 sum
  of the same fp32 |pred - gt|: within one fp32 rounding (u |sum|) plus the double accumulation error (n 2^-53 |sum|)."""
  gt = torch.rand(B, H, W, generator=gen(B + 1)) * 80 - 8
  pred = gt + 4.0 * rnd(B, H, W, seed=B + 2)
  ref = metrics_ref(pred, gt)
  got = ops.eval_metrics(pred.to(DEV), gt.to(DEV)).cpu()
  what = f"snb_eval_metrics (random) {B}x{H}x{W}"
  exact(got[:, 1:], ref[:, 1:].float(), what + ": counts")
  bounded(got[:, 0], ref[:, 0], (U + H * W * 2.0 ** -53) * ref[:, 0].abs(), what + ": sum |e|")
