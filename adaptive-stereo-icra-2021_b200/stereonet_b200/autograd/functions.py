"""torch.autograd.Function wrappers for the adaptation step (adapt.py:381-394).  Forward and backward both run in the
library's CUDA kernels; torch only carries the graph, the saved tensors and a few layout views.

The layers with a weight gradient worth moving off the data path (ConvBnLrelu, ConvC32, RefineHead) serve both schedules of the
adaptation step.  Without fused.WGRAD_STREAM, the weight is their input and they compute its gradient.  With it, the weight's
WgradToken takes the weight's place, and the layer returns its output gradient as the token's gradient and computes no weight
gradient (RefineHead, whose forward reads the weight, then also takes the weight detached: see refine_head_autograd)."""
import torch

from .. import ops
from . import fused


def _c(t):
  return t if t.is_contiguous() else t.contiguous()


def _on_this_stream(*tensors):
  """Tensors allocated on another stream are about to be read by kernels of the current one: tell the caching allocator, or
  their memory could be handed out again on the owning stream while these kernels still run."""
  cur = torch.cuda.current_stream(tensors[0].device)
  for t in tensors:
    t.record_stream(cur)


class WgradToken(torch.autograd.Function):
  """Carries the weight of a conv into the graph on its OWN stream.  forward returns a zero-stride token of the conv's output
  `shape` (one float of storage, no kernel); the layer's Function returns its output gradient dz as the token's gradient, so THIS
  node's backward — which autograd runs on the stream this forward ran on, with the proper event waits — computes the weight
  gradient `wgrad(*saved, dz)` next to the data path instead of inside it: the tensor-bound wgrad kernel overlaps the HBM-bound
  BatchNorm backward of the next layer."""

  @staticmethod
  def forward(ctx, w, shape, wgrad, *saved):
    ctx.save_for_backward(*saved)
    ctx.wgrad = wgrad
    return fused.wgrad_token(shape, w.device)

  @staticmethod
  def backward(ctx, dz):
    saved = ctx.saved_tensors
    dz = _c(dz)
    _on_this_stream(*saved, dz)
    return (ctx.wgrad(*saved, dz), None, None) + (None,) * len(saved)


def _token(conv, shape, wgrad, *saved):
  """conv.weight's WgradToken, made on fused.WGRAD_STREAM; None when no such stream is installed or the weight is frozen."""
  ws = fused.WGRAD_STREAM
  if ws is None or not conv.weight.requires_grad:
    return None
  with torch.cuda.stream(ws):
    return WgradToken.apply(conv.weight, shape, wgrad, *saved)


class ConvBnLrelu(torch.autograd.Function):
  """[x +] LeakyReLU(BN(conv3x3(x) + b)), train (batch stats) or eval (running stats).  `w`: conv.weight, or its WgradToken."""

  @staticmethod
  def forward(ctx, x, w, b, gamma, beta, conv, bn, dil, residual, training):
    g = ops.geom(x.shape, 3, stride=1, dil=dil)
    z, stats = fused.conv3x3_c32(x, conv, g, bias=b.detach(), want_stats=training)
    y, bn_saved = fused.bn_lrelu(z, stats, bn, training, residual=x if residual else None)
    ctx.save_for_backward(x, z, *bn_saved)
    ctx.conv, ctx.g, ctx.residual, ctx.training, ctx.token = conv, g, residual, training, w is not conv.weight
    return y

  @staticmethod
  def backward(ctx, dy):
    x, z, scale, shift, mean, invstd = ctx.saved_tensors
    dy = _c(dy)
    dz, dgamma, dbeta, dbias = ops.bn_lrelu_bwd(z, dy, scale, shift, mean, invstd, ctx.training, lrelu=True)
    dx = None
    if ctx.needs_input_grad[0]:
      dx, _ = fused.conv3x3_c32_dgrad(dz, ctx.conv, ctx.g, residual=dy if ctx.residual else None)
    dw = dz if ctx.token else fused.conv3x3_c32_wgrad(x, dz, ctx.g, tuple(ctx.conv.weight.shape))
    return dx, dw, dbias, dgamma, dbeta, None, None, None, None, None


def conv_bn_lrelu_autograd(x, conv, bn, dil, residual, training):
  g, wshape = ops.geom(x.shape, 3, stride=1, dil=dil), tuple(conv.weight.shape)
  tok = _token(conv, x.shape, lambda x, dz: fused.conv3x3_c32_wgrad(x, dz, g, wshape), x.detach())
  return ConvBnLrelu.apply(x, conv.weight if tok is None else tok, conv.bias, bn.weight, bn.bias, conv, bn, dil, residual, training)


class ConvC32(torch.autograd.Function):
  """Conv2d 32->32 with bias only: 5x5 stride 2 (downsample[1:]) or 3x3 stride 1 (conv_alone).  `w`: conv.weight, or its
  WgradToken."""

  @staticmethod
  def forward(ctx, x, w, b, conv, ksize, stride):
    g = fused.plain_geom(x.shape, ksize, stride)
    ctx.conv, ctx.g, ctx.token = conv, g, w is not conv.weight
    if not ctx.token:
      ctx.save_for_backward(x)               # for the weight gradient; with a token, x is the token's to keep
    return fused.plain_conv(x, conv, g, b.detach())

  @staticmethod
  def backward(ctx, dy):
    dy = _c(dy)
    dx = fused.plain_conv_dgrad(dy, ctx.conv, ctx.g) if ctx.needs_input_grad[0] else None
    dw = dy
    if not ctx.token:
      (x,) = ctx.saved_tensors
      dw = fused.plain_conv_wgrad(x, dy, ctx.g, tuple(ctx.conv.weight.shape))
    return dx, dw, ops.channel_sum(dy), None, None, None


def conv_c32_autograd(x, conv, ksize, stride):
  g, wshape = fused.plain_geom(x.shape, ksize, stride), tuple(conv.weight.shape)
  tok = _token(conv, ops.out_shape(g, False), lambda x, dy: fused.plain_conv_wgrad(x, dy, g, wshape), x.detach())
  return ConvC32.apply(x, conv.weight if tok is None else tok, conv.bias, conv, ksize, stride)


class Conv5x5s2First(torch.autograd.Function):
  """downsample[0]: NCHW image -> channels-last features; only weight/bias gradients (the image needs none)."""

  @staticmethod
  def forward(ctx, img, w, b):
    ctx.save_for_backward(img)
    return ops.conv5x5s2_c3(img, w, b)

  @staticmethod
  def backward(ctx, dy):
    (img,) = ctx.saved_tensors
    dy = _c(dy)
    return None, ops.conv5x5s2_c3_wgrad(img, dy), ops.channel_sum(dy)


class CostVolume(torch.autograd.Function):
  @staticmethod
  def forward(ctx, left, right, D):
    return ops.cost_volume(left, right, D)

  @staticmethod
  def backward(ctx, dcost):
    dl, dr = ops.cost_volume_bwd(_c(dcost))
    return dl, dr, None


class Conv3dOutSoftargmin(torch.autograd.Function):
  """conv3d_alone (32->1) + softmax + expectation.  Outputs (cost [B,D,H,W], pred [B,H,W])."""

  @staticmethod
  def forward(ctx, x, w, b):
    cost, pred, fcs = ops.conv3d_out_softargmin(x, w, b, want_cost=True, want_fcs=x.shape[1] > 2)
    ctx.save_for_backward(x, w, cost, pred)
    ctx.mark_non_differentiable(fcs) if fcs is not None else None
    return cost, pred, fcs

  @staticmethod
  def backward(ctx, dcost_out, dpred, _dfcs=None):
    x, w, cost, pred = ctx.saved_tensors
    dcost = ops.softargmin_bwd(cost, pred, _c(dpred), _c(dcost_out))
    dx, dw, db = ops.conv_c32_taps_bwd(x, w, dcost, 27)
    return dx, dw, db


def conv3d_out_softargmin_autograd(x, conv, want_cost):
  cost, pred, fcs = Conv3dOutSoftargmin.apply(x, conv.weight, conv.bias)
  if want_cost and fcs is not None:
    cost._snb_fcs = fcs
  return (cost if want_cost else None), pred


class Upsample(torch.autograd.Function):
  @staticmethod
  def forward(ctx, pred, H, W, mul):
    ctx.hw, ctx.mul = tuple(pred.shape[-2:]), mul
    return ops.upsample_bilinear(pred, H, W, mul)

  @staticmethod
  def backward(ctx, dout):
    return ops.upsample_bilinear_bwd(_c(dout), ctx.hw[0], ctx.hw[1], ctx.mul), None, None, None


class RefineHead(torch.autograd.Function):
  """Upsample + scale + concat + Conv2d(4->32) + BN + LeakyReLU.  Outputs (up [B,H,W], y [B,H,W,32]).  `tok, w`: None and
  conv.weight, or the weight's WgradToken and the weight detached."""

  @staticmethod
  def forward(ctx, coarse, rgb, tok, w, b, gamma, beta, bn, training):
    up, z, stats = ops.refine_in_conv(coarse, rgb, w, b.detach(), want_stats=training)
    y, bn_saved = fused.bn_lrelu(z, stats, bn, training)
    ctx.save_for_backward(coarse, rgb, w, z, *bn_saved)
    ctx.training, ctx.token = training, tok is not None
    return up, y

  @staticmethod
  def backward(ctx, dup, dy):
    coarse, rgb, w, z, scale, shift, mean, invstd = ctx.saved_tensors
    dz, dgamma, dbeta, dbias = ops.bn_lrelu_bwd(z, _c(dy), scale, shift, mean, invstd, ctx.training, lrelu=True)
    dw = None if ctx.token else ops.refine_in_wgrad(coarse, rgb, dz)
    dcoarse = fused.refine_in_dgrad(dz, dup, w, coarse, rgb) if ctx.needs_input_grad[0] else None
    return dcoarse, None, dz if ctx.token else None, dw, dbias, dgamma, dbeta, None, None


def refine_head_autograd(coarse, rgb, conv, bn, training):
  tok = _token(conv, (rgb.shape[0], rgb.shape[2], rgb.shape[3], 32), ops.refine_in_wgrad, coarse.detach(), rgb)
  w = conv.weight if tok is None else conv.weight.detach()
  return RefineHead.apply(coarse, rgb, tok, w, conv.bias, bn.weight, bn.bias, bn, training)


class RefineTail(torch.autograd.Function):
  """Conv2d(32->1) + add upsampled disparity + ReLU."""

  @staticmethod
  def forward(ctx, x, w, b, up):
    taps = ops.conv_c32_taps(x, w, 9)
    out = ops.tapsum_refine_out(taps, b, up)
    ctx.save_for_backward(x, w, out)
    return out

  @staticmethod
  def backward(ctx, dout):
    x, w, out = ctx.saved_tensors
    dres = ops.relu_bwd(out, _c(dout))
    dx, dw, db = ops.conv_c32_taps_bwd(x, w, dres, 9)
    return dx, dw, db, dres


def refine_tail_autograd(x, conv, up):
  return RefineTail.apply(x, conv.weight, conv.bias, up)
