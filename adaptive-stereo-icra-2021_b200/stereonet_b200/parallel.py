"""Multi-GPU partitioning of the hot path (SURVEY.md §8e): batched inference and independent adaptation streams are
embarrassingly parallel — one process per GPU, contiguous shards, no data-path collective.  The only exchange step in
scope is shared-model multi-stream adaptation: ONE NCCL all-reduce per step over a flat fp32 buffer that holds the gradients of
the used parameters (optim.FusedAdamClip.flat_grad — autograd's per-parameter gradients are gathered into it by one kernel and
the fused clip + Adam kernel reads it directly: no unpack) followed by the BatchNorm running statistics (BNBucket), so that the
replicas stay identical INCLUDING buffers (the reference has no SyncBN; averaging the running statistics is what §8e specifies)."""
import torch
import torch.distributed as dist


def shard_range(n_items, rank, world):
  """Contiguous balanced shard [lo, hi) of n_items for `rank` of `world` (first n_items % world ranks get one more)."""
  if not (0 <= rank < world):
    raise ValueError("rank out of range")
  base, rem = divmod(n_items, world)
  lo = rank * base + min(rank, rem)
  return lo, lo + base + (1 if rank < rem else 0)


def used_parameters(stereo_net, feature_net):
  """Parameters that ever receive a gradient, in optimizer order (stereo_net first, adapt.py:208-210).
  BasicBlock.conv2 is constructed but never called (stereo_net.py:40,44-51) -> excluded, as Adam skips grad=None."""
  out = []
  for net in (stereo_net, feature_net):
    for name, p in net.named_parameters():
      if ".conv2." not in name:
        out.append(p)
  return out


def used_bn_buffers(stereo_net, feature_net):
  """running_mean / running_var of every BatchNorm layer that runs (conv2's never does), stereo_net first."""
  out = []
  for net in (stereo_net, feature_net):
    for name, m in net.named_modules():
      if isinstance(m, (torch.nn.BatchNorm2d, torch.nn.BatchNorm3d)) and ".conv2." not in "." + name + ".":
        out += [m.running_mean, m.running_var]
  return out


class DPBucket:
  """One flat fp32 tensor = [gradient bucket | BN running statistics].  The BN buffers of the modules are re-pointed to views of
  the second part (values preserved; state_dict is unaffected), the gradient part is `optimizer.flat_grad` re-pointed likewise —
  so a step needs no gather / scatter around the collective: all_reduce(SUM) over the whole tensor, the 1 / world of the gradient
  part is folded into the fused clip + Adam kernel, the statistics part is scaled in place (one tiny kernel)."""

  def __init__(self, optimizer, stereo_net, feature_net):
    self.opt = optimizer
    bufs = used_bn_buffers(stereo_net, feature_net)
    n_g = optimizer.n_total
    n_b = sum(b.numel() for b in bufs)
    self.flat = torch.zeros(n_g + n_b, device=optimizer.flat_grad.device, dtype=torch.float32)
    optimizer.flat_grad = self.flat[:n_g]
    self.stats = self.flat[n_g:]
    off = 0
    with torch.no_grad():
      for b in bufs:
        v = self.stats[off:off + b.numel()]
        v.copy_(b)
        b.data = v                               # the module's buffer now lives inside the bucket
        off += b.numel()
    self.n_grad = n_g

  def allreduce(self, group=None):
    """SUM all-reduce of gradients and BN statistics; the statistics are averaged here, the gradients by the optimizer step
    (grad_scale = 1 / world).  Returns 1 / world."""
    world = dist.get_world_size(group)
    dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group)
    return self.average(world)

  def average(self, world):
    """What follows the SUM all-reduce of `flat` over `world` replicas: the statistics are averaged in place.  Returns 1 / world,
    the grad_scale of the optimizer step that averages the gradients."""
    self.stats.mul_(1.0 / world)
    return 1.0 / world


# ---- torch.optim path (kept for callers that drive a plain torch optimizer, e.g. the reference's own loop)
def pack_gradients(params, out=None):
  """Flat fp32 bucket of the gradients of `params` (zeros where a parameter has no gradient).  `out` reuses a buffer."""
  flat = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])
  if out is not None:
    out.copy_(flat)
    return out
  return flat


def unpack_gradients(params, flat, world):
  """p.grad <- flat / world, parameter by parameter (creates the gradient where a rank had none)."""
  flat = flat / world
  off = 0
  for p in params:
    n = p.numel()
    g = flat[off:off + n].view_as(p)
    if p.grad is None:
      p.grad = g.clone()
    else:
      p.grad.copy_(g)
    off += n


def allreduce_gradients(params, group=None):
  """One flat-bucket SUM all-reduce then divide by world size (classic DP; 288 066 floats = 1.15 MB for k=3).
  A rank whose frame went to the validation set contributes zeros so the collective stays matched (adapt.py:385)."""
  world = dist.get_world_size(group)
  flat = pack_gradients(params)
  dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
  unpack_gradients(params, flat, world)
  return flat.numel()


def broadcast_state(stereo_net, feature_net, src=0, group=None):
  """Make every rank start from rank `src`'s parameters and buffers (one flat broadcast)."""
  ts = [t for net in (stereo_net, feature_net) for t in list(net.parameters()) + list(net.buffers()) if t.dtype.is_floating_point]
  flat = torch.cat([t.detach().reshape(-1) for t in ts])
  dist.broadcast(flat, src=src, group=group)
  off = 0
  with torch.no_grad():
    for t in ts:
      t.copy_(flat[off:off + t.numel()].view_as(t))
      off += t.numel()
