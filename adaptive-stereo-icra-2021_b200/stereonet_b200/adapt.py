"""Host-side mirror of one iteration of the reference's online-adaptation loop (adapt.py:304-396, NONSTOP/ER path):
train-mode forward with the cost volume, Monodepth photometric loss, backward, clip_grad_norm_ on the stereo_net
parameters only, Adam step.  The state machine / OVS / logging of adapt.py stay in the caller (out of scope)."""
import torch
import torch.nn as nn

from .losses import feature_contrast_mean, khamis_robust_loss, monodepth_single_loss


def make_optimizer(feature_net, stereo_net, lr=5e-5, capturable=False, fused=False):
  """adapt.py:208-210: two parameter groups, stereo_net first.  fused=True: optim.FusedAdamClip — clip_grad_norm_ on the stereo_net
  group + Adam as three launches of this library over one flat gradient bucket (always capturable; checkpoint-compatible with
  torch.optim.Adam).  Otherwise torch.optim.Adam as in the reference; capturable=True keeps its step counters on the device
  (needed by AdaptStepper(use_graph=True))."""
  if fused:
    from .optim import FusedAdamClip
    return FusedAdamClip(stereo_net, feature_net, lr=lr)
  # capturable: step counters live on the device; fused: one multi-tensor kernel per group instead of ~220 tiny
  # per-parameter bias-correction kernels (same update rule, torch.optim.Adam defaults)
  return torch.optim.Adam([{"params": stereo_net.parameters()}, {"params": feature_net.parameters()}], lr=lr,
                          capturable=capturable, fused=True if capturable else None)


class AdaptStepper:
  """use_graph=True captures the WHOLE update (forward, loss, backward, [gradient all-reduce,] clip, Adam) in one CUDA
  graph per input shape and replays it per frame: at batch 1 the step is ~700 launches of 3-100 us kernels, so eager
  execution is bound by host launch latency.  Requires an optimizer built with capturable=True.  The experience-replay term
  (`replay=(left, right, gt)`) is captured too (static replay buffers, fused Khamis loss)."""

  def __init__(self, feature_net, stereo_net, optimizer, height=None, width=None, clip_grad_norm=True, er_loss_weight=0.05,
               use_graph=False, batched_replay=False, two_streams=True):
    self.feature_net, self.stereo_net, self.optimizer = feature_net, stereo_net, optimizer
    self.clip, self.er_loss_weight = clip_grad_norm, er_loss_weight
    self.use_graph = use_graph              # (height / width are accepted for call-site compatibility with the reference's warper)
    # SURVEY.md section 8 row f3: run the replay sample through the model in the SAME batch-2 forward/backward as the stream
    # frame instead of a second full pass (adapt.py:339-349).  Off by default: train-mode BatchNorm then normalises with the
    # statistics of both samples together, which is NOT what the reference's two batch-1 passes compute.
    self.batched_replay = batched_replay
    self.two_streams, self._wstream, self._acc_stream, self._acc_nodes = two_streams, None, None, None
    self._forks = {}                        # the side streams of _fork, by name
    self._feature_fork = "side"             # which of them predict's right feature pass runs on
    self._graphs = {}
    self._wprep = None                      # fused.WeightPrepBatch: all derived weight images in one launch per step
    self.launches_per_step = None
    from .optim import FusedAdamClip
    self.fused_opt = isinstance(optimizer, FusedAdamClip)
    if self.fused_opt:
      optimizer.clip_norm = 1.0 if clip_grad_norm else None
    elif use_graph and not all(g.get("capturable", False) for g in optimizer.param_groups):
      raise RuntimeError("AdaptStepper(use_graph=True) needs make_optimizer(..., capturable=True) or fused=True")

  def predict(self, left, right):
    # The two feature passes (and, through autograd, their backward passes) are independent chains of small, latency-bound
    # kernels on a fraction of the SMs: in the two-stream schedule the right-image pass runs on a side stream next to the left one.
    # Both passes update the same BatchNorm buffers, left first in the reference: the fork applies the right pass's updates after.
    join = self._fork(self._feature_fork, left)
    fl = self.feature_net(left)                                                     # adapt.py:72
    fr = join(self.feature_net, right)
    return self.stereo_net(left, fl, fr, "l", output_cost_volume=True)             # adapt.py:73

  def _fork(self, side, like):
    """Forks the work that follows onto the side stream named `side` (created on first use): the stream waits here for what
    is already enqueued on the current one, and the returned `join(fn, *args)` runs fn on it, with its train-mode BatchNorm
    running-statistics updates deferred — into the enclosing fork's list, if there is one, else applied after the join on the
    current stream, behind whatever ran there since the fork.  In the single-stream schedule (two_streams=False, a CPU
    tensor, no grad) nothing forks and join(fn, *args) is fn(*args)."""
    if not (self.two_streams and like.is_cuda and torch.is_grad_enabled()):
      return lambda fn, *args: fn(*args)
    from .autograd import fused
    stream = self._forks.get(side)
    if stream is None:
      stream = self._forks[side] = torch.cuda.Stream(device=like.device)
    main = torch.cuda.current_stream(like.device)
    stream.wait_stream(main)

    def join(fn, *args):
      outer = fused.DEFER_BN
      pending = outer if outer is not None else []
      with torch.cuda.stream(stream):
        fused.DEFER_BN = pending
        try:
          out = fn(*args)
        finally:
          fused.DEFER_BN = outer
      main.wait_stream(stream)
      if not torch.cuda.is_current_stream_capturing():
        out.record_stream(main)
      if outer is None:
        fused.flush_deferred_bn(pending)
      return out
    return join

  def step(self, left, right, replay=None, sync_grads=None, dp_params=None, dp_group=None, dp_bucket=None):
    """One gradient update (adapt.py:313-314,328-337,381-394).  `replay` = (left, right, gt_disp) adds the
    experience-replay term (adapt.py:339-349).  Shared-model data parallelism:
      * `dp_bucket` (parallel.DPBucket, with an optim.FusedAdamClip optimizer): gradients are gathered into the flat bucket by one
        kernel, the bucket (gradients + BatchNorm running statistics) is SUM-all-reduced by ONE NCCL call, the statistics are
        averaged in place and the fused clip + Adam kernel applies 1 / world — no per-parameter pack / unpack;
      * `dp_params` (+ `dp_group`) with a torch optimizer: pack -> all-reduce -> unpack (round-1 path);
      * `sync_grads`: a callable run between backward and the update (eager path only).
    The update after backward has three parts, run back to back in the eager step: before the collective, the collective, after
    it.  With use_graph=True the step is graph(fwd + loss + bwd + before) -> eager collective -> graph(after)."""
    update = self._split_update(dp_params, dp_group, dp_bucket, sync_grads)
    if self.use_graph and sync_grads is None:
      key = (tuple(left.shape), str(left.device), None if dp_params is None else len(dp_params), dp_bucket is not None,
             None if replay is None else tuple(tuple(t.shape) for t in replay), self.batched_replay)
      return self._step_graph(key, left, right, replay, update)
    return self._step_eager(left, right, replay, update)

  def _split_update(self, dp_params, dp_group, dp_bucket, sync_grads):
    """The update after backward as (before, collective, after).  before() returns the tensor that collective(flat) reduces and
    after(flat) finishes from; without a collective (None) before() is the whole update.  The graph step captures before() and
    after() in one graph each and runs the collective eagerly between them: a captured NCCL collective hung a two-GPU run."""
    if dp_bucket is None and sync_grads is not None:
      return (lambda: None), (lambda flat: sync_grads()), (lambda flat: self._update())
    if dp_bucket is None and dp_params is None:
      return self._update, None, None
    import torch.distributed as dist
    from . import parallel
    world = dist.get_world_size(dp_group)
    collective = lambda flat: dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=dp_group)
    if dp_bucket is not None:
      def before():
        self.optimizer.pack()
        return dp_bucket.flat
      return before, collective, lambda flat: self._update(grad_scale=dp_bucket.average(world), packed=True)

    def after(flat):
      parallel.unpack_gradients(dp_params, flat, world)
      self._update()
    return (lambda: parallel.pack_gradients(dp_params)), collective, after

  def _step_eager(self, left, right, replay, update):
    before, collective, after = update
    out = self._fwd_bwd(left, right, replay)
    flat = before()
    if collective is not None:
      collective(flat)
      after(flat)
    return out

  def _fwd_bwd(self, left, right, replay):
    self.feature_net.train(); self.stereo_net.train()
    self._refresh_weights()
    loss, outputs = (self._loss_batched if replay is not None and self.batched_replay else self._loss)(left, right, replay)
    fcs = feature_contrast_mean(outputs["cost_volume_l/{}".format(self.stereo_net.input_scale + self.stereo_net.k)]).mean()
    self.optimizer.zero_grad()
    loss.backward()
    return loss.detach(), fcs, outputs

  def _loss(self, left, right, replay):
    s = self.stereo_net.input_scale
    from .autograd import fused
    if self.two_streams and left.is_cuda:
      if self._wstream is None:
        self._wstream = torch.cuda.Stream(device=left.device)
        # Gradient accumulation gets a stream of its own.  autograd runs a parameter's AccumulateGrad node on the stream that was
        # current when the node was created and makes THAT stream wait for the producer of every incoming gradient: with the
        # nodes on the main stream, each weight gradient finishing on the side streams would stall the main chain.  The nodes
        # are created here, under the accumulation stream, and kept alive (autograd holds them weakly).
        self._acc_stream = torch.cuda.Stream(device=left.device)
        with torch.cuda.stream(self._acc_stream):
          self._acc_nodes = [p.view_as(p).grad_fn.next_functions[0][0]
                             for net in (self.stereo_net, self.feature_net) for p in net.parameters() if p.requires_grad]
      fused.WGRAD_STREAM = self._wstream                                            # weight gradients next to the data path
      fused.wgrad_token((1,), left.device)                                          # (creates the token buffer outside any capture)
    try:
      # The replay pass (adapt.py:339-349) is independent of the stream pass until the two losses are added: it runs on its own
      # stream (its feature passes side by side on a second one) with ALL its BatchNorm running-statistics updates applied after
      # the stream pass's, the reference's order.  The fork comes before the stream pass is enqueued: forking where the replay
      # pass starts would make it wait for the whole stream pass.
      join_replay = self._fork("replay", left) if replay is not None else None
      outputs = self.predict(left, right)
      loss = monodepth_single_loss(left, right, outputs, s)                        # adapt.py:328-337 (snb_photo_loss)
      if replay is not None:
        loss = loss + self.er_loss_weight * join_replay(self._replay_loss, replay)
    finally:
      fused.WGRAD_STREAM = None
    return loss, outputs

  def _replay_loss(self, replay):
    self._feature_fork = "replay side"      # the replay pass runs on a side stream already: its right feature pass needs another
    try:
      out = self.predict(replay[0], replay[1])                                      # adapt.py:339-349: a second full pass
    finally:
      self._feature_fork = "side"
    return khamis_robust_loss(out["pred_disp_l/{}".format(self.stereo_net.input_scale)], replay[2])

  def _refresh_weights(self):
    from .autograd import fused
    if fused.CONV_BACKEND == "ffma" or not torch.is_grad_enabled():
      return
    if self._wprep is None or not self._wprep.valid():
      self._wprep = fused.WeightPrepBatch([self.feature_net, self.stereo_net])
    self._wprep.refresh()

  def _loss_batched(self, left, right, replay):
    """Row f3: one batch-(n+m) pass for the n stream frames and the m replay samples; Monodepth loss on the first n
    predictions (the outputs returned), Khamis robust loss on the rest (snb_khamis_loss), 1 : er_loss_weight as adapt.py:383-388."""
    s = self.stereo_net.input_scale
    n = left.shape[0]
    outputs = self.predict(torch.cat([left, replay[0]], 0), torch.cat([right, replay[1]], 0))
    key = "pred_disp_l/{}".format(s)
    head = {k: v[:n] for k, v in outputs.items()}
    loss = monodepth_single_loss(left, right, head, s)
    loss = loss + self.er_loss_weight * khamis_robust_loss(outputs[key][n:], replay[2])
    return loss, head

  def _update(self, grad_scale=1.0, packed=False):
    if self.fused_opt:
      self.optimizer.step(grad_scale=grad_scale, packed=packed)                   # clip (adapt.py:391-392) + Adam (:393), 3 launches
      return
    if self.clip:
      nn.utils.clip_grad_norm_(self.stereo_net.parameters(), 1.0)                 # adapt.py:391-392
    self.optimizer.step()

  # ---------------------------------------------------------------------------------------------- CUDA-graph path
  def _state_tensors(self):
    ts = [p for net in (self.stereo_net, self.feature_net) for p in net.parameters()]
    ts += [b for net in (self.stereo_net, self.feature_net) for b in net.buffers()]
    if self.fused_opt:
      ts += [self.optimizer.exp_avg, self.optimizer.exp_avg_sq, self.optimizer.step_t]
    else:
      for st in self.optimizer.state.values():
        ts += [v for v in st.values() if isinstance(v, torch.Tensor)]
    return ts

  def _capture(self, left, right, replay, update):
    from . import ops
    from .autograd import fused
    before, collective, after = update
    self.feature_net.train(); self.stereo_net.train()
    dev = left.device
    sl, sr = left.clone(), right.clone()
    srep = None if replay is None else tuple(t.clone() for t in replay)        # static replay buffers (left, right, gt)
    fresh = (not self.fused_opt) and len(self.optimizer.state) == 0
    snap = [(t, t.detach().clone()) for t in self._state_tensors()]
    cur = torch.cuda.current_stream(dev)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(cur)
    with torch.cuda.stream(side):
      # One eager warm-up step allocates the lazily-created state (Adam moments and step counters, derived-weight
      # caches, allocator pools); model and optimizer state are restored afterwards so that capturing does not advance
      # the adaptation.
      self._step_eager(sl, sr, srep, update)
      self.optimizer.zero_grad(set_to_none=True)
      with torch.no_grad():
        for t, saved in snap:                 # in place: the graphs will hold these addresses
          t.copy_(saved)
        if fresh:
          for st in self.optimizer.state.values():
            for v in st.values():
              if isinstance(v, torch.Tensor):
                v.zero_()
    cur.wait_stream(side)
    fused.bump_epoch()
    n0 = ops.LAUNCHES
    g1 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g1):
      out = self._fwd_bwd(sl, sr, srep)
      flat = before()
    g2 = None
    if collective is not None:
      g2 = torch.cuda.CUDAGraph()
      with torch.cuda.graph(g2, pool=g1.pool()):
        after(flat)
    self.launches_per_step = ops.LAUNCHES - n0          # library kernels inside one replay
    return dict(g1=g1, g2=g2, flat=flat, left=sl, right=sr, replay=srep, out=out)

  def _step_graph(self, key, left, right, replay, update):
    from .autograd import fused
    e = self._graphs.get(key)
    if e is None:
      e = self._graphs[key] = self._capture(left, right, replay, update)
    e["left"].copy_(left, non_blocking=True)
    e["right"].copy_(right, non_blocking=True)
    if replay is not None:
      for dst, src in zip(e["replay"], replay):
        dst.copy_(src, non_blocking=True)
    e["g1"].replay()
    if e["g2"] is not None:
      update[1](e["flat"])                  # the collective, eager between the two graphs
      e["g2"].replay()
    fused.bump_epoch()                      # the replay rewrote the parameters behind torch's version counters
    return e["out"]
