"""Inference engine: CUDA-graph replay of the whole forward (feature_net x2 + stereo_net) with static device buffers
and pinned-host staging.  At batch 1 every kernel is 3-100 us, so per-launch host latency would otherwise dominate
(SURVEY.md §7 step 7).  One engine per (process, GPU).  A captured graph bakes in the derived tensors (tensor-core weight
images, folded BatchNorm) of the moment of capture, so every entry remembers the state epoch it was captured at
(autograd.fused.state_epoch(): advanced by optimizer steps, graph-replayed adaptation steps and train-mode BatchNorm updates) and
is re-captured on the next call after a change — an adaptation loop that alternates AdaptStepper.step and engine(left, right)
(adapt.py's validate / evaluate pattern) never sees stale weights.  `invalidate()` is only needed after parameters were
re-assigned by other means (e.g. raw `.data` writes).

precision="fp16" selects the opt-in reduced-precision forward for throughput inference: the 32->32 3x3 and 3x3x3 walk-kernel
layers run one fp16 product per tap (snb_conv_c32_ws_f16) instead of the fp32-grade split.  Its disparities are reported separately
from the fp32 parity contract (DESIGN.md section 4.2f16 lists the measured errors); it is bit-identical to snb_stereonet_forward_f16.
Eval mode only: train-mode BatchNorm statistics stay on the fp32-grade path."""
import torch

from . import ops
from .autograd import fused


class StereoEngine:
  def __init__(self, feature_net, stereo_net, output_cost_volume=False, use_graph=True, precision="fp32"):
    if precision not in ("fp32", "fp16"):
      raise ValueError(f"precision must be 'fp32' or 'fp16', got {precision!r}")
    self.precision = precision
    self.feature_net, self.stereo_net = feature_net, stereo_net
    self.output_cost_volume = output_cost_volume
    self.use_graph = use_graph
    self._graphs = {}
    self._pipes = {}

  def invalidate(self):
    self.synchronize()
    self._graphs.clear()

  def _forward(self, pair):
    """pair = [left; right] stacked on the batch dim.  In eval mode both images go through the feature extractor as
    one batch (no op mixes samples when BN uses running statistics, SURVEY.md §8e: bit-identical to two calls, half
    the launches); in train mode the two calls stay separate because BN batch statistics are per call
    (adapt.py:72: feature_net(left), feature_net(right))."""
    if self.precision == "fp32":
      return self._forward_pair(pair)
    if self.feature_net.training or self.stereo_net.training:
      raise RuntimeError("stereonet_b200: StereoEngine(precision='fp16') runs eval-mode modules only")
    old = fused.F16_LAYERS
    fused.F16_LAYERS = fused.F16_SHIPPED
    try:
      return self._forward_pair(pair)
    finally:
      fused.F16_LAYERS = old

  def _forward_pair(self, pair):
    B = pair.shape[0] // 2
    left, right = pair[:B], pair[B:]
    if self.feature_net.training:
      fl, fr = self.feature_net(left), self.feature_net(right)
    else:
      feats = self.feature_net(pair)
      fl, fr = feats[:B], feats[B:]
    return self.stereo_net(left, fl, fr, "l", output_cost_volume=self.output_cost_volume)

  def _entry(self, shape, device, slot=0):
    """The captured forward for this input shape.  `slot` selects one of several independent captures (own static input and
    output buffers): the streaming API alternates between two so that the copies of one frame never touch the buffers the
    forward of its neighbour is using."""
    key = (tuple(shape), str(device), self.feature_net.training, slot, self.precision)
    e = self._graphs.get(key)
    if e is not None:
      if e["epoch"] == fused.state_epoch():
        return e
      self.synchronize()                       # weights / BN statistics changed since the capture: drain the copy streams that
      del self._graphs[key]                    # still use the old static buffers, then re-capture on this call
    pair = torch.zeros((2 * shape[0],) + tuple(shape[1:]), device=device, dtype=torch.float32)
    left, right = pair[:shape[0]], pair[shape[0]:]
    with torch.no_grad():
      side = torch.cuda.Stream(device=device)
      side.wait_stream(torch.cuda.current_stream(device))
      with torch.cuda.stream(side):
        for _ in range(2):                       # warm the derived-weight caches / allocator outside the capture
          self._forward(pair)
      torch.cuda.current_stream(device).wait_stream(side)
      n0 = ops.LAUNCHES
      if self.use_graph:
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
          out = self._forward(pair)
      else:
        graph, out = None, self._forward(pair)
      launches = ops.LAUNCHES - n0
    e = dict(pair=pair, left=left, right=right, graph=graph, out=out, launches=launches, epoch=fused.state_epoch())
    self._graphs[key] = e
    return e

  @torch.no_grad()
  def run_static(self, shape, device, slot=0):
    """Replay on whatever currently sits in the static input buffers. Returns (outputs dict, launches per step)."""
    e = self._entry(shape, device, slot)
    if e["graph"] is not None:
      e["graph"].replay()
      if self.feature_net.training:            # the replay updated BN running statistics behind Python's back: whatever was folded
        fused.bump_bn_epoch()                  # from them (eval-mode graphs, bn_fold caches) is stale; this graph itself is not
        e["epoch"] = fused.state_epoch()
    else:
      e["out"] = self._forward(e["pair"])
    return e["out"], e["launches"]

  @torch.no_grad()
  def __call__(self, left, right):
    """Device tensors in, dict of device tensors out (valid until the next call)."""
    e = self._entry(left.shape, left.device)
    e["left"].copy_(left, non_blocking=True)
    e["right"].copy_(right, non_blocking=True)
    return self.run_static(left.shape, left.device)[0]

  @torch.no_grad()
  def infer_host(self, left_host, right_host, out_host, key=None):
    """Host (pinned) images in, host (pinned) full-resolution disparity out; everything stream-ordered."""
    dev = next(self.stereo_net.parameters()).device
    e = self._entry(left_host.shape, dev)
    e["left"].copy_(left_host, non_blocking=True)
    e["right"].copy_(right_host, non_blocking=True)
    out, _ = self.run_static(left_host.shape, dev)
    if key is None:
      key = "pred_disp_l/{}".format(self.stereo_net.input_scale)
    out_host.copy_(out[key], non_blocking=True)
    return out_host

  # ------------------------------------------------------------------------------------------------ streaming API
  def _pipe(self, shape, dev):
    p = self._pipes.get((tuple(shape), str(dev)))
    if p is None:
      key = "pred_disp_l/{}".format(self.stereo_net.input_scale)
      p = dict(i=0, key=key, s_in=torch.cuda.Stream(device=dev), s_out=torch.cuda.Stream(device=dev),
               ev_in=[torch.cuda.Event() for _ in range(2)], ev_free=[torch.cuda.Event() for _ in range(2)],
               ev_out=[torch.cuda.Event() for _ in range(2)], ev_outfree=[torch.cuda.Event() for _ in range(2)])
      cur = torch.cuda.current_stream(dev)
      for k in range(2):
        p["ev_free"][k].record(cur); p["ev_outfree"][k].record(cur)
      self._pipes[(tuple(shape), str(dev))] = p
    return p

  @torch.no_grad()
  def infer_host_async(self, left_host, right_host, out_host):
    """Streaming variant of infer_host for frame sequences: the H2D copy of frame i+1 (copy-in stream), the forward of
    frame i (current stream, CUDA graph) and the D2H copy of frame i-1 (copy-out stream) overlap.  Two captures of the forward
    alternate (slots 0 / 1): the host images land directly in a capture's static input and the disparity leaves directly from its
    static output, so no device-to-device staging copy sits on the compute stream.  `out_host` is valid after `synchronize()`;
    the caller must not overwrite `left_host`/`right_host` of a frame before the next-but-one call returns (or before
    `synchronize()`)."""
    dev = next(self.stereo_net.parameters()).device
    p = self._pipe(left_host.shape, dev)
    k = p["i"] & 1
    e = self._entry(left_host.shape, dev, slot=k)
    cur = torch.cuda.current_stream(dev)
    p["s_in"].wait_event(p["ev_free"][k])                 # capture k consumed its input two frames ago
    with torch.cuda.stream(p["s_in"]):
      e["left"].copy_(left_host, non_blocking=True)
      e["right"].copy_(right_host, non_blocking=True)
      p["ev_in"][k].record(p["s_in"])
    cur.wait_event(p["ev_in"][k])
    cur.wait_event(p["ev_outfree"][k])                    # the D2H of two frames ago has drained capture k's output
    out, _ = self.run_static(left_host.shape, dev, slot=k)
    p["ev_free"][k].record(cur)
    p["ev_out"][k].record(cur)
    p["s_out"].wait_event(p["ev_out"][k])
    with torch.cuda.stream(p["s_out"]):
      out_host.copy_(out[p["key"]], non_blocking=True)
      p["ev_outfree"][k].record(p["s_out"])
    p["i"] += 1
    return out_host

  def synchronize(self):
    """Block the host until every copy issued by infer_host_async has completed: afterwards the `out_host` buffers are valid
    and the pinned input buffers may be overwritten.  (The current stream is also made to wait for the copy streams.)"""
    for (_, devs), p in self._pipes.items():
      dev = torch.device(devs)
      cur = torch.cuda.current_stream(dev)
      cur.wait_stream(p["s_in"]); cur.wait_stream(p["s_out"])
      p["s_in"].synchronize(); p["s_out"].synchronize()
