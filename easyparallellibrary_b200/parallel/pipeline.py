"""Pipeline executor: interprets a stage program (``parallel/schedule.py``) on one rank.

Reference mechanics (``graph_editor.py:397-421`` micro-batch clones + ``scheduler.py`` control
edges + implicit TF ``_Send/_Recv``) become: a loop over instructions, micro-batch activations kept
in a dict, and explicit NCCL point-to-point transfers.  Transfers in the two directions use two
independent process groups (hence independent NCCL streams), receives are posted ``prefetch``
slots early into per-micro-batch buffers (double buffering) and sends are asynchronous, so under
1F1B a transfer overlaps the neighbouring micro-batch's compute instead of sitting on the
critical path.
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional, Tuple

import torch
import torch.distributed as dist

from easyparallellibrary_b200.ir.graph import Graph
from easyparallellibrary_b200.ir.phase import ModelPhase, phase_scope
from easyparallellibrary_b200.parallel import schedule as S

_META_LEN = 10
_DTYPES = [torch.float32, torch.bfloat16, torch.float16, torch.int64, torch.int32]


class _TorchP2P(object):
  """CPU / gloo transport: torch.distributed point-to-point on two process groups (one per direction)."""

  def __init__(self, prev: Optional[int], nxt: Optional[int]):
    self.prev, self.next = prev, nxt
    self.pg_fwd = dist.new_group()
    self.pg_bwd = dist.new_group()

  def send_fwd(self, t):
    return dist.isend(t, self.next, group=self.pg_fwd)

  def recv_fwd(self, t):
    return dist.irecv(t, self.prev, group=self.pg_fwd)

  def send_bwd(self, t):
    return dist.isend(t, self.prev, group=self.pg_bwd)

  def recv_bwd(self, t):
    return dist.irecv(t, self.next, group=self.pg_bwd)

  def send_meta(self, meta):
    dist.send(meta, self.next, group=self.pg_fwd)

  def recv_meta(self, meta):
    dist.recv(meta, self.prev, group=self.pg_fwd)


class _EventHandle(object):
  def __init__(self, ev):
    self.ev = ev

  def wait(self):
    torch.cuda.current_stream().wait_event(self.ev)


class _NativeP2P(object):
  """GPU transport: the in-tree NCCL communicator (``csrc/communicator.cpp``), one 2-rank communicator — hence one
  dedicated side stream — per neighbour and direction.  A receive posted early never blocks the host or an unrelated
  transfer, and every transfer hands back its own event, so a compute instruction waits for exactly its tensor."""

  def __init__(self, me: int, prev: Optional[int], nxt: Optional[int], device):
    from easyparallellibrary_b200.communicators.native import NativeBackend
    self.fwd_in = self.bwd_out = self.fwd_out = self.bwd_in = None
    if prev is not None:          # lower pair first on every rank: creation order is deadlock free
      self.fwd_in = NativeBackend([prev, me], device)
      self.bwd_out = NativeBackend([prev, me], device)
    if nxt is not None:
      self.fwd_out = NativeBackend([me, nxt], device)
      self.bwd_in = NativeBackend([me, nxt], device)
    self._keep = []
    # NCCL connects a send/recv pair lazily, on the HOST, inside the first call, and that call blocks until the peer
    # makes the matching one.  Under 1F1B the first RECV_B of a stage is posted long before its neighbour reaches the
    # matching SEND_B, so a lazy connect deadlocks the schedule (seen on B200: stage 0 inside ncclRecv, stage 1 waiting
    # for stage 0's next activation).  Connect every channel here, in chain order, with one tiny transfer each.
    probe = torch.zeros(8, dtype=torch.float32, device=device)
    if prev is not None:
      self.fwd_in.recv(probe, 0)
      self.bwd_out.send(probe, 0)
    if nxt is not None:
      self.fwd_out.send(probe, 1)
      self.bwd_in.recv(probe, 1)
    for be in (self.fwd_in, self.bwd_out, self.fwd_out, self.bwd_in):
      if be is not None:
        be.stream.synchronize()

  @staticmethod
  def _done(be):
    ev = torch.cuda.Event()
    ev.record(be.stream)
    return _EventHandle(ev)

  def send_fwd(self, t):
    self._keep.append(t)
    self.fwd_out.send(t, 1)
    return self._done(self.fwd_out)

  def recv_fwd(self, t):
    self.fwd_in.recv(t, 0)
    return self._done(self.fwd_in)

  def send_bwd(self, t):
    self._keep.append(t)
    self.bwd_out.send(t, 0)
    return self._done(self.bwd_out)

  def recv_bwd(self, t):
    self.bwd_in.recv(t, 1)
    return self._done(self.bwd_in)

  def send_meta(self, meta):
    self.send_fwd(meta).wait()
    torch.cuda.current_stream().synchronize()

  def recv_meta(self, meta):
    self.recv_fwd(meta).wait()
    torch.cuda.current_stream().synchronize()

  def flush(self):
    self._keep.clear()


class _StageFn(torch.nn.Module):
  """What one F instruction runs — the stage's layers and, on the last stage, the loss scaled for backward — as a module
  of its own, so ``torch.cuda.make_graphed_callables`` can capture it.  Several instances share the same inner module
  (one per micro-batch that may be in flight: the captured graphs own the saved activations)."""

  def __init__(self, module, loss_fn, factor: float, device=None):
    super().__init__()
    self.module, self.loss_fn, self.factor = module, loss_fn, float(factor)
    # loss scale x 1/M as a DEVICE scalar: a dynamic loss scale changes between steps, and a Python float would be baked into
    # the captured graph (set_factor refreshes it before a replay)
    self.factor_t = torch.full((), float(factor), dtype=torch.float32, device=device) if loss_fn is not None else None

  def set_factor(self, factor: float) -> None:
    if self.factor_t is not None and float(factor) != self.factor:
      self.factor = float(factor)
      self.factor_t.fill_(self.factor)

  def forward(self, x, *labels):
    y = self.module(x)
    if self.loss_fn is not None:
      y = self.loss_fn(y, *labels)
      return y * self.factor_t.to(y.dtype)
    return y


class _GraphedStage(object):
  """Forward and backward of one pipeline stage as two CUDA graphs with static input / output buffers.

  Unlike ``torch.cuda.make_graphed_callables`` nothing goes through autograd at replay time: the backward graph ends with the
  accumulation of every parameter gradient into the trainer's flat gradient buckets (weight-gradient GEMMs write there
  directly, the other gradients are added by captured ``add_`` kernels), so an F or B instruction costs the host a few small
  copies and one graph launch — no per-parameter AccumulateGrad nodes, hooks or Python per micro-batch.

  Every stage keeps static copies of every tensor of the micro-batch, and the capture runs with ``current_micro_batch``
  pointing at them: a layer that reads the micro-batch (BERT's attention reads its key lengths from the input mask) bakes
  the static copy's address into the graph, and each replay first copies the micro-batch being executed into it."""

  def __init__(self, fn, x, mb, last, pool):
    """Phase 1: capture the forward graph.  ALL forward graphs of a stage are captured before any backward graph, so that a
    backward's temporaries can never be placed (by the shared pool) where another instance's saved activations live.
    ``mb``: static copies of the micro-batch; on stage 0 ``x`` is ``mb[0]``."""
    self.fn = fn
    self.x = x                                       # static input (requires_grad for stages > 0)
    self.mb = tuple(mb)
    self.labels = self.mb[1:] if last else ()
    self.pool = pool
    self.g_fwd, self.g_bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    Graph.get().current_micro_batch = self.mb
    with torch.cuda.graph(self.g_fwd, pool=pool):
      self.y = fn(self.x, *self.labels)              # keeps the autograd graph (and with it the saved activations) alive
    self.y_out = self.y.detach()
    self.gx = None

  def capture_backward(self, grad_views, ones_grad: bool) -> None:
    params = [p for p in self.fn.parameters() if p.requires_grad]
    inputs = ([self.x] if self.x.requires_grad else []) + params
    self.gy = torch.ones_like(self.y) if ones_grad else torch.zeros_like(self.y)
    Graph.get().current_micro_batch = self.mb
    with torch.cuda.graph(self.g_bwd, pool=self.pool):
      grads = torch.autograd.grad(outputs=(self.y,), inputs=tuple(inputs), grad_outputs=(self.gy,), allow_unused=True, retain_graph=True)
      k = 0
      if self.x.requires_grad:
        self.gx = grads[0]
        k = 1
      for p, g in zip(params, grads[k:]):
        if g is not None:
          grad_views[id(p)].add_(g.view_as(grad_views[id(p)]))

  def forward(self, x, mb):
    for s, t in zip(self.mb, mb):
      if isinstance(s, torch.Tensor) and s.data_ptr() != t.data_ptr():
        s.copy_(t)
    if self.x is not self.mb[0] and x.data_ptr() != self.x.data_ptr():
      self.x.detach().copy_(x)
    self.g_fwd.replay()
    return self.y_out

  def backward(self, gy=None):
    if gy is not None:
      self.gy.copy_(gy)
    self.g_bwd.replay()
    return self.gx


class PipelineExecutor(object):
  def __init__(self, trainer):
    self.tr = trainer
    plan = trainer.plan
    if len(plan.local_stages) != 1:
      raise RuntimeError("pipeline execution expects exactly one stage per rank (got %s)" % plan.local_stages)
    self.stage = plan.local_stages[0]
    self.num_stages = plan.num_stages
    self.M = plan.num_micro_batch
    self.first = self.stage == 0
    self.last = self.stage == self.num_stages - 1
    self.prev = plan.prev_rank(self.stage)
    self.next = plan.next_rank(self.stage)
    self.module = trainer.stage_modules[self.stage]
    policy = trainer.config.pipeline.strategy
    self.program = S.build_stage_program(policy, self.stage, self.num_stages, self.M, prefetch=1)
    try:      # the native runtime generates the same program; use it when built (cross-checked in the tests)
      from easyparallellibrary_b200.runtime import native
      if native.available():
        self.program = [S.Instr(op, mb) for op, mb in native.schedule_stage(policy, self.stage, self.num_stages, self.M, 1)]
    except Exception:  # pragma: no cover
      pass
    # activations and activation-gradients travel on independent streams / communicators
    if trainer.device.type == "cuda":
      self.p2p = _NativeP2P(plan.rank, self.prev, self.next, trainer.device)
    else:
      self.p2p = _TorchP2P(self.prev, self.next)
    # one group per model replica (all stages of that replica) for cross-stage reductions
    self.replica_group = None
    for r in range(plan.num_replicas):
      ranks = [plan.stage_ranks[s][r][0] for s in range(self.num_stages)]
      g = dist.new_group(ranks)
      if plan.rank in ranks:
        self.replica_group = g
        self.replica_ranks = ranks
    self._shape_fwd: Optional[Tuple[torch.Size, torch.dtype]] = None
    self.device = trainer.device
    # CUDA graphs of the stage's forward and backward (one pair per micro-batch that can be in flight): a micro-batch of a
    # few thousand tokens is ~2400 launches of ~30 us kernels, i.e. host-launch bound by 3x when issued from Python
    # (profiles/r1_bench_pp2_xl_v1.json); replayed from graphs the stage is GPU bound.
    import os
    self.use_graphs = (trainer.device.type == "cuda" and os.environ.get("EPL_PIPE_GRAPH", "1") != "0" and not trainer.zero3
                       and not trainer.config.gradient_checkpoint.type and not trainer.config.offload.level)
    self.graphed: List[Any] = []
    self._bufs_f: Dict[int, torch.Tensor] = {}
    self._bufs_b: Dict[int, torch.Tensor] = {}

  def _in_flight(self) -> int:
    policy = (self.tr.config.pipeline.strategy or "").lower()
    if "forward" in policy:                      # GPipe order: every micro-batch is in flight before the first backward
      return self.M
    return max(1, min(self.M, self.num_stages - self.stage + (1 if "optimizer" in policy else 0)))

  def _build_graphs(self, micro: List[Tuple[Any, ...]]) -> None:
    """Capture forward/backward CUDA graphs of this stage, one pair per micro-batch that can be in flight (``_GraphedStage``:
    static input/output buffers, every parameter gradient accumulated into the flat buckets inside the backward graph).
    Any failure leaves the executor on the eager path."""
    tr = self.tr
    k = self._in_flight()
    if k > 4:
      self.use_graphs = False
      return
    mb = micro[0]
    mean = tr._mean
    factor = tr.scaler.loss_scale * ((1.0 / self.M) if (mean and self.M > 1) else 1.0)
    loss_fn = tr.loss_fn if self.last else None
    if self.last and loss_fn is None:
      self.use_graphs = False
      return
    fn = _StageFn(self.module, loss_fn, factor if self.last else 1.0, device=self.device)
    self.stage_fn = fn
    self.stage_factor = fn.factor
    if self.last and not all(isinstance(t, torch.Tensor) for t in mb[1:]):
      self.use_graphs = False
      return
    labels = tuple(mb[1:]) if self.last else ()
    for p in self.module.parameters():           # captured weight-gradient GEMMs must accumulate (the buckets are zeroed per step)
      if hasattr(p, "epl_sink_fresh"):
        p.epl_sink_fresh = False
    tr._first_micro_batch, tr._last_micro_batch = False, False
    Graph.get().current_micro_batch = mb
    grad_views = {pid: v[0] for pid, v in tr._grad_view.items()}

    def make_x():
      x = torch.zeros(self._shape_fwd[0], dtype=self._shape_fwd[1], device=self.device)
      return x.requires_grad_() if x.is_floating_point() else x

    def make_stage():
      static_mb = tuple(t.clone() if isinstance(t, torch.Tensor) else t for t in mb)
      return _GraphedStage(fn, static_mb[0] if self.first else make_x(), static_mb, self.last, pool)
    try:
      # one eager pass on a side stream first (torch's capture recipe), then k (forward, backward) graph pairs in one pool
      side = torch.cuda.Stream(device=self.device)
      side.wait_stream(torch.cuda.current_stream())
      with torch.cuda.stream(side):
        xw = mb[0].clone() if self.first else make_x()
        yw = fn(xw, *labels)
        ins_w = ([xw] if xw.requires_grad else []) + [p for p in fn.parameters() if p.requires_grad]
        torch.autograd.grad((yw,), tuple(ins_w), (torch.ones_like(yw),), allow_unused=True)
        del xw, yw, ins_w
      torch.cuda.current_stream().wait_stream(side)
      torch.cuda.synchronize(self.device)
      pool = torch.cuda.graph_pool_handle()
      self.graphed = [make_stage() for _ in range(k)]
      for st in reversed(self.graphed):
        st.capture_backward(grad_views, ones_grad=self.last)
    except Exception as e:      # pragma: no cover - depends on the CUDA runtime
      from easyparallellibrary_b200.utils.logging import get_logger
      get_logger().warning("pipeline stage %d: CUDA graph capture failed (%s); running the stage eagerly", self.stage, e)
      self.graphed, self.use_graphs = [], False
      torch.cuda.synchronize(self.device)
    Graph.get().pop_collections()
    for flat in tr.flats.values():               # the warm-up / capture passes ran real weight-gradient GEMMs into the buckets
      flat.zero_grad()
    torch.cuda.synchronize(self.device)

  # ------------------------------------------------------------------ metadata handshake (first step only)
  def _send_meta(self, t: torch.Tensor) -> None:
    vals = [t.dim(), _DTYPES.index(t.dtype)] + list(t.shape)
    meta = torch.tensor(vals + [0] * (_META_LEN - len(vals)), dtype=torch.int64, device=self.device)
    self.p2p.send_meta(meta)

  def _recv_meta(self) -> Tuple[torch.Size, torch.dtype]:
    meta = torch.zeros(_META_LEN, dtype=torch.int64, device=self.device)
    self.p2p.recv_meta(meta)
    meta = meta.cpu().tolist()
    return torch.Size(meta[2:2 + meta[0]]), _DTYPES[meta[1]]

  # ------------------------------------------------------------------ kernel warm-up (first step, GPU only)
  def _warmup(self, micro: List[Tuple[Any, ...]]) -> None:
    """Run this stage's forward + backward once, with no pipeline transfer in flight, before the first schedule.

    CUDA loads kernels lazily, and the first launch of a kernel cannot complete while another kernel of the process is
    spinning on the device.  A posted NCCL receive spins until its peer sends, so under 1F1B the first step can deadlock:
    stage 0 sits in the lazy load of its first backward kernel behind its own posted RECV_B, stage 1 sits in the lazy load
    of its first forward kernel behind its posted RECV_F, and neither reaches the send the other waits for (observed on
    B200).  After this pass every kernel of F and B is resident, so launches never block again.  Model buffers
    (e.g. BatchNorm statistics), the RNG state and the gradient buckets are restored, so training is unaffected.
    """
    tr = self.tr
    mb = micro[0]
    saved = [b.detach().clone() for b in self.module.buffers()]
    cpu_rng, dev_rng = torch.get_rng_state(), torch.cuda.get_rng_state(self.device)
    tr._first_micro_batch, tr._last_micro_batch = True, False     # no bucket reduction is launched from the grad hooks
    if self.first:
      x = mb[0]
    else:
      self._shape_fwd = self._recv_meta()
      x = torch.zeros(self._shape_fwd[0], dtype=self._shape_fwd[1], device=self.device)
      if x.is_floating_point():
        x.requires_grad_()
    Graph.get().current_micro_batch = mb
    with phase_scope(ModelPhase.FORWARD):
      y = self.module(x)
      if self.last and tr.loss_fn is not None:
        y = tr.loss_fn(y, *mb[1:])
    if not self.last:
      self._send_meta(y)
      self._meta_sent = True
    with phase_scope(ModelPhase.BACKWARD):
      if self.last:
        (y if y.dim() == 0 else y.float().sum()).backward()
      else:
        torch.autograd.backward(y, grad_tensors=torch.zeros_like(y))
    Graph.get().pop_collections()
    for z in getattr(tr, "zero3", {}).values():
      z.finish_backward()
      z.zero_grad()
    for flat in tr.flats.values():
      flat.zero_grad()
    with torch.no_grad():
      for b, v in zip(self.module.buffers(), saved):
        b.copy_(v)
    torch.set_rng_state(cpu_rng)
    torch.cuda.set_rng_state(dev_rng, self.device)
    torch.cuda.synchronize(self.device)
    dist.barrier(group=self.replica_group)      # nobody starts the schedule before every stage has loaded its kernels

  # ------------------------------------------------------------------ one training step
  def run(self, micro: List[Tuple[Any, ...]], mean: bool):
    tr, graph = self.tr, Graph.get()
    if self.device.type == "cuda" and not getattr(self, "_warm", False):
      self._warmup(micro)
      self._warm = True
      if self.use_graphs:
        self._build_graphs(micro)
        dist.barrier(group=self.replica_group)
    use_graphs = bool(self.graphed) and torch.is_grad_enabled()
    if use_graphs:
      for p in self.module.parameters():
        if hasattr(p, "epl_sink_fresh"):
          p.epl_sink_fresh = False
      if self.last:                               # the (dynamic) loss scale of THIS step, read by the captured graph from device memory
        self.stage_fn.set_factor(tr.scaler.loss_scale * ((1.0 / self.M) if (mean and self.M > 1) else 1.0))
        self.stage_factor = self.stage_fn.factor
    inputs: Dict[int, torch.Tensor] = {}
    outputs: Dict[int, torch.Tensor] = {}
    recv_f: Dict[int, Tuple[torch.Tensor, Any]] = {}
    recv_b: Dict[int, Tuple[torch.Tensor, Any]] = {}
    grads_in: Dict[int, torch.Tensor] = {}          # graph mode: the static input-gradient buffer of each backward
    sends: List[Any] = []
    losses: List[torch.Tensor] = []
    collected = []
    tr._first_micro_batch, tr._last_micro_batch = True, False
    n_back = 0
    debug = bool(int(__import__("os").environ.get("EPL_PIPE_DEBUG", "0")))
    timing = bool(int(__import__("os").environ.get("EPL_PIPE_TIMING", "0")))
    import time as _time
    host_t: Dict[str, float] = {}
    t_prev = _time.perf_counter()
    for ins in self.program:
      if timing:                                   # host time spent issuing each instruction kind (no device sync)
        now = _time.perf_counter()
        if getattr(self, "_last_op", None) is not None:
          host_t[self._last_op] = host_t.get(self._last_op, 0.0) + (now - t_prev)
        t_prev, self._last_op = now, ins.op
      if debug:
        print("[pipe rank %d stage %d] %r" % (tr.plan.rank, self.stage, ins), flush=True)
      if ins.op == S.RECV_F:
        if self._shape_fwd is None:
          self._shape_fwd = self._recv_meta()
        buf = self._bufs_f.get(ins.mb)           # per-micro-batch receive buffers are allocated once and reused every step
        if buf is None or buf.shape != self._shape_fwd[0]:
          buf = self._bufs_f[ins.mb] = torch.empty(self._shape_fwd[0], dtype=self._shape_fwd[1], device=self.device)
        else:
          buf = self._bufs_f[ins.mb] = buf.detach()
          buf.grad = None
        recv_f[ins.mb] = (buf, self.p2p.recv_fwd(buf))
      elif ins.op == S.RECV_B:
        out = outputs[ins.mb]
        buf = self._bufs_b.get(ins.mb)
        if buf is None or buf.shape != out.shape or buf.dtype != out.dtype:
          buf = self._bufs_b[ins.mb] = torch.empty_like(out)
        recv_b[ins.mb] = (buf, self.p2p.recv_bwd(buf))
      elif ins.op == S.F:
        mb = micro[ins.mb]
        graph.current_micro_batch = mb
        if self.first:
          x = mb[0]
        else:
          x, req = recv_f.pop(ins.mb)
          req.wait()
          if x.is_floating_point():
            x.requires_grad_()
        with phase_scope(ModelPhase.FORWARD):
          if use_graphs:
            st = self.graphed[ins.mb % len(self.graphed)]
            y = st.forward(x, mb)
            if self.last:
              losses.append(y / self.stage_factor if self.stage_factor != 1.0 else y.clone())
          else:
            y = self.module(x)
            if self.last:
              loss = tr.loss_fn(y, *mb[1:]) if tr.loss_fn is not None else y
              losses.append(loss.detach())
              y = tr.scaler.scale(loss)
              if mean and self.M > 1:
                y = y / self.M
        collected.append(graph.pop_collections())
        inputs[ins.mb], outputs[ins.mb] = x, y
      elif ins.op == S.SEND_F:
        y = outputs[ins.mb]
        if not getattr(self, "_meta_sent", False):
          self._send_meta(y)
          self._meta_sent = True
        # graph mode: y is the static output buffer of a captured graph, overwritten by the instance's next replay -> send a copy
        sends.append(self.p2p.send_fwd(y.detach().clone() if use_graphs else y.detach().contiguous()))
      elif ins.op == S.B:
        n_back += 1
        tr._last_micro_batch = n_back == self.M
        y = outputs.pop(ins.mb)
        # a recomputed forward (gradient checkpointing) re-reads the micro-batch: it must be this one, not the last one run
        graph.current_micro_batch = micro[ins.mb]
        if timing and self.last:                   # split the last stage's backward into host-issue and device time
          torch.cuda.current_stream().synchronize()    # (never a device-wide sync here: a posted NCCL receive would never drain)
          _tb0 = _time.perf_counter()
        with phase_scope(ModelPhase.BACKWARD):
          if use_graphs:
            st = self.graphed[ins.mb % len(self.graphed)]
            if self.last:
              gin = st.backward()
            else:
              g, req = recv_b.pop(ins.mb)
              req.wait()
              gin = st.backward(g)
            grads_in[ins.mb] = gin
          elif self.last:
            y.backward()
          else:
            g, req = recv_b.pop(ins.mb)
            req.wait()
            torch.autograd.backward(y, grad_tensors=g)
        if timing and self.last:
          _tb1 = _time.perf_counter()
          torch.cuda.current_stream().synchronize()
          _tb2 = _time.perf_counter()
          host_t["B_issue"] = host_t.get("B_issue", 0.0) + (_tb1 - _tb0)
          host_t["B_device_after_issue"] = host_t.get("B_device_after_issue", 0.0) + (_tb2 - _tb1)
        tr._first_micro_batch = False
      elif ins.op == S.SEND_B:
        x = inputs.pop(ins.mb)
        sends.append(self.p2p.send_bwd(grads_in.pop(ins.mb).clone() if use_graphs else x.grad.contiguous()))
      # REDUCE / APPLY are executed by the trainer after the program
    if timing:
      t_issue = _time.perf_counter()
      torch.cuda.current_stream().synchronize()
      t_done = _time.perf_counter()
      self._timing_rows = getattr(self, "_timing_rows", 0) + 1
      if self._timing_rows in (3, 5):
        print("[pipe timing rank %d stage %d graphs=%s] host issue per op (ms): %s | device tail after last issue %.1f ms" % (
            tr.plan.rank, self.stage, bool(self.graphed), {str(k): round(v * 1e3, 1) for k, v in host_t.items()},
            (t_done - t_issue) * 1e3), flush=True)
      self._last_op = None
    for w in sends:
      w.wait()
    inputs.clear()
    if hasattr(self.p2p, "flush"):
      self.p2p.flush()
    # the loss lives on the last stage; share its mean with every stage of the replica
    stat = torch.zeros(1, device=self.device, dtype=torch.float32)
    if self.last and losses:
      stat[0] = torch.stack([l.float() for l in losses]).mean() if mean else torch.stack([l.float() for l in losses]).sum()
    dist.all_reduce(stat, group=self.replica_group)
    return [stat[0]], collected

  @torch.no_grad()
  def forward_only(self, batch: Tuple[Any, ...]):
    """Evaluation: stages run back to back, no micro-batching."""
    Graph.get().current_micro_batch = batch
    if self.first:
      x = batch[0]
    else:
      if self._shape_fwd is None:
        self._shape_fwd = self._recv_meta()
      x = torch.empty((batch[0].shape[0],) + tuple(self._shape_fwd[0][1:]), dtype=self._shape_fwd[1], device=self.device)
      self.p2p.recv_fwd(x).wait()
    y = self.module(x)
    if not self.last:
      if not getattr(self, "_meta_sent", False):
        self._send_meta(y)
        self._meta_sent = True
      self.p2p.send_fwd(y.contiguous()).wait()
      return None
    if self.tr.loss_fn is not None and len(batch) > 1:
      return self.tr.loss_fn(y, *batch[1:])
    return y                                         # no labels: the last stage returns the model's output (predictions)

  def all_reduce_over_stages(self, t: torch.Tensor) -> torch.Tensor:
    dist.all_reduce(t, group=self.replica_group)
    return t
