#!/usr/bin/env python
"""Benchmarks of BASELINE.json's configs on N B200s of one node; the default is the headline.

  python bench.py --gpus 1 --steps 20 --warmup 5                         # GPT-2-XL, data parallel (headline)
  torchrun ... bench.py --gpus 8                                         # same, 8-way DP with the fused K1 path overlapped
  torchrun ... bench.py --gpus 8 --parallelism pp2 --micro-batches 8     # config 4: 2-stage 1F1B pipeline x 4-way DP
  torchrun ... bench.py --gpus 8 --zero v3 --gc auto --offload v0        # config 5: ZeRO-3 + recompute + CPU offload
  torchrun ... bench.py --gpus 8 --workload bert --model large --parallelism tp8     # config 3: BERT-large split(8)
  torchrun ... bench.py --gpus 8 --workload resnet50                     # config 2: ResNet-50 DP (images/s)
  ... --impl baseline     the library arm (baseline/torch_library_arm.py: cuBLASLt + SDPA + DDP + fused multi-tensor AdamW;
                          for tp: NCCL collectives + separate GEMMs) — none of the repo's kernels for gpt2 / resnet50
  ... --impl reference    the TF-1.15 reference: not installable in this image, prints {"unavailable": ...}
  ... --dump-outputs DIR  after the timed steps, save the last one's loss and a fixed sample of the updated parameters as .npy
                          (same arguments -> same inputs and, for one build, the same outputs, so two builds compare
                          output for output)

Metric/config follow BASELINE.json: GPT-2-XL (48 layers, d=1600, 25 heads), sequence 1024, bf16 compute with fp32 master
weights, synthetic tokens, random-init weights, full training step (forward + backward + gradient reduction + AdamW)
through the public ``epl.Trainer`` API.

Timed region: exactly K steps bracketed by barrier + ``torch.cuda.synchronize()``, CUDA events on the launching stream,
max over ranks.  ``value`` uses device-resident inputs; ``e2e`` repeats the measurement with every step's inputs copied
from pinned host memory and the loss read back.  ``reduce_apply.exposed_ms`` is the CUDA-event span from the end of
backward to the end of the step (what gradient reduction + optimizer add to the critical path).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def parse():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=10)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="epl", choices=["epl", "reference", "baseline"])
  ap.add_argument("--workload", default="gpt2", choices=["gpt2", "bert", "resnet50"])
  ap.add_argument("--model", default="", help="gpt2: tiny|small|medium|large|xl (default xl); bert: tiny|base|large (default large)")
  ap.add_argument("--batch", type=int, default=0, help="sequences (images) per GPU per step (per micro-batch for pipelines)")
  ap.add_argument("--seq", type=int, default=0)
  ap.add_argument("--layers", type=int, default=0, help="override the number of transformer layers (diagnostics)")
  ap.add_argument("--parallelism", default="auto", help="auto | dp | pp<S> (S-stage pipeline x DP) | tp<N> (bert: split(N))")
  ap.add_argument("--micro-batches", type=int, default=1)
  ap.add_argument("--zero", default="")
  ap.add_argument("--gc", default="")
  ap.add_argument("--offload", default="")
  ap.add_argument("--no-e2e", action="store_true")
  ap.add_argument("--no-graph", action="store_true", help="do not capture the training step in a CUDA graph")
  ap.add_argument("--profile", default="", help="write a per-kernel GPU time table of 2 extra steps to this file")
  ap.add_argument("--dump-outputs", default="", metavar="DIR",
                  help="write what the last timed step returned on rank 0 (loss, sample of rank 0's updated parameters: its "
                       "shard or stage under ZeRO-3 / tensor / pipeline parallelism) to DIR/<name>.npy")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  return args


class ClockSampler(threading.Thread):
  """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

  def __init__(self, index: int):
    super().__init__(daemon=True)
    self.index, self.rows, self._halt = index, [], threading.Event()

  def run(self):
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    while not self._halt.is_set():
      try:
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
          self.rows.append([c.strip() for c in out.split(",")])
      except Exception:
        pass
      self._halt.wait(0.2)

  def stop(self):
    self._halt.set()
    self.join(timeout=3)
    sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
    reasons = []
    for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
      if any(len(r) > col and r[col].lower().startswith("active") for r in self.rows):
        reasons.append(name)
    smax = max((float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()), default=0.0)
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax or None, "reasons": reasons, "samples": len(self.rows)}


DUMP_PARAM_SAMPLE = 1 << 22          # 16 MB of float32: enough to see a wrong update, small enough to store and compare


def dump_outputs(wl, loss, out_dir):
  """What a caller of the timed step receives: its loss, and the model parameters it updated in place.

  All parameters, flattened and concatenated in ``named_parameters()`` order, are sampled at fixed positions (seeded, sorted),
  so two builds run with the same arguments write arrays that compare element for element; a model smaller than the sample
  is written whole."""
  import numpy as np
  import torch
  model = wl.trainer.model if wl.trainer is not None else wl.lib.raw
  params = [p.detach() for _, p in model.named_parameters()]
  total = sum(p.numel() for p in params)
  if total <= DUMP_PARAM_SAMPLE:
    sample = torch.cat([p.reshape(-1).float().cpu() for p in params])
  else:
    idx = torch.randint(total, (DUMP_PARAM_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
    parts, start = [], 0
    for p in params:
      lo, hi = torch.searchsorted(idx, torch.tensor([start, start + p.numel()])).tolist()
      if hi > lo:
        parts.append(p.reshape(-1)[(idx[lo:hi] - start).to(p.device)].float().cpu())
      start += p.numel()
    sample = torch.cat(parts)
  os.makedirs(out_dir, exist_ok=True)
  np.save(os.path.join(out_dir, "loss.npy"), np.asarray(float(loss), dtype=np.float32))
  np.save(os.path.join(out_dir, "parameters.npy"), sample.numpy())


# ============================================================================================ workloads
class Workload(object):
  """What a benchmark needs from a model family: the trainer (product or library arm), pinned host batches, units/step."""
  unit = "tokens"

  def __init__(self, args, dev, world, rank):
    self.args, self.dev, self.world, self.rank = args, dev, world, rank
    self.trainer = None               # epl.Trainer (product / in-engine baseline)
    self.lib = None                   # baseline.torch_library_arm.LibraryTrainer
    self.meta = {}

  def step(self, batch):
    if self.lib is not None:
      return self.lib.step(*batch)
    return self.trainer.step(*batch).loss


def _epl_conf(args, stages, M):
  conf = {"amp.level": "bf16", "zero.level": args.zero, "gradient_checkpoint.type": args.gc, "offload.level": args.offload,
          "pipeline.num_micro_batch": M}
  if args.impl == "baseline":
    conf["communication.fused_kernels"] = False
  return conf


class GPT2Workload(Workload):
  def __init__(self, args, dev, world, rank):
    super().__init__(args, dev, world, rank)
    import torch
    import easyparallellibrary_b200 as epl
    from easyparallellibrary_b200.models.gpt2 import GPT2, GPT2Config, lm_loss
    name = args.model or "xl"
    seq = args.seq or 1024
    par = "dp" if args.parallelism == "auto" else args.parallelism
    stages = int(par[2:] or 2) if par.startswith("pp") else 1
    if par.startswith("tp"):
      raise SystemExit("GPT-2-XL has 25 attention heads: no tensor-parallel degree in {2,4,8} divides them; "
                       "the tensor-parallel config of BASELINE.json is --workload bert --model large --parallelism tp8")
    M = args.micro_batches if args.micro_batches > 1 else (8 if stages > 1 else 1)
    batch = args.batch or 8                                    # pipeline: 8 micro-batches of 8 sequences = 64 per replica
    extra = {"n_layer": args.layers} if args.layers else {}
    cfg = GPT2Config.named(name, num_pipeline_stages=stages, tie_embeddings=(stages == 1), n_positions=max(1024, seq), **extra)
    self.cfg, self.seq, self.stages, self.M = cfg, seq, stages, M
    torch.manual_seed(1234)
    pure_library = args.impl == "baseline" and stages == 1 and not args.zero and not args.offload
    if pure_library:
      from baseline.torch_library_arm import LibraryTrainer, TorchGPT2
      with torch.device(dev):
        model = TorchGPT2(cfg.vocab_size, cfg.n_positions, cfg.n_embd, cfg.n_layer, cfg.n_head)
      self.lib = LibraryTrainer(model, dev, world, lr=1e-4, weight_decay=0.01)
      replicas = world
      self.meta["arm"] = "library: cuBLASLt linears + SDPA + DDP(bf16 grads, overlapped) + fused multi-tensor AdamW on fp32 masters"
    else:
      epl.init(epl.Config(_epl_conf(args, stages, M)))
      with torch.device(dev):                      # random-init weights directly on the GPU
        if stages == 1:
          with epl.replicate(device_count=1):
            model = GPT2(cfg)
        else:
          model = GPT2(cfg)
      self.trainer = epl.Trainer(model, "adamw", lr=1e-4, weight_decay=0.01, baseline=(args.impl == "baseline"),
                                 loss_fn=lm_loss if stages > 1 else None, cuda_graph=not args.no_graph).build()
      replicas = self.trainer.plan.num_replicas
    self.replicas = replicas
    B = batch * (M if stages > 1 else 1)
    gen = torch.Generator(device="cpu").manual_seed(rank)
    self.host = [tuple(t.pin_memory() for t in [torch.randint(0, 50257, (B, seq), generator=gen)] * 2) for _ in range(4)]
    self.units_per_step = B * seq * replicas
    self.flops_per_unit = cfg.flops_per_token(seq)
    self.num_params = cfg.num_params
    self.config = {"model": "gpt2-" + name, "params": cfg.num_params, "global_batch": B * replicas, "seq_len": seq,
                   "parallelism": ("dp%d" % replicas) + ("xpp%d" % stages if stages > 1 else ""), "micro_batches": M,
                   "zero": args.zero or "none", "gradient_checkpoint": args.gc or "none", "offload": args.offload or "none",
                   "optimizer": "adamw fp32 master",
                   "l2": "working set (3 GB bf16 weights + activations) >> 126 MB L2; no flush needed"}
    self.metric = "tokens/sec (whole job, device-timed, max over ranks) GPT-2-XL training step"


class BertWorkload(Workload):
  def __init__(self, args, dev, world, rank):
    super().__init__(args, dev, world, rank)
    import torch
    import easyparallellibrary_b200 as epl
    from easyparallellibrary_b200.models.bert import Bert, BertConfig
    from easyparallellibrary_b200.ops import tp_fused
    name = args.model or "large"
    seq = args.seq or 384                         # the reference's SQuAD sequence length (examples/bert/run_squad.py)
    par = "dp" if args.parallelism == "auto" else args.parallelism
    tp = int(par[2:] or world) if par.startswith("tp") else 1
    stages = int(par[2:] or 2) if par.startswith("pp") else 1
    M = args.micro_batches if args.micro_batches > 1 else (8 if stages > 1 else 1)
    batch = args.batch or (32 if tp > 1 else 12)  # per TP group / per replica
    conf = _epl_conf(args, stages, M)
    if tp > 1:
      conf["cluster.colocate_split_and_replicate"] = True
      tp_fused.USE_FUSED = args.impl != "baseline"          # baseline: NCCL all-gather / reduce-scatter + separate GEMMs
      conf.pop("communication.fused_kernels", None)
    epl.init(epl.Config(conf))
    if tp > 1:
      epl.set_default_strategy(epl.replicate(device_count=1))
    cfg = BertConfig.named(name, num_pipeline_stages=stages, tensor_parallel=tp)
    torch.manual_seed(1234)
    with torch.device(dev):
      model = Bert(cfg)
    self.trainer = epl.Trainer(model, "adamw", lr=1e-4, weight_decay=0.01, baseline=(args.impl == "baseline" and tp == 1),
                               cuda_graph=(not args.no_graph and args.impl != "baseline")).build()
    groups = world // tp if tp > 1 else self.trainer.plan.num_replicas
    self.replicas = groups
    B = batch * (M if stages > 1 else 1)
    gen = torch.Generator(device="cpu").manual_seed(rank // tp if tp > 1 else rank)      # a TP group shares its batch
    self.host = []
    for _ in range(4):
      ids = torch.randint(0, cfg.vocab_size, (B, seq), generator=gen)
      s, e = torch.randint(0, seq, (B,), generator=gen), torch.randint(0, seq, (B,), generator=gen)
      self.host.append(tuple(t.pin_memory() for t in (ids, s, e)))
    self.units_per_step = B * seq * groups
    self.flops_per_unit = cfg.flops_per_token(seq)
    self.num_params = sum(p.numel() for p in model.parameters()) * (tp if tp > 1 else 1)
    self.config = {"model": "bert-" + name, "global_batch": B * groups, "seq_len": seq,
                   "parallelism": ("tp%d" % tp if tp > 1 else "") + ("dp%d" % groups) + ("xpp%d" % stages if stages > 1 else ""),
                   "micro_batches": M, "tp_collectives": ("fused all-gather->GEMM / GEMM->reduce-scatter kernels" if tp > 1 and tp_fused.USE_FUSED
                                                           else ("NCCL + separate GEMMs" if tp > 1 else "none")),
                   "optimizer": "adamw fp32 master", "l2": "weights + activations >> 126 MB L2; no flush needed"}
    self.metric = "tokens/sec (whole job, device-timed, max over ranks) BERT-%s SQuAD-head training step" % name


class ResNetWorkload(Workload):
  unit = "images"

  def __init__(self, args, dev, world, rank):
    super().__init__(args, dev, world, rank)
    import torch
    import easyparallellibrary_b200 as epl
    from easyparallellibrary_b200.models.resnet import ResNet50
    batch = args.batch or 128
    classes = 10000                               # the reference's wide head (examples/resnet/resnet_dp.py:26-66)
    torch.manual_seed(1234)
    if args.impl == "baseline":
      from baseline.torch_library_arm import LibraryTrainer

      class Net(torch.nn.Module):
        def __init__(self):
          super().__init__()
          from easyparallellibrary_b200.models.resnet import ResNet50Backbone
          self.backbone = ResNet50Backbone()
          self.head = torch.nn.Linear(self.backbone.out_features, classes)

        def forward(self, images, labels):
          return torch.nn.functional.cross_entropy(self.head(self.backbone(images)).float(), labels)
      with torch.device(dev):
        model = Net()
      self.lib = LibraryTrainer(model.to(memory_format=torch.channels_last), dev, world, lr=1e-4, weight_decay=0.01)
      self.replicas = world
    else:
      epl.init(epl.Config(_epl_conf(args, 1, 1)))
      with torch.device(dev):
        with epl.replicate(device_count=1):
          model = ResNet50(num_classes=classes)
      self.trainer = epl.Trainer(model, "adamw", lr=1e-4, weight_decay=0.01, cuda_graph=not args.no_graph).build()
      self.replicas = self.trainer.plan.num_replicas
    gen = torch.Generator(device="cpu").manual_seed(rank)
    self.host = [(torch.randn(batch, 3, 224, 224, generator=gen).bfloat16().pin_memory(),
                  torch.randint(0, classes, (batch,), generator=gen).pin_memory()) for _ in range(2)]
    self.units_per_step = batch * self.replicas
    self.flops_per_unit = 3.0 * 2.0 * (4.09e9 + 2048 * classes)          # fwd MACs of ResNet-50 (4.09 G) + head, x2 flops, x3 fwd+bwd
    self.num_params = 25.6e6 - 2.05e6 + 2048 * classes
    self.config = {"model": "resnet50 + %d-class head" % classes, "global_batch": batch * self.replicas, "image": "3x224x224 bf16 channels-last",
                   "parallelism": "dp%d" % self.replicas, "convolutions": "cuDNN (library op in both arms)", "optimizer": "adamw fp32 master",
                   "l2": "activations (GBs) >> 126 MB L2; no flush needed"}
    self.metric = "images/sec (whole job, device-timed, max over ranks) ResNet-50 training step"


# ============================================================================================ main
def main():
  args = parse()
  if os.environ.get("EPL_HANG_DUMP"):          # debugging aid: dump every Python stack if the run stalls
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ["EPL_HANG_DUMP"]), exit=True)
  if args.impl == "reference":
    print(json.dumps({"impl": "reference", "unavailable":
                      "reference is TensorFlow-1.15/Python<=3.8 only (setup.py imports tensorflow; csrc links TF libs); "
                      "offline pip install into baseline/_ref fails with ModuleNotFoundError: tensorflow (see DESIGN.md)"}))
    return 0

  if args.parallelism.startswith("pp"):
    # pipeline: a first-time kernel launch must never block behind a posted NCCL receive (see parallel/pipeline.py), so load
    # every CUDA module up front instead of lazily; must be set before the CUDA context exists
    os.environ.setdefault("CUDA_MODULE_LOADING", "EAGER")
  import torch
  import torch.distributed as dist
  from easyparallellibrary_b200.ops import _lib

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  if world != args.gpus and world == 1 and args.gpus > 1:
    # convenience: re-launch ourselves under torchrun
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
           "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000)] + sys.argv
    return subprocess.call(cmd)
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  if world > 1 and not dist.is_initialized():
    dist.init_process_group("nccl", device_id=dev)

  wl = {"gpt2": GPT2Workload, "bert": BertWorkload, "resnet50": ResNetWorkload}[args.workload](args, dev, world, rank)
  trainer = wl.trainer
  dev_batches = [tuple(t.to(dev) for t in b) for b in wl.host]
  n_host = len(wl.host)

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def run(n, e2e):
    sink, loss = 0.0, None
    for i in range(n):
      if e2e:
        batch = tuple(t.to(dev, non_blocking=True) for t in wl.host[i % n_host])      # pinned host -> device, every step
        loss = wl.step(batch)
        sink += float(loss)                        # device -> host read of the step's result
      else:
        loss = wl.step(dev_batches[i % n_host])
    return loss, sink

  # exposed reduce + optimizer phase per step: CUDA events on the main stream around Trainer._reduce_and_apply.  With the
  # overlapped K1 path the bucket kernels of all but the last bucket were launched during backward, so this span is what
  # the gradient reduction + optimizer really add to the step.
  phase = None
  if trainer is not None:
    try:
      from easyparallellibrary_b200.utils.metric import PhaseTimer
      phase = PhaseTimer(trainer, "_reduce_and_apply", use_cuda=True)
    except Exception:
      phase = None
  apply_ms = [None]

  def timed(n, e2e):
    barrier()
    if phase is not None:
      phase.reset()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
      sampler.start()
    l0 = _lib.launches
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    loss, _ = run(n, e2e)
    t1.record()
    barrier()
    ms = t0.elapsed_time(t1)
    clocks = sampler.stop() if sampler else None
    try:
      pm = phase.total_ms() / n if (phase is not None and not e2e) else -1.0
    except Exception:
      pm = -1.0
    t = torch.tensor([ms, pm], device=dev, dtype=torch.float64)
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if not e2e:
      apply_ms[0] = float(t[1].item()) if float(t[1].item()) >= 0 else None
    return float(t[0].item()), loss, clocks, _lib.launches - l0

  # set-up, not warm-up: the trainer runs its first GraphedStep.WARMUP steps eagerly and CAPTURES the CUDA graph of the step in
  # the next one (a pipeline captures its stage graphs in its first step).  Do that here, so that whatever --warmup says, the W
  # warm-up steps and the K timed steps all run the steady-state program (with --warmup 3 the capture used to land on the first
  # timed step: 8-GPU session of round 2, profiles/r2_session_8gpu.md).
  setup_steps = 0
  g = getattr(trainer, "_graphed", None) if trainer is not None else None
  if g is not None and g.enabled:
    setup_steps = g.WARMUP + 1
  elif getattr(wl, "stages", 1) > 1:
    setup_steps = 1
  if setup_steps:
    run(setup_steps, False)
    barrier()
  run(max(args.warmup, 3), False)
  if args.profile:                               # kernel timeline of 2 steps (CUPTI via torch.profiler); never a bench value
    from torch.profiler import profile, ProfilerActivity
    barrier()
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
      run(2, False)
      torch.cuda.synchronize()
    if rank == int(os.environ.get("EPL_BENCH_PROFILE_RANK", "0")):
      from easyparallellibrary_b200.profiler.timeline import kernel_table
      text, _ = kernel_table(prof.events())
      with open(args.profile, "w") as f:
        f.write(text)
    barrier()
  ms, loss, clocks, launches = timed(args.steps, False)
  if args.dump_outputs and rank == 0:            # before the untimed steps below move the weights on
    dump_outputs(wl, loss, args.dump_outputs)
  value = wl.units_per_step * args.steps / (ms / 1e3)
  graphed = trainer is not None and getattr(trainer, "_graphed", None) is not None and trainer._graphed.graph is not None
  if graphed and phase is not None:
    # the replayed graph contains the reduce/apply phase but not the host-side timer: measure its exposed span on a few
    # eager steps (same kernels, same streams), outside the timed region
    trainer._graphed.enabled = False
    keep = (ms, loss, clocks, launches)
    run(1, False)
    timed(3, False)
    trainer._graphed.enabled = True
    ms, loss, clocks, launches = keep
  e2e = None
  if not args.no_e2e:
    run(2, True)
    ms_e, _, _, _ = timed(args.steps, True)
    e2e = {"value": wl.units_per_step * args.steps / (ms_e / 1e3), "unit": wl.unit + "/s",
           "h2d_bytes_per_step": int(sum(t.numel() * t.element_size() for t in wl.host[0])), "d2h_bytes_per_step": 4,
           "ms_per_step": ms_e / args.steps}
  if rank == 0:
    peaks = {}
    try:
      peaks = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "MEASURED_PEAKS.json")))
    except Exception:
      pass
    flops = wl.flops_per_unit * value / world
    cfg = dict(wl.config)
    if trainer is not None and getattr(trainer, "fused", None) is not None:
      dp_size = max(c.size for c in trainer.dp_comms.values())
      overlapped = (trainer.fused.overlap and dp_size >= trainer.fused.overlap_min_world and not trainer.plan.pipeline
                    and trainer.max_grad_norm is None)
      cfg["dp_gradient_path"] = "fused reduce-scatter + AdamW + all-gather kernel (K1 %s), %s" % (
          trainer.fused.kernel,
          "overlapped with backward on %d CTAs, last bucket on the whole GPU" % trainer.fused.overlap_blocks if overlapped
          else "after backward (overlap starts at %d-way data parallelism)" % trainer.fused.overlap_min_world)
      cfg["gradient_buckets"] = sum(len(f.buckets) for f in trainer.flats.values())
    cfg.update(wl.meta)
    cfg["cuda_graph"] = bool(graphed)
    pipe = getattr(trainer, "pipe", None) if trainer is not None else None
    if pipe is not None and getattr(pipe, "graphed", None):
      cfg["cuda_graph"] = "per stage: forward and backward of a micro-batch replay from CUDA graphs"
    cfg["setup_steps_before_warmup"] = setup_steps
    line = {
        "metric": wl.metric, "value": value, "unit": wl.unit + "/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic, random-init weights", "impl": args.impl, "config": cfg,
        "model_tflops_per_gpu": flops / 1e12,
        "mfu_of_measured_bf16_sustained": (flops / 1e12) / peaks["bf16_tflops_sustained"] if peaks.get("bf16_tflops_sustained") else None,
        "loss": float(loss), "clocks": clocks, "gpu_launches": launches, "e2e": e2e,
    }
    try:
      if apply_ms[0] is not None and getattr(wl, "stages", 1) == 1 and trainer is not None and not trainer.zero3:
        from easyparallellibrary_b200.utils.metric import fused_dp_roofline_ms
        roof = fused_dp_roofline_ms(int(wl.num_params), wl.replicas, hbm_gbs=float(peaks.get("hbm_gbs", 6400.0)))
        line["reduce_apply"] = {
            "exposed_ms_per_step": apply_ms[0], "ms_per_step": apply_ms[0],
            "whole_phase_roofline_ms": roof,
            "what": ("fused reduce-scatter + AdamW + all-gather kernels (NVLink peer memory)" if trainer.fused is not None
                     else ("bucketed NCCL all-reduce + Adam" if world > 1 else "fused AdamW")),
            "roofline": "max(per-direction NVLink bytes = 2 x (W-1)/W x 2 B/param at 770 GB/s measured peer bandwidth, HBM bytes of the "
                        "1/W AdamW shard + the gradient/weight streams at measured HBM bandwidth); the exposed span can be below "
                        "it because all but the last bucket run during backward"}
    except Exception:
      pass
    print(json.dumps(line))
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()
  return 0


if __name__ == "__main__":
  sys.exit(main())
