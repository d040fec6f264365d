"""Single-process CPU tests of the runtime features: gradient checkpoint, offload, AMP loss scale, grouped apply,
checkpoint save/resume, ShardingLoader, IO slicing, profiler hooks, auto stage search, launcher command lines.
Tolerances follow the reference's A/B tests (|dloss| < 1e-6 offload / grouped apply, < 1e-5 checkpoint)."""
import json
import os
import time

import pytest
import torch
from torch import nn

import easyparallellibrary_b200 as epl


def _net(seed=0):
  torch.manual_seed(seed)
  blocks = [nn.Sequential(nn.Linear(16, 16), nn.Tanh(), nn.Linear(16, 16), nn.Dropout(0.0)) for _ in range(6)]
  return nn.Sequential(nn.Linear(8, 16), *blocks, nn.Linear(16, 1))


def _run(conf, steps=4, opt="adamw", **kw):
  epl.init(epl.Config(conf), init_process_group=False)
  with epl.replicate(1):
    model = _net()
  kw.setdefault("lr", 1e-2)
  tr = epl.Trainer(model, opt, loss_fn=lambda o, y: ((o - y) ** 2).mean(), **kw)
  torch.manual_seed(1)
  X, Y = torch.randn(steps, 8, 8), torch.randn(steps, 8, 1)
  return [tr.step(X[i], Y[i]).item() for i in range(steps)], tr


def test_gradient_checkpoint_auto_and_collection_match_plain():
  base, _ = _run({})
  auto, tr = _run({"gradient_checkpoint.type": "auto"}, example_inputs=[torch.randn(8, 8)])
  assert max(abs(a - b) for a, b in zip(base, auto)) < 1e-5
  from easyparallellibrary_b200.runtime.gradient_checkpoint import _Checkpointed
  assert sum(isinstance(m, _Checkpointed) for m in tr.model.modules()) == 6      # the six repeated blocks
  epl.init(epl.Config({"gradient_checkpoint.type": "collection"}), init_process_group=False)
  with epl.replicate(1):
    model = _net()
  for blk in list(model)[1:4]:
    epl.add_to_collection(blk, epl.GraphKeys.GC_CHECKPOINTS)
  tr = epl.Trainer(model, "adamw", loss_fn=lambda o, y: ((o - y) ** 2).mean(), lr=1e-2)
  torch.manual_seed(1)
  X, Y = torch.randn(4, 8, 8), torch.randn(4, 8, 1)
  coll = [tr.step(X[i], Y[i]).item() for i in range(4)]
  assert max(abs(a - b) for a, b in zip(base, coll)) < 1e-5
  with pytest.raises(RuntimeError):
    _run({"gradient_checkpoint.type": "collection"})


def test_offload_and_grouped_apply_match_plain():
  base, _ = _run({})
  off, tr = _run({"offload.level": "v0", "offload.weights": False})            # optimizer state only
  assert max(abs(a - b) for a, b in zip(base, off)) < 1e-6
  from easyparallellibrary_b200.runtime.offload import OffloadedOptimizer
  assert all(isinstance(o, OffloadedOptimizer) for o in tr.optimizers[0]) and not tr.zero3
  off, tr = _run({"offload.level": "v0"})                                       # weights too: the per-layer engine, shards on the host
  assert max(abs(a - b) for a, b in zip(base, off)) < 1e-6
  units = tr.zero3[0].units
  assert units and all(u.offload and isinstance(u.opt, OffloadedOptimizer) for u in units)
  assert all(p.numel() == 0 for u in units for p in u.params)                   # released between steps
  grp, _ = _run({"optimizer.num_apply_group": 4})
  assert max(abs(a - b) for a, b in zip(base, grp)) < 1e-6
  ga, _ = _run({"pipeline.num_micro_batch": 4})
  assert max(abs(a - b) for a, b in zip(base, ga)) < 1e-5


def test_dynamic_loss_scale_skips_and_recovers():
  from easyparallellibrary_b200.runtime.amp import DynamicLossScale, FixedLossScale, make_scaler
  s = DynamicLossScale(initial=2.0 ** 15, increment_period=3)
  assert s.update(True) and s.loss_scale == 2.0 ** 14
  assert not s.update(False) and not s.update(False)
  assert not s.update(False) and s.loss_scale == 2.0 ** 15            # doubled after 3 good steps
  for _ in range(40):
    s.update(True)
  assert s.loss_scale == 1.0                                           # floor
  assert isinstance(make_scaler("o1", 128.0), FixedLossScale) and make_scaler("o1", 128.0).loss_scale == 128.0
  assert make_scaler("", "dynamic").loss_scale == 1.0
  # an overflowing step is skipped (weights untouched) and the scale halves — reference dnn_data_parallel.py:68-74
  epl.init(epl.Config({"amp.level": "O1", "amp.loss_scale": "dynamic"}), init_process_group=False)
  with epl.replicate(1):
    model = nn.Linear(4, 1)
  tr = epl.Trainer(model, "sgd", loss_fn=lambda o, y: ((o.float() - y) ** 2).mean(), lr=0.1)
  x, y = torch.full((2, 4), 3e4), torch.zeros(2, 1)
  before = None
  out = tr.step(x, y)
  w0 = model.weight.detach().float().clone()
  assert out.skipped and tr.scaler.loss_scale == 2.0 ** 14 and tr.global_step == 0
  out = tr.step(x * 0, y)
  assert not out.skipped and tr.global_step == 1


def test_checkpoint_save_and_resume(tmp_path):
  from easyparallellibrary_b200.runtime.saver import load_checkpoint, save_checkpoint
  losses, tr = _run({}, steps=3)
  save_checkpoint(tr, str(tmp_path), bucket_bytes=1024)
  assert len([f for f in os.listdir(tmp_path) if f.startswith("model-")]) > 1       # bounded-memory buckets
  torch.manual_seed(5)
  x, y = torch.randn(8, 8), torch.randn(8, 1)
  expect = [tr.step(x, y).item() for _ in range(2)]
  _, tr2 = _run({}, steps=0)
  step = load_checkpoint(tr2.build(), str(tmp_path))
  assert step == 3 and tr2.global_step == 3
  got = [tr2.step(x, y).item() for _ in range(2)]
  assert max(abs(a - b) for a, b in zip(expect, got)) < 1e-6 and tr2.global_step == 5


def test_sharding_loader_rename_and_slice():
  from easyparallellibrary_b200.ops import tensor_parallel as tp
  from easyparallellibrary_b200.runtime.saver import ShardingLoader
  ckpt = {"enc.w": torch.arange(24.0).view(6, 4), "enc.b": torch.arange(6.0)}
  m = nn.Linear(4, 3)
  loaded = ShardingLoader(ckpt, {r"enc\.w": "weight", r"enc\.b": "bias"}, {"weight": ((3, 3), (0, 4)), "bias": (3, 3)}).load_into(m)
  assert sorted(loaded) == ["bias", "weight"]
  assert torch.equal(m.weight.data, ckpt["enc.w"][3:6]) and torch.equal(m.bias.data, ckpt["enc.b"][3:6])
  epl.init(init_process_group=False)
  with epl.split(1):
    holder = nn.Module()
    holder.w = tp.add_weight((6, 4))
  assert ShardingLoader({"w": ckpt["enc.w"]}).load_into(holder) == ["w"]


def test_io_slicing_cases():
  from easyparallellibrary_b200.utils.io_slicing import slice_files
  f = list(range(12))
  assert slice_files(f, [1, 1], 0) == f[:6] and slice_files(f, [1, 1], 1) == f[6:]
  assert slice_files(f, [2, 1], 0) == f[:8] and slice_files(f, [2, 1], 1) == f[8:]
  assert slice_files(f, [2, 2], 1) == f[6:]                              # gcd-normalised
  assert slice_files(list(range(10)), [1, 1, 1], 0, drop_last_files=True) == [0, 1, 2]
  assert slice_files(list(range(10)), [1, 1, 1], 2, drop_last_files=True) == [6, 7, 8]
  assert slice_files(list(range(10)), [1, 1, 1], 0, unbalanced_io_slicing=True) == [0, 1, 2, 3]
  assert sorted(slice_files([0, 1], [1, 1, 1], 1)) == [0, 1]              # too few files: everyone reads all, rotated
  with pytest.raises(RuntimeError):
    slice_files([0, 1], [1, 1, 1], 1, drop_last_files=True)


def test_profiler_hooks(tmp_path):
  from easyparallellibrary_b200.profiler import FlopsProfilerHook, MemoryProfilerHook, profile_flops, profile_memory
  epl.init(init_process_group=False)
  with epl.replicate(1):
    model = _net()
  fl = profile_flops(model, [torch.randn(8, 8)], by="op")
  assert fl["Linear"] == 2.0 * 8 * (8 * 16 + 12 * 16 * 16 + 16) and fl["__total__"] >= fl["Linear"]
  tr = epl.Trainer(model, "adamw", loss_fn=lambda o, y: ((o - y) ** 2).mean(), lr=1e-2)
  fh, mh = FlopsProfilerHook(3 * fl["__total__"], use_cuda_events=False), MemoryProfilerHook(output_dir=str(tmp_path))
  tr.hooks += [fh, mh]
  for _ in range(3):
    tr.step(torch.randn(8, 8), torch.randn(8, 1))
  s = fh.summary()
  assert s["tflops"] > 0 and 0 < s["median_step_s"]
  assert mh.save() and os.path.exists(os.path.join(tmp_path, "memory_timeline.csv"))
  phases = [r["phase"] for r in mh.rows if r["step"] == 0]
  assert phases == ["persistent", "forward", "backward", "apply", "after_step"]       # sampled at every phase boundary of the step
  assert set(mh.phase_peaks()) == {"persistent", "forward", "backward", "apply", "after_step"}
  mh.close()
  mem = profile_memory(tr)
  assert mem["weights"] == mem["gradients"] > 0 and mem["optimizer_state_device"] >= 2 * mem["weights"]


def test_auto_parallel_stage_search():
  epl.init(epl.Config({"auto.auto_parallel": True, "pipeline.num_stages": 3, "pipeline.num_micro_batch": 2}), init_process_group=False)
  model = _net()
  tr = epl.Trainer(model, "adamw", loss_fn=lambda o, y: ((o - y) ** 2).mean(), lr=1e-2, example_inputs=[torch.randn(4, 8)]).build()
  g = epl.Graph.get()
  assert len(g.taskgraphs) == 3 and tr.plan.num_stages == 3
  sizes = [len(list(tr.stage_modules[s])) for s in range(3)]
  assert sum(sizes) == 8 and max(sizes) - min(sizes) <= 2
  out = tr.step(torch.randn(4, 8), torch.randn(4, 1))          # colocated on one device: stages run back to back
  assert out.loss is not None


def test_launcher_command_lines():
  from easyparallellibrary_b200.utils import launcher
  args = launcher.parse(["--num_workers", "2", "--gpu_per_worker", "2", "train.py", "--lr", "1"])
  cmds = launcher.build_commands(args)
  assert [c["rank"] for c in cmds] == [0, 1, 2, 3]
  assert cmds[3]["env"]["WORLD_SIZE"] == "4" and cmds[3]["env"]["LOCAL_RANK"] == "3" and cmds[3]["argv"][-2:] == ["--lr", "1"]
  tf = json.loads(cmds[2]["env"]["TF_CONFIG"])
  assert tf["task"] == {"type": "worker", "index": 1} and len(tf["cluster"]["worker"]) == 2
  args = launcher.parse(["--num_workers", "4", "--gpu_per_worker", "8", "--machine_list", "10.0.0.1:29500,10.0.0.2:29500",
                         "--machine_rank", "1", "run.sh"])
  cmds = launcher.build_commands(args)
  assert len(cmds) == 16 and cmds[0]["rank"] == 16 and cmds[0]["env"]["MASTER_ADDR"] == "10.0.0.1" and cmds[0]["argv"][0] == "bash"


def test_launcher_restarts_a_failed_job(tmp_path):
  """``epl-launch --max_restarts``: a job whose rank 1 dies in the first attempt is torn down and relaunched; the script sees
  which attempt it is (EPL_RESTART_COUNT) and, like a real job resuming from a checkpoint, succeeds the second time."""
  from easyparallellibrary_b200.utils import launcher
  script = tmp_path / "job.py"
  script.write_text(
      "import os, sys, time\n"
      "rank, attempt = int(os.environ['RANK']), int(os.environ['EPL_RESTART_COUNT'])\n"
      "open(os.path.join(%r, 'ran_%%d_%%d' %% (attempt, rank)), 'w').close()\n"
      "if attempt == 0 and rank == 1:\n"
      "  sys.exit(3)\n"
      "if attempt == 0:\n"
      "  time.sleep(30)          # a healthy rank of the failed attempt must be terminated, not waited for\n" % str(tmp_path))
  t0 = time.time()
  assert launcher.main(["--num_workers", "1", "--gpu_per_worker", "2", "--backend", "gloo", "--log_dir", str(tmp_path), str(script)]) == 3
  assert launcher.main(["--num_workers", "1", "--gpu_per_worker", "2", "--backend", "gloo", "--log_dir", str(tmp_path), "--max_restarts", "1",
                        str(script)]) == 0
  assert time.time() - t0 < 25
  assert all((tmp_path / ("ran_%d_%d" % (a, r))).exists() for a in (0, 1) for r in (0, 1))


def test_models_build_and_step_on_cpu():
  from easyparallellibrary_b200.models.bert import Bert, BertConfig
  from easyparallellibrary_b200.models.gpt2 import GPT2, GPT2Config
  from easyparallellibrary_b200.models.moe_transformer import MoEConfig, MoETransformer
  from easyparallellibrary_b200.models.resnet import ResNet50
  epl.init(init_process_group=False)
  with epl.replicate(1):
    m = GPT2(GPT2Config.named("tiny"))
  tr = epl.Trainer(m, "adamw", lr=1e-3)
  x = torch.randint(0, 512, (2, 32))
  a, b = tr.step(x, x).item(), tr.step(x, x).item()
  assert b < a
  epl.init(init_process_group=False)
  m = GPT2(GPT2Config.named("tiny", num_pipeline_stages=2, tie_embeddings=False))
  assert len(epl.Graph.get().taskgraphs) == 2 and epl.Graph.get().taskgraph_of(m.h[1]).index == 1
  epl.init(epl.Config({"cluster.colocate_split_and_replicate": True}), init_process_group=False)
  epl.set_default_strategy(epl.replicate(1))
  moe = MoETransformer(MoEConfig(vocab_size=128, d_model=32, d_ff=64, n_layer=2, n_head=4, num_experts=4, n_positions=32))
  tr = epl.Trainer(moe, "adamw", lr=1e-3)
  x = torch.randint(0, 128, (2, 16))
  assert tr.step(x, x).loss.isfinite()
  epl.init(init_process_group=False)
  with epl.replicate(1):
    bert = Bert(BertConfig.named("tiny"))
  tr = epl.Trainer(bert, "adamw", lr=1e-3)
  ids, pos = torch.randint(0, 1024, (2, 16)), torch.randint(0, 16, (2,))
  assert tr.step(ids, pos, pos).loss.isfinite()
  epl.init(epl.Config({"cluster.colocate_split_and_replicate": True}), init_process_group=False)
  r = ResNet50(num_classes=64, width=8, layers=(1, 1, 1, 1), split_head=True)
  tr = epl.Trainer(r, "sgd", lr=1e-2)
  assert tr.step(torch.randn(2, 3, 32, 32), torch.randint(0, 64, (2,))).loss.isfinite() and tr.has_split


def test_throughput_meter_and_plan_summary():
  """utils/metric.py + utils/summary_info.py (reference: utils/metric.py, utils/summary_info.py, Graph.format())."""
  import time
  import torch
  import easyparallellibrary_b200 as epl
  from easyparallellibrary_b200.utils.metric import ThroughputMeter
  from easyparallellibrary_b200.utils.summary_info import plan_summary
  meter = ThroughputMeter(items_per_step=64, warmup=2, unit="samples")
  for _ in range(5):
    time.sleep(0.002)
    meter.step()
  out = meter.summary()
  assert out["steps"] == 3 and out["ms_per_step"] > 1.0 and out["per_second"] > 0
  epl.init(epl.Config({"pipeline.num_micro_batch": 2}), init_process_group=False)
  with epl.replicate(1):
    model = torch.nn.Sequential(torch.nn.Linear(8, 8), torch.nn.ReLU(), torch.nn.Linear(8, 2))
  tr = epl.Trainer(model, "sgd", lr=0.1, loss_fn=lambda y, t: torch.nn.functional.cross_entropy(y, t))
  tr.build()
  text = plan_summary(tr)
  assert "stages=1" in text and "micro_batches=2" in text and "param group" in text


def _run_job(cmd, cwd, env, timeout, attempts=2):
  """Run a multi-process job; one retry absorbs transient failures of the host (port reuse, a loaded box) — a real defect
  fails twice."""
  import subprocess
  r = None
  for _ in range(attempts):
    r = subprocess.run(cmd, cwd=cwd, env=env, capture_output=True, text=True, timeout=timeout)
    if r.returncode == 0:
      break
  return r


@pytest.mark.parametrize("amp", [False, True])
def test_launcher_runs_a_two_process_job(tmp_path, amp):
  """True multi-process job through ``epl-launch`` (reference: tests/Makefile:12-13 -> test_launcher.sh / test_amp_parallel.sh):
  2 workers x 1 process on CPUs (gloo), a 2-layer MLP for 10 steps; success = exit code 0, identical replicas, and (amp) an
  overflowing step skipped on every rank."""
  import subprocess
  import sys
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  cmd = [sys.executable, "-m", "easyparallellibrary_b200.utils.launcher", "--num_workers", "2", "--gpu_per_worker", "1", "--backend", "gloo",
         "--log_dir", str(tmp_path), os.path.join(root, "tests", "scripts", "dnn_data_parallel.py")] + (["--amp"] if amp else [])
  env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
  r = _run_job(cmd, root, env, 300)
  logs = "".join(open(os.path.join(tmp_path, f)).read()[-1500:] for f in sorted(os.listdir(tmp_path)))
  assert r.returncode == 0, r.stdout[-1500:] + logs
  assert r.stdout.count(" ok: ") == 2, r.stdout


@pytest.mark.parametrize("script,argv", [
    ("train_gpt2.py", ["--model", "tiny", "--batch", "2", "--seq", "32", "--steps", "2"]),
    ("train_gpt2.py", ["--model", "tiny", "--batch", "2", "--seq", "32", "--steps", "2", "--zero", "v3", "--gc", "auto"]),
    ("train_bert_pipeline.py", ["--size", "tiny", "--batch", "2", "--seq", "16", "--steps", "2"]),
    ("train_moe.py", ["--batch", "2", "--seq", "16", "--steps", "2", "--experts", "4"]),
    ("moe/train_t5_moe.py", ["--size", "tiny", "--batch", "2", "--seq", "32", "--steps", "3", "--experts", "4"]),
    ("resnet/resnet_dp.py", ["--width", "8", "--classes", "32", "--image", "32", "--batch", "4", "--steps", "2", "--gc", "auto"]),
    ("resnet/resnet_split.py", ["--width", "8", "--classes", "32", "--image", "32", "--batch", "4", "--steps", "2"]),
    ("bert/run_squad.py", ["--model", "tiny", "--do_train", "--do_predict", "--num_train_steps", "3", "--train_batch_size", "4", "--synthetic_paragraphs", "8",
                           "--auto_parallel", "--num_pipe_stages", "2", "--num_micro_batch", "2"]),
    ("bert/run_squad.py", ["--model", "tiny", "--do_train", "--do_predict", "--num_train_steps", "3", "--train_batch_size", "4",
                           "--synthetic_paragraphs", "8"]),
])
def test_example_scripts_run_on_cpu(script, argv, tmp_path):
  """The examples (reference: examples/{bert,resnet,moe}) stay runnable: two steps of a tiny configuration on one CPU process."""
  import subprocess
  import sys
  if script == "bert/run_squad.py":                  # its corpus, features and checkpoint go to a directory of this test only
    argv = argv + ["--output_dir", str(tmp_path)]
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""), CUDA_VISIBLE_DEVICES="")
  for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "TF_CONFIG"):
    env.pop(k, None)
  r = subprocess.run([sys.executable, os.path.join(root, "examples", script)] + argv, cwd=root, env=env, capture_output=True, text=True,
                     timeout=600)
  assert r.returncode == 0 and "step 1 loss" in r.stdout, r.stdout[-1500:] + r.stderr[-2500:]


def test_step_watchdog_and_timeline_hook(tmp_path):
  """Failure detection (runtime/watchdog.py) and the kernel/operator timeline hook (profiler/timeline.py)."""
  import time
  from easyparallellibrary_b200.profiler.timeline import TimelineHook
  from easyparallellibrary_b200.runtime.watchdog import StepWatchdog
  fired = []
  dog = StepWatchdog(timeout_s=0.15, on_timeout=lambda step, elapsed: fired.append((step, elapsed)), poll_s=0.02)
  try:
    dog.before_step(None); time.sleep(0.05); dog.after_step(None, None)          # a healthy step
    assert not fired
    dog.before_step(None); time.sleep(0.4)                                       # a hung step fires exactly once
    assert len(fired) == 1 and fired[0][0] == 1 and fired[0][1] > 0.15
    dog.after_step(None, None)
  finally:
    dog.close()
  epl.init(init_process_group=False)
  with epl.replicate(1):
    model = nn.Sequential(nn.Linear(16, 32), nn.Tanh(), nn.Linear(32, 4))
  tr = epl.Trainer(model, "adamw", lr=1e-3, loss_fn=lambda y, t: nn.functional.cross_entropy(y, t))
  hook = TimelineHook(output_dir=str(tmp_path), start_step=1, steps=2)
  tr.hooks.append(hook)
  for _ in range(4):
    tr.step(torch.randn(8, 16), torch.randint(0, 4, (8,)))
  text = open(os.path.join(tmp_path, "kernel_table.txt")).read()
  assert "timeline: span" in text and hook.by_name and any("addmm" in k or "linear" in k or "mm" in k for k in hook.by_name)


def test_bench_reference_arm_reports_unavailable():
  """bench.py contract: the reference (TensorFlow 1.15) cannot be installed offline, so `--impl reference` prints one JSON line with
  `unavailable` and exits 0 (DESIGN.md section 5)."""
  import subprocess
  import sys
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "3"],
                     cwd=root, capture_output=True, text=True, timeout=120)
  assert r.returncode == 0
  line = json.loads(r.stdout.strip().splitlines()[-1])
  assert line["impl"] == "reference" and "unavailable" in line


@pytest.mark.parametrize("nproc,argv", [
    (2, ["train_gpt2.py", "--model", "tiny", "--batch", "2", "--seq", "32", "--steps", "2", "--stages", "2", "--micro", "2"]),
    (2, ["train_bert_pipeline.py", "--size", "tiny", "--batch", "4", "--seq", "16", "--steps", "2", "--tp", "2"]),
    (2, ["train_moe.py", "--batch", "2", "--seq", "16", "--steps", "2", "--experts", "4"]),
])
def test_examples_run_distributed_through_the_launcher(tmp_path, nproc, argv):
  """Pipeline, tensor-parallel and expert-parallel examples as real multi-process jobs (gloo) started by ``epl-launch``."""
  import subprocess
  import sys
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  cmd = [sys.executable, "-m", "easyparallellibrary_b200.utils.launcher", "--num_workers", "1", "--gpu_per_worker", str(nproc),
         "--backend", "gloo", "--log_dir", str(tmp_path), os.path.join(root, "examples", argv[0])] + argv[1:]
  env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
  r = _run_job(cmd, root, env, 400)
  logs = "".join(open(os.path.join(tmp_path, f)).read()[-1500:] for f in sorted(os.listdir(tmp_path)))
  assert r.returncode == 0 and "step 1 loss" in r.stdout, r.stdout[-1500:] + logs


def test_common_helpers():
  from easyparallellibrary_b200.utils import common
  assert common.strip_stage_prefix(common.add_stage_prefix("h.0.weight", 3)) == (3, "h.0.weight")
  assert common.strip_stage_prefix("embed.wte.weight") == (None, "embed.wte.weight")
  assert common.parse_device_string(common.device_string(2, 5)) == (2, "GPU", 5)
  with pytest.raises(ValueError):
    common.parse_device_string("cuda:0")
  assert common.gcd_many([4, 6, 10]) == 2 and common.lcm_many([2, 3, 4]) == 12


def test_phase_timer_and_roofline_helper():
  from easyparallellibrary_b200.utils.metric import PhaseTimer, fused_dp_roofline_ms

  class Obj(object):
    def work(self, x, k=1):
      return x * k

  o = Obj()
  t = PhaseTimer(o, "work", use_cuda=False)
  assert o.work(3, k=2) == 6 and o.work(1) == 1 and len(t.spans) == 2 and t.total_ms() >= 0.0
  t.reset()
  assert t.spans == []
  t.restore()
  assert o.work(2) == 2 and t.spans == []
  # GPT-2-XL on 8 GPUs: 5.45 GB per direction over the measured 770 GB/s = 7.08 ms (HBM side 1.7 ms, overlapped); 1 GPU: 30 B/param ~ 7.3 ms
  assert abs(fused_dp_roofline_ms(1557686400, 8) - 7.08) < 0.05 and abs(fused_dp_roofline_ms(1557686400, 1) - 7.30) < 0.05


def test_train_evaluate_loops_and_resume(tmp_path):
  """``epl.train`` / ``evaluate`` / ``train_and_evaluate`` (the reference's Estimator entry points, tests/estimator_test.py:95-175):
  stop at a GLOBAL step, checkpoint, resume in a fresh trainer, keep the data position across evaluation breaks."""
  def make():
    epl.init(epl.Config({"zero.level": "v1"}), init_process_group=False)
    torch.manual_seed(0)
    with epl.replicate(1):
      model = _net()
    return epl.Trainer(model, "adamw", loss_fn=lambda o, y: ((o - y) ** 2).mean(), lr=1e-2)

  g = torch.Generator().manual_seed(3)
  data = [(torch.randn(8, 8, generator=g), torch.randn(8, 1, generator=g)) for _ in range(5)]
  evald = data[:2]
  # uninterrupted run: 6 steps (wraps around the 5 batches), evaluation every 2 steps
  seen = []
  tr = make()
  tr.hooks.append(type("H", (), {"before_step": lambda s, t: None, "after_step": lambda s, t, out: seen.append(t.global_step)})())
  hist = epl.train_and_evaluate(tr, data, evald, max_steps=6, eval_every=2)
  assert [h["global_step"] for h in hist] == [2, 4, 6] and all(h["batches"] == 2 and h["loss"] > 0 for h in hist)
  assert seen == [1, 2, 3, 4, 5, 6]
  assert hist[-1]["loss"] < hist[0]["loss"]
  ref = epl.evaluate(tr, evald)["loss"]
  # interrupted run: 4 steps with a checkpoint, then a NEW trainer continues to step 6 from the checkpoint
  d = str(tmp_path / "ckpt")
  a = make()
  first = epl.train(a, data, max_steps=4, checkpoint_dir=d, save_every=2)
  assert len(first) == 4 and a.global_step == 4
  b = make()
  it = iter(data[4:] + data)                                # the data position is the caller's (a dataset with set_epoch / a sampler)
  rest = epl.train(b, it, max_steps=6, checkpoint_dir=d)
  assert len(rest) == 2 and b.global_step == 6
  assert abs(epl.evaluate(b, evald)["loss"] - ref) < 1e-6
  # evaluate with a metric function on the model output (no labels in the batch)
  acc = epl.evaluate(b, [x for x, _ in evald], metric_fn=lambda out, batch: {"mean_abs": out.abs().mean()})
  assert acc["batches"] == 2 and acc["mean_abs"] > 0


def test_learning_rate_schedules():
  """``Trainer(lr=schedule)``: the schedule is evaluated per global step, equals setting ``trainer.lr`` by hand, and resumes with
  the checkpointed step (reference: tf.train.exponential_decay in tests/multi_optimizer_test.py:59-62, BERT warm-up + decay)."""
  from easyparallellibrary_b200.runtime import lr_schedule as L
  s = L.warmup_linear_decay(1e-3, total_steps=10, warmup_steps=4)
  assert [round(s(i) / 1e-3, 4) for i in (0, 3, 4, 9, 10, 50)] == [0.25, 0.7, 0.6, 0.1, 0.0, 0.0]
  e = L.exponential_decay(0.1, 5, 0.96)
  assert abs(e(5) - 0.096) < 1e-12 and abs(L.exponential_decay(0.1, 5, 0.96, staircase=True)(9) - 0.096) < 1e-12
  c = L.warmup_cosine(1.0, 100, 10, 0.1)
  assert abs(c(9) - 1.0) < 1e-9 and abs(c(100) - 0.1) < 1e-9 and abs(c(55) - 0.55) < 1e-9 and c(4) == 0.5
  sched = L.warmup(L.exponential_decay(2e-2, 3, 0.5), 2)
  auto, tr = _run({}, steps=5, lr=sched)
  assert tr.lr_schedule is sched and abs(tr.lr - sched(4)) < 1e-12
  # the same learning rates assigned by hand
  epl.init(epl.Config({}), init_process_group=False)
  with epl.replicate(1):
    model = _net()
  tr2 = epl.Trainer(model, "adamw", loss_fn=lambda o, y: ((o - y) ** 2).mean(), lr=123.0)
  torch.manual_seed(1)
  X, Y = torch.randn(5, 8, 8), torch.randn(5, 8, 1)
  manual = []
  for i in range(5):
    tr2.lr = sched(i)
    manual.append(tr2.step(X[i], Y[i]).item())
  assert max(abs(a - b) for a, b in zip(auto, manual)) < 1e-7
  const, _ = _run({}, steps=5, lr=2e-2)
  assert max(abs(a - b) for a, b in zip(auto[2:], const[2:])) > 1e-6          # the schedule does change the trajectory


def test_weight_ema_hook_with_clipping():
  """The reference's nested optimizer (Adam -> clip_gradients_by_norm -> MovingAverageOptimizer, tests/multi_optimizer_test.py:30-36)
  as ``max_grad_norm`` + a ``WeightEMA`` hook: the shadow weights follow TF's formula and can be swapped in for evaluation."""
  from easyparallellibrary_b200.runtime.ema import WeightEMA
  epl.init(epl.Config({"communication.clip_after_allreduce": True}), init_process_group=False)
  with epl.replicate(1):
    model = _net()
  tr = epl.Trainer(model, "adam", loss_fn=lambda o, y: ((o - y) ** 2).mean(), lr=1e-2, max_grad_norm=0.5)
  ema = WeightEMA(decay=0.1, num_updates=True)
  tr.hooks.append(ema)
  torch.manual_seed(1)
  X, Y = torch.randn(4, 8, 8), torch.randn(4, 8, 1)
  p0 = next(model.parameters())
  expect = p0.detach().clone()
  for i in range(4):
    out = tr.step(X[i], Y[i])
    assert out.grad_norm is not None
    d = min(0.1, (1.0 + i) / (10.0 + i))
    expect = d * expect.to(p0.device) + (1 - d) * p0.detach()      # the trainer moved the model to its device in step 1
  name = ema._names[0]
  assert torch.allclose(ema.shadow[name], expect, atol=1e-7) and ema.updates == 4
  trained = p0.detach().clone()
  plain = tr.eval_step(X[0], Y[0]).item()
  with ema.swapped(tr):
    assert torch.allclose(p0, expect, atol=1e-7)
    averaged = tr.eval_step(X[0], Y[0]).item()
  assert torch.equal(p0.detach(), trained) and averaged != plain
  other = WeightEMA(decay=0.1, num_updates=True)
  other.load_state_dict(ema.state_dict())
  assert other.updates == 4 and torch.equal(other.shadow[name], ema.shadow[name])


def test_named_summaries_are_merged_and_written(tmp_path):
  """``epl.summary.scalar / histogram`` inside the model (reference: tf.summary under EPL, tests/summary_test.py:31-110): merged over
  the micro-batches like their collection, described in ``Graph.summary_map``, written by ``SummaryHook``."""
  import json as _json

  class Net(nn.Module):
    def __init__(self):
      super().__init__()
      self.fc = nn.Linear(8, 4)

    def forward(self, x, labels):
      logits = self.fc(x)
      epl.summary.histogram("features", x)
      epl.summary.scalar("mean_acc", (logits.argmax(-1) == labels).float().mean())
      epl.summary.scalar("rows", torch.tensor(float(x.shape[0])), reduce="sum")
      return nn.functional.cross_entropy(logits, labels)

  epl.init(epl.Config({"pipeline.num_micro_batch": 2}), init_process_group=False)
  with epl.replicate(1):
    model = Net()
  tr = epl.Trainer(model, "sgd", lr=0.1)
  hook = epl.summary.SummaryHook(str(tmp_path), every=2)
  tr.hooks.append(hook)
  torch.manual_seed(0)
  x, y = torch.randn(6, 8), torch.randint(0, 4, (6,))
  outs = [tr.step(x, y) for _ in range(4)]
  hook.close()
  smap = epl.Graph.get().summary_map
  assert sorted(smap) == ["features", "mean_acc", "rows"]
  assert smap["features"].summary_type == "SUMMARY_HISTOGRAM_TYPE" and smap["features"].collection == epl.GraphKeys.GLOBAL_CONCAT_OBJECTS
  assert smap["mean_acc"].summary_type == "SUMMARY_SCALAR_TYPE" and smap["rows"].collection == epl.GraphKeys.GLOBAL_SUM_OBJECTS
  merged = epl.summary.merged_summaries(outs[-1])
  assert merged["features"].shape == (6, 8) and float(merged["rows"]) == 6.0 and 0.0 <= float(merged["mean_acc"]) <= 1.0
  rows = [_json.loads(l) for l in open(os.path.join(tmp_path, "summaries.jsonl"))]
  assert [r["step"] for r in rows] == [2, 4] and rows[0]["rows"] == 6.0 and rows[0]["features"]["count"] == 48
  assert all(k in rows[1] for k in ("loss", "lr", "loss_scale", "mean_acc"))
  assert any(f.startswith("events.out.tfevents") for f in os.listdir(tmp_path))      # TensorBoard events next to the JSON lines


@pytest.mark.parametrize("cls,kw", [(torch.optim.Adagrad, {}), (torch.optim.RMSprop, {"momentum": 0.5}), (torch.optim.Adam, {"amsgrad": True})])
def test_any_torch_optimizer_class(cls, kw, tmp_path):
  """``Trainer(model, torch.optim.X, ...)``: the reference accepts whatever TF optimizer the model uses; here any torch optimizer
  class runs on the fp32 master shards and must match the same optimizer on a plain model — also with ZeRO-1, gradient
  accumulation, a learning-rate schedule, no-decay parameters and a checkpoint round trip."""
  from easyparallellibrary_b200.runtime import lr_schedule as L, saver
  sched = L.exponential_decay(1e-2, 2, 0.5)
  torch.manual_seed(0)
  ref_model = _net()
  decay = [p for p in ref_model.parameters() if p.dim() > 1]
  nodecay = [p for p in ref_model.parameters() if p.dim() <= 1]
  ref_opt = cls([{"params": decay, "weight_decay": 0.1}, {"params": nodecay, "weight_decay": 0.0}], lr=1e-2, **kw)
  torch.manual_seed(1)
  X, Y = torch.randn(5, 8, 8), torch.randn(5, 8, 1)
  ref = []
  for i in range(5):
    for g in ref_opt.param_groups:
      g["lr"] = sched(i)
    ref_opt.zero_grad()
    loss = ((ref_model(X[i]) - Y[i]) ** 2).mean()
    loss.backward()
    ref_opt.step()
    ref.append(loss.item())

  def make(conf):
    epl.init(epl.Config(conf), init_process_group=False)
    torch.manual_seed(0)
    with epl.replicate(1):
      model = _net()
    return epl.Trainer(model, cls, loss_fn=lambda o, y: ((o - y) ** 2).mean(), lr=sched, weight_decay=0.1, **kw)

  for conf in ({}, {"zero.level": "v1"}, {"pipeline.num_micro_batch": 2}):
    tr = make(conf)
    got = [tr.step(X[i], Y[i]).item() for i in range(5)]
    assert max(abs(a - b) for a, b in zip(got, ref)) < 2e-6, (conf, got, ref)
  a = make({})
  for i in range(3):
    a.step(X[i], Y[i])
  saver.save_checkpoint(a, str(tmp_path))
  b = make({})
  assert saver.load_checkpoint(b, str(tmp_path)) == 3
  assert abs(b.step(X[3], Y[3]).item() - ref[3]) < 2e-6 and abs(b.step(X[4], Y[4]).item() - ref[4]) < 2e-6
  with pytest.raises(ValueError):
    make({"offload.level": "v0"}).build()


def test_torch_optimizer_instance_is_taken_over():
  """``Trainer(model, torch.optim.X(model.parameters(), ...))``: class, defaults and the groups' weight-decay split are taken over."""
  torch.manual_seed(0)
  ref_model = _net()
  ref_opt = torch.optim.RMSprop(ref_model.parameters(), lr=3e-3, alpha=0.9, weight_decay=0.05)      # decays biases too
  torch.manual_seed(1)
  X, Y = torch.randn(4, 8, 8), torch.randn(4, 8, 1)
  ref = []
  for i in range(4):
    ref_opt.zero_grad()
    loss = ((ref_model(X[i]) - Y[i]) ** 2).mean()
    loss.backward()
    ref_opt.step()
    ref.append(loss.item())
  epl.init(epl.Config({}), init_process_group=False)
  torch.manual_seed(0)
  with epl.replicate(1):
    model = _net()
  decay = [p for p in model.parameters() if p.dim() > 1]
  inst = torch.optim.RMSprop(model.parameters(), lr=3e-3, alpha=0.9, weight_decay=0.05)
  tr = epl.Trainer(model, inst, loss_fn=lambda o, y: ((o - y) ** 2).mean())
  assert tr.opt_kind == "torch" and tr.hyper.factory is torch.optim.RMSprop and tr.hyper.kwargs["alpha"] == 0.9 and tr.lr == 3e-3
  got = [tr.step(X[i], Y[i]).item() for i in range(4)]
  assert max(abs(a - b) for a, b in zip(got, ref)) < 2e-6
  # two groups: the zero-weight-decay group becomes the no-decay set
  epl.init(epl.Config({}), init_process_group=False)
  torch.manual_seed(0)
  with epl.replicate(1):
    model = _net()
  decay = [p for p in model.parameters() if p.dim() > 1]
  rest = [p for p in model.parameters() if p.dim() <= 1]
  inst = torch.optim.SGD([{"params": decay, "weight_decay": 0.1}, {"params": rest, "weight_decay": 0.0}], lr=1e-2, momentum=0.9)
  tr = epl.Trainer(model, inst, loss_fn=lambda o, y: ((o - y) ** 2).mean())
  assert tr.hyper.weight_decay == 0.1 and all(tr.no_decay(p) for p in rest) and not any(tr.no_decay(p) for p in decay)
  tr.step(X[0], Y[0])


def test_fix_randomness_makes_runs_repeatable():
  from easyparallellibrary_b200.utils.common import fix_randomness

  def run():
    fix_randomness(7)
    epl.init(epl.Config({}), init_process_group=False)
    with epl.replicate(1):
      model = nn.Sequential(nn.Linear(8, 16), nn.Dropout(0.5), nn.Linear(16, 1))      # unseeded init AND dropout
    tr = epl.Trainer(model, "adamw", loss_fn=lambda o, y: ((o - y) ** 2).mean(), lr=1e-2)
    return [tr.step(torch.randn(4, 8), torch.randn(4, 1)).item() for _ in range(3)]

  try:
    assert run() == run()
  finally:
    fix_randomness(0, deterministic=False)
