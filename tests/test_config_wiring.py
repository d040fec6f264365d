"""Every config key must change behaviour: one test per key that used to parse and do nothing (round-1 verdict), plus a
static coverage test that fails when a key of the schema has no reader in the package."""
import os
import re

import numpy as np
import pytest
import torch
from torch import nn

import easyparallellibrary_b200 as epl
from easyparallellibrary_b200.config import Config
from dist_utils import run_distributed

PKG = os.path.join(os.path.dirname(__file__), "..", "easyparallellibrary_b200")


def test_every_config_key_has_a_reader():
  """``config.<group>.<attr>`` (or ``cfg.<group>.<attr>`` / ``<group>_cfg.<attr>``) must be read somewhere outside config.py."""
  src = {}
  for root, _, files in os.walk(PKG):
    for f in files:
      if f.endswith(".py") and f != "config.py":
        src[os.path.join(root, f)] = open(os.path.join(root, f)).read()
  blob = "\n".join(src.values())
  missing = []
  for key, _default, _help in Config.describe():
    group, attr = key.split(".")
    pat = re.compile(r"\b%s\.%s\b" % (re.escape(group), re.escape(attr)))
    alt = re.compile(r"\b(ccfg|cfg|c)\.%s\b" % re.escape(attr))      # a group bound to a local (cfg = env.config.communication)
    if not pat.search(blob) and not alt.search(blob):
      missing.append(key)
  assert not missing, "config keys nobody reads: %s" % missing


# ------------------------------------------------------------------------------------------------ communication.fp16
def _fp32_dp(rank, world, conf):
  epl.init(epl.Config(conf))
  torch.manual_seed(0)
  with epl.replicate(1):
    model = nn.Sequential(nn.Linear(12, 32), nn.Tanh(), nn.Linear(32, 1))
  tr = epl.Trainer(model, "sgd", lr=0.05, loss_fn=lambda o, y: ((o - y) ** 2).mean())
  g = torch.Generator().manual_seed(5 + rank)
  kinds = set()
  orig = tr.build()._launch_bucket_reduce

  def spy(s, b):
    orig(s, b)
    kinds.add(type(tr._pending[-1][2]).__name__)
  tr._launch_bucket_reduce = spy
  for _ in range(3):
    tr.step(torch.randn(8, 12, generator=g) * 3, torch.randn(8, 1, generator=g))
  return [p.detach().numpy().copy() for p in model.parameters()], sorted(kinds)


def test_fp16_wire_compression_is_on_the_gradient_path():
  plain = run_distributed(_fp32_dp, 2, args=({},))
  comp = run_distributed(_fp32_dp, 2, args=({"communication.fp16": True, "communication.fp16_scale": 128},))
  assert "_Decompress" in comp[0][1] and "_Decompress" not in plain[0][1]
  d = max(float(np.abs(a - b).max()) for a, b in zip(plain[0][0], comp[0][0]))
  assert 0.0 < d < 5e-3                                     # half precision on the wire: close, not identical
  assert all(np.array_equal(a, b) for a, b in zip(comp[0][0], comp[1][0]))


# ------------------------------------------------------------------------------------------------ sparse gradients
class _Emb(nn.Module):
  def __init__(self, sparse=True):
    super().__init__()
    self.e = nn.Embedding(64, 8, sparse=sparse)
    self.l = nn.Linear(8, 1)

  def forward(self, idx, y):
    return ((self.l(self.e(idx).mean(1)) - y) ** 2).mean()


def _sparse_dp(rank, world, conf, sparse=True):
  epl.init(epl.Config(conf))
  torch.manual_seed(0)
  with epl.replicate(1):
    model = _Emb(sparse)
  tr = epl.Trainer(model, "sgd", lr=0.1).build()
  g = torch.Generator().manual_seed(3)
  for _ in range(3):
    idx, y = torch.randint(0, 64, (8, 4), generator=g), torch.randn(8, 1, generator=g)
    if world > 1:
      idx, y = idx.chunk(world)[rank], y.chunk(world)[rank]
    tr.step(idx, y)
  return [p.detach().numpy().copy() for p in model.parameters()], getattr(tr, "sparse_wire_elems", 0), len(tr._sparse)


def test_sparse_gradients_travel_as_indices_and_values():
  dense1 = run_distributed(_sparse_dp, 1, args=({}, False))[0]
  sp2 = run_distributed(_sparse_dp, 2, args=({},))
  as_dense = run_distributed(_sparse_dp, 2, args=({"communication.sparse_as_dense": True},))
  for res in (sp2, as_dense):
    assert res[0][2] == 1                                    # the embedding table is kept out of the dense buckets
    assert max(float(np.abs(a - b).max()) for a, b in zip(dense1[0], res[0][0])) < 1e-6
  assert sp2[0][1] > 0 and sp2[0][1] < 3 * 64 * 8            # rows touched, not the whole table, crossed the wire
  assert as_dense[0][1] == 0                                 # communication.sparse_as_dense: densified before the reduction


# ------------------------------------------------------------------------------------------------ io.*
def test_io_slicing_keys_drive_the_sharded_dataset():
  from easyparallellibrary_b200.utils.dataset import ShardedFileDataset, shard_files, synthetic_token_files
  files = list(range(10))
  off = Config({})
  assert shard_files(files, config=off, replicas_per_worker=[1, 1, 1], worker_index=1) == files          # io.slicing off: everything
  on = Config({"io.slicing": True, "io.unbalanced_io_slicing": True})
  parts = [shard_files(files, config=on, replicas_per_worker=[1, 1, 1], worker_index=w) for w in range(3)]
  assert sorted(sum(parts, [])) == files and [len(p) for p in parts] == [4, 3, 3]
  drop = Config({"io.slicing": True, "io.drop_last_files": True})
  parts = [shard_files(files, config=drop, replicas_per_worker=[1, 1, 1], worker_index=w) for w in range(3)]
  assert [len(p) for p in parts] == [3, 3, 3]
  fl, reader = synthetic_token_files(6, 2, 5, 100)
  ds = ShardedFileDataset(fl, reader, config=Config({"io.slicing": True}))       # single process: one replica -> all files
  assert len(list(ds)) == 12 and list(ds)[0].shape == (5,)


def _sliced_files(rank, world):
  epl.init(epl.Config({"io.slicing": True}))
  with epl.replicate(1):
    model = nn.Linear(4, 1)
  epl.Trainer(model, "sgd", lr=0.1).build()
  from easyparallellibrary_b200.utils.dataset import shard_files
  return shard_files(list(range(8)))


def test_io_slicing_follows_the_parallel_plan():
  parts = run_distributed(_sliced_files, 2)
  assert parts[0] == [0, 1, 2, 3] and parts[1] == [4, 5, 6, 7]


# ------------------------------------------------------------------------------------------------ amp.level = O1
class _TinyLM(nn.Module):
  def __init__(self):
    super().__init__()
    from easyparallellibrary_b200.ops.layernorm import LayerNorm
    from easyparallellibrary_b200.ops.linear import Linear
    self.fc, self.ln, self.out = Linear(16, 32), LayerNorm(32), Linear(32, 4)
    self.seen = []

  def forward(self, x, y):
    h = self.fc(x)
    self.seen.append(("linear", h.dtype))
    h = self.ln(torch.nn.functional.gelu(h))
    self.seen.append(("layer_norm", h.dtype))
    logits = self.out(h)
    from easyparallellibrary_b200.ops.cross_entropy import softmax_cross_entropy
    return softmax_cross_entropy(logits, y)


def test_amp_o1_is_an_op_level_policy_with_fp32_master_weights():
  from easyparallellibrary_b200.runtime import amp
  losses = {}
  for level in ("", "O1"):
    epl.init(epl.Config({"amp.level": level, "amp.loss_scale": 128}), init_process_group=False)
    torch.manual_seed(0)
    with epl.replicate(1):
      model = _TinyLM()
    tr = epl.Trainer(model, "adamw", lr=1e-2)
    g = torch.Generator().manual_seed(1)
    x, y = torch.randn(8, 16, generator=g), torch.randint(0, 4, (8,), generator=g)
    losses[level] = [tr.step(x, y).item() for _ in range(4)]
    assert all(p.dtype == torch.float32 for p in model.parameters())          # O1 never casts the variables themselves
    if level == "O1":
      assert ("linear", torch.float16) in model.seen and ("layer_norm", torch.float32) in model.seen
      assert tr.scaler.loss_scale == 128.0
  assert not amp.o1_active() and amp.op_dtype("linear") is None
  with amp.o1_autocast("cpu"):
    assert amp.op_dtype("linear") == torch.float16 and amp.op_dtype("layer_norm") == torch.float32 and amp.op_dtype("add") is None
  assert max(abs(a - b) for a, b in zip(losses[""], losses["O1"])) < 2e-2
  assert losses["O1"][-1] < losses["O1"][0]


# ------------------------------------------------------------------------------------------------ gradient_checkpoint.check_gradients
class _Impure(nn.Module):
  """A block whose output depends on how often it ran: recomputation changes the gradient."""

  def __init__(self):
    super().__init__()
    self.l = nn.Linear(6, 6)
    self.calls = 0

  def forward(self, x):
    self.calls += 1
    return self.l(x) * float(self.calls)


def _gc_model(impure):
  torch.manual_seed(0)
  blocks = [(_Impure() if impure and i == 1 else nn.Sequential(nn.Linear(6, 6), nn.Tanh())) for i in range(4)]
  return nn.Sequential(*blocks, nn.Linear(6, 1))


def test_check_gradients_flag_validates_recompute():
  conf = {"gradient_checkpoint.type": "auto", "gradient_checkpoint.check_gradients": True}
  epl.init(epl.Config(conf), init_process_group=False)
  with epl.replicate(1):
    model = _gc_model(False)
  tr = epl.Trainer(model, "sgd", lr=0.1, loss_fn=lambda o, y: ((o - y) ** 2).mean())
  x, y = torch.randn(4, 6), torch.randn(4, 1)
  tr.step(x, y)
  assert tr.gc_check_result < 1e-5
  epl.init(epl.Config(conf), init_process_group=False)
  with epl.replicate(1):
    model = _gc_model(True)
  tr = epl.Trainer(model, "sgd", lr=0.1, loss_fn=lambda o, y: ((o - y) ** 2).mean())
  with pytest.raises(RuntimeError, match="check_gradients"):
    tr.step(x, y)


# ------------------------------------------------------------------------------------------------ cluster.run_visible_devices
def test_run_visible_devices_is_exported_before_cuda_starts():
  """Checked in a fresh interpreter: on a machine with a GPU, earlier tests of this process have already started CUDA."""
  import subprocess
  import sys
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  code = ("import os\nimport easyparallellibrary_b200 as epl\n"
          "epl.init(epl.Config({'cluster.run_visible_devices': '2,3'}), init_process_group=False)\n"
          "print(os.environ.get('CUDA_VISIBLE_DEVICES'))\n")
  env = {k: v for k, v in os.environ.items() if k != "CUDA_VISIBLE_DEVICES"}
  env["PYTHONPATH"] = root + os.pathsep + env.get("PYTHONPATH", "")
  r = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=300)
  assert r.returncode == 0 and r.stdout.split()[-1:] == ["2,3"], r.stdout[-2000:] + r.stderr[-2000:]
