"""Small shared helpers (reference ``epl/utils/common.py``).

The reference's name codecs encode the replica / micro-batch clone of an op into its *name*
(``EPL_REPLICA_<i>/`` and ``EPL_MICRO_BATCH_<j>/`` prefixes, ``common.py:108-153``).  Nothing is cloned here, so the only
names that need a codec are checkpoint keys: a parameter of pipeline stage ``s`` is stored as ``stage<s>.<name>``
(``runtime/saver.py``).  Device strings follow the reference's ``/job:worker/replica:0/task:<w>/device:GPU:<g>`` form so
logs and ``Cluster`` dumps read the same.
"""
from __future__ import annotations

import math
import re
from functools import reduce
from typing import Iterable, Optional, Tuple

_STAGE_RE = re.compile(r"^stage(\d+)\.(.*)$")
_DEVICE_RE = re.compile(r"^/job:worker/replica:0/task:(\d+)/device:(GPU|CPU):(\d+)$")


def add_stage_prefix(name: str, stage: int) -> str:
  return "stage%d.%s" % (stage, name)


def strip_stage_prefix(key: str) -> Tuple[Optional[int], str]:
  """``'stage3.h.0.weight'`` -> ``(3, 'h.0.weight')``; keys without a prefix -> ``(None, key)``."""
  m = _STAGE_RE.match(key)
  return (int(m.group(1)), m.group(2)) if m else (None, key)


def device_string(worker: int, index: int, kind: str = "GPU") -> str:
  return "/job:worker/replica:0/task:%d/device:%s:%d" % (worker, kind, index)


def parse_device_string(dev: str) -> Tuple[int, str, int]:
  """-> (worker index, 'GPU' | 'CPU', device index)."""
  m = _DEVICE_RE.match(dev)
  if not m:
    raise ValueError("not an EPL device string: %r" % dev)
  return int(m.group(1)), m.group(2), int(m.group(3))


def gcd_many(values: Iterable[int]) -> int:
  return reduce(math.gcd, values, 0)


def lcm_many(values: Iterable[int]) -> int:
  return reduce(lambda a, b: a * b // math.gcd(a, b) if a and b else 0, values, 1)


def fix_randomness(seed: int = 0, deterministic: bool = True) -> None:
  """Seed every generator and ask the libraries for deterministic algorithms — what the reference's A/B tests do before comparing
  two runs to 1e-5 / 1e-6 (``tests/test_utils.py:25-33``: seeds + ``TF_DETERMINISTIC_OPS``).  Call it before building the model.

  The in-tree kernels are deterministic for a fixed launch configuration except where partial results meet in memory in arrival
  order: bf16 weight-gradient accumulation across micro-batches; runs then agree to rounding, not bit for bit.  (The dQ
  accumulation of the attention backward and the bias-gradient column sums are reproducible bit for bit.)"""
  import os
  import random
  import numpy as np
  import torch
  random.seed(seed)
  np.random.seed(seed % (2 ** 32))
  torch.manual_seed(seed)
  if torch.cuda.is_available():
    torch.cuda.manual_seed_all(seed)
  if deterministic:
    os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False
    torch.use_deterministic_algorithms(True, warn_only=True)
  else:
    torch.use_deterministic_algorithms(False)
