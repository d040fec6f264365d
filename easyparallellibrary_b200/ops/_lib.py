"""ctypes bindings for ``lib/libepl_kernels.so``.

On a machine with a GPU a missing library is a hard error (``require()``): the
CUDA path must be the one that runs, never a silent eager fallback.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB_PATH = os.path.join(_HERE, "lib", "libepl_kernels.so")
_lib: Optional[ctypes.CDLL] = None
launches = 0          # number of EPL kernel launches issued by this process (bench.py reports it)

F32, BF16, F16 = 0, 1, 2
_DT = {torch.float32: F32, torch.bfloat16: BF16, torch.float16: F16}


def dtype_code(dt: torch.dtype) -> int:
  try:
    return _DT[dt]
  except KeyError:
    raise TypeError("unsupported dtype %s (float32 / bfloat16 / float16)" % dt)


def available() -> bool:
  return os.path.exists(_LIB_PATH)


def require() -> ctypes.CDLL:
  global _lib
  if _lib is None:
    if not os.path.exists(_LIB_PATH):
      try:
        from easyparallellibrary_b200.build import build_all
        build_all()
      except Exception as e:
        raise RuntimeError("EPL-B200 native kernels are not built (%s missing) and building failed: %s. "
                           "Run `python -m easyparallellibrary_b200.build`." % (_LIB_PATH, e))
    _lib = ctypes.CDLL(_LIB_PATH)
    for name in dir(_Sigs):
      if name.startswith("epl_"):
        fn = getattr(_lib, name)
        fn.restype = ctypes.c_int
        fn.argtypes = getattr(_Sigs, name)
  return _lib


_p, _i, _l, _f = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float


class _Sigs:
  epl_adamw = [_p, _p, _i, _p, _p, _p, _i, _p, _l, _f, _f, _f, _f, _f, _f, _f, _f, _p]
  epl_adamw_dyn = [_p, _p, _i, _p, _p, _p, _i, _p, _l, _p, _f, _f, _f, _f, _p]
  epl_sgd = [_p, _p, _i, _p, _p, _i, _l, _f, _f, _f, _f, _p]
  epl_sumsq = [_p, _i, _l, _p, _p]
  epl_norm_fwd = [_p, _p, _p, _p, _p, _p, _i, _i, _f, _i, _i, _p]
  epl_norm_bwd_grid = [_i]
  epl_norm_bwd = [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p]
  epl_bias_gelu_fwd = [_p, _p, _p, _p, _l, _i, _i, _p]
  epl_gelu_bwd = [_p, _p, _p, _l, _i, _p]
  epl_colsum = [_p, _p, _p, _i, _i, _i, _i, _p]
  epl_colsum_parts = [_i, _i, _i]
  epl_add = [_p, _p, _p, _l, _i, _p]
  epl_xent = [_p, _p, _p, _p, _p, _p, _i, _i, _i, _f, _l, _i, _i, _i, _p]
  epl_scale_by_device_scalar = [_p, _p, _l, _i, _p]
  epl_gemm_fp8 = [_p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p, _p, _i, _i, _f, _p, _p, _i, _p]
  epl_quantize_e4m3 = [_p, _i, _l, _p, _p, _p, _p]
  epl_gemm = [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p, _i, _i, _i, _f, _i, _i, _i, _p]


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
  return None if t is None else t.data_ptr()


def stream() -> int:
  return torch.cuda.current_stream().cuda_stream


def check(rc: int, what: str) -> None:
  global launches
  launches += 1
  if rc != 0:
    raise RuntimeError("EPL kernel %s failed with code %d (%s)" % (what, rc, _err(rc)))


def _err(rc: int) -> str:
  if rc > 0:
    try:
      return torch.cuda.cudart().cudaGetErrorString(rc)  # type: ignore[attr-defined]
    except Exception:
      return "cuda error"
  return {-1: "bad dtype combination", -2: "row too long", -3: "row does not fit shared memory",
          -10: "cuTensorMapEncodeTiled unavailable", -11: "tensor map encode failed"}.get(rc, "?")
