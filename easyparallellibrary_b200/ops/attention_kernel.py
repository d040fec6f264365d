"""Autograd wrapper of the tcgen05 flash-attention kernels (``csrc/attention.cu``).

``flash_attention_packed(qkv, causal)`` takes the fused QKV projection output ``[B, S, 3, H, 64]`` and returns
``[B, S, H*64]`` — the exact layouts of the neighbouring GEMMs, so no permute / contiguous / cat kernels run
around attention in either direction (the gradient comes back packed as ``[B, S, 3, H, 64]`` too).

``kv_len`` (optional, int32 ``[B]`` on the same device) limits batch row ``b`` to keys ``[0, kv_len[b])``: key padding.
The lengths are read by the kernels only (no host sync, so the call can be captured in a CUDA graph and the tensor's contents
refreshed between replays) and clamped to ``[1, S]``.  Padded Q/K/V rows may hold any finite values.
"""
from __future__ import annotations

import ctypes
import math

import torch

from easyparallellibrary_b200.ops import _lib

_ready = [False]


def _lib_attn():
  lib = _lib.require()
  if not _ready[0]:
    p, i, f = ctypes.c_void_p, ctypes.c_int, ctypes.c_float
    lib.epl_attn_fwd.argtypes = [p, p, p, i, i, i, f, i, p]
    lib.epl_attn_bwd.argtypes = [p, p, p, p, p, p, p, i, i, i, f, i, p]
    lib.epl_attn_fwd_len.argtypes = [p, p, p, i, i, i, f, i, p, p]
    lib.epl_attn_bwd_len.argtypes = [p, p, p, p, p, p, p, i, i, i, f, i, p, p]
    lib.epl_attn_dq_slots.argtypes = [i]
    _ready[0] = True
  return lib


def supported_packed(qkv: torch.Tensor) -> bool:
  return (qkv.is_cuda and qkv.dtype == torch.bfloat16 and qkv.dim() == 5 and qkv.shape[2] == 3 and qkv.shape[4] == 64
          and qkv.is_contiguous() and qkv.data_ptr() % 16 == 0)


class _FlashPacked(torch.autograd.Function):
  @staticmethod
  def forward(ctx, qkv, causal, kv_len):
    lib = _lib_attn()
    B, S, _, H, D = qkv.shape
    out = torch.empty((B, S, H, D), dtype=qkv.dtype, device=qkv.device)
    lse = torch.empty((B, H, S), dtype=torch.float32, device=qkv.device)
    scale = 1.0 / math.sqrt(D)
    rc = lib.epl_attn_fwd_len(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), B, S, H, scale, int(causal), _lib.stream(),
                              _len_ptr(kv_len))
    _lib.check(rc, "attn_fwd")
    ctx.save_for_backward(qkv, out, lse, kv_len)
    ctx.causal, ctx.scale = causal, scale
    return out.view(B, S, H * D)

  @staticmethod
  def backward(ctx, d_out):
    lib = _lib_attn()
    qkv, out, lse, kv_len = ctx.saved_tensors
    B, S, _, H, D = qkv.shape
    d_out = d_out.contiguous()
    dqkv = torch.empty_like(qkv)
    delta = torch.empty((B, H, S), dtype=torch.float32, device=qkv.device)
    dq_acc = torch.empty((lib.epl_attn_dq_slots(S), B, S, H, D), dtype=torch.float32, device=qkv.device)  # see csrc/attention.cu
    rc = lib.epl_attn_bwd_len(qkv.data_ptr(), out.data_ptr(), d_out.data_ptr(), lse.data_ptr(), delta.data_ptr(), dq_acc.data_ptr(),
                              dqkv.data_ptr(), B, S, H, ctx.scale, int(ctx.causal), _lib.stream(), _len_ptr(kv_len))
    _lib.check(rc, "attn_bwd")
    _lib.launches += 3
    return dqkv, None, None


def _len_ptr(kv_len):
  return None if kv_len is None else kv_len.data_ptr()


def check_kv_len(qkv: torch.Tensor, kv_len: torch.Tensor) -> None:
  B = qkv.shape[0]
  if not (isinstance(kv_len, torch.Tensor) and kv_len.dtype == torch.int32 and kv_len.is_cuda and kv_len.device == qkv.device
          and kv_len.dim() == 1 and kv_len.shape[0] == B and kv_len.is_contiguous()):
    raise ValueError("kv_len must be a contiguous int32 tensor of shape [%d] on %s (got %s)" % (
        B, qkv.device, "%s %s %s" % (tuple(kv_len.shape), kv_len.dtype, kv_len.device) if isinstance(kv_len, torch.Tensor)
        else type(kv_len).__name__))


def flash_attention_packed(qkv: torch.Tensor, causal: bool = True, kv_len: torch.Tensor = None) -> torch.Tensor:
  if kv_len is not None:
    check_kv_len(qkv, kv_len)
  return _FlashPacked.apply(qkv, causal, kv_len)
