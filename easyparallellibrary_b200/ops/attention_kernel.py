"""Autograd wrapper of the tcgen05 flash-attention kernels (``csrc/attention.cu``).

``flash_attention_packed(qkv, causal)`` takes the fused QKV projection output ``[B, S, 3, H, 64]`` and returns
``[B, S, H*64]`` — the exact layouts of the neighbouring GEMMs, so no permute / contiguous / cat kernels run
around attention in either direction (the gradient comes back packed as ``[B, S, 3, H, 64]`` too).
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
    lib.epl_attn_dq_slots.argtypes = [i]
    _ready[0] = True
  return lib


def supported_packed(qkv: torch.Tensor) -> bool:
  return (qkv.is_cuda and qkv.dtype == torch.bfloat16 and qkv.dim() == 5 and qkv.shape[2] == 3 and qkv.shape[4] == 64
          and qkv.is_contiguous() and qkv.data_ptr() % 16 == 0)


class _FlashPacked(torch.autograd.Function):
  @staticmethod
  def forward(ctx, qkv, causal):
    lib = _lib_attn()
    B, S, _, H, D = qkv.shape
    out = torch.empty((B, S, H, D), dtype=qkv.dtype, device=qkv.device)
    lse = torch.empty((B, H, S), dtype=torch.float32, device=qkv.device)
    scale = 1.0 / math.sqrt(D)
    rc = lib.epl_attn_fwd(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), B, S, H, scale, int(causal), _lib.stream())
    _lib.check(rc, "attn_fwd")
    ctx.save_for_backward(qkv, out, lse)
    ctx.causal, ctx.scale = causal, scale
    return out.view(B, S, H * D)

  @staticmethod
  def backward(ctx, d_out):
    lib = _lib_attn()
    qkv, out, lse = ctx.saved_tensors
    B, S, _, H, D = qkv.shape
    d_out = d_out.contiguous()
    dqkv = torch.empty_like(qkv)
    delta = torch.empty((B, H, S), dtype=torch.float32, device=qkv.device)
    dq_acc = torch.empty((lib.epl_attn_dq_slots(S), B, S, H, D), dtype=torch.float32, device=qkv.device)  # see csrc/attention.cu
    rc = lib.epl_attn_bwd(qkv.data_ptr(), out.data_ptr(), d_out.data_ptr(), lse.data_ptr(), delta.data_ptr(), dq_acc.data_ptr(),
                          dqkv.data_ptr(), B, S, H, ctx.scale, int(ctx.causal), _lib.stream())
    _lib.check(rc, "attn_bwd")
    _lib.launches += 3
    return dqkv, None


def flash_attention_packed(qkv: torch.Tensor, causal: bool = True) -> torch.Tensor:
  return _FlashPacked.apply(qkv, causal)
