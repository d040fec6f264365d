"""Causal / bidirectional multi-head attention.

``attention_packed(qkv, causal, kv_len)`` takes the fused QKV projection output ``[B, S, 3, H, D]``.  On sm_100a it runs the
hand-written flash-style kernels in ``csrc/attention.cu`` (bf16, head dim 64); the ``torch`` SDPA call is the numerics
reference and the CPU path.  ``attention(q, k, v, causal, kv_len=...)`` takes ``[B, H, S, D]`` tensors and runs SDPA.

``kv_len`` (int32 ``[B]``, optional) is a key-padding length per batch row: row ``b`` attends to keys ``[0, kv_len[b])`` only,
and with ``causal`` key ``j`` is visible to query ``i`` iff ``j < kv_len[b]`` and ``j <= i``.  Query rows at padded positions
are still computed (over the valid keys).  Lengths are clamped to ``[1, S]`` on every path.
"""
from __future__ import annotations

import math

import torch

from easyparallellibrary_b200.ops import _lib

import os

# "auto" | "epl" | "sdpa".  auto: the hand-written tcgen05 kernel whenever it supports the input (bf16, head dim 64 —
# measured faster end to end than the cuDNN path on GPT-2-XL because it consumes the packed QKV layout directly),
# else torch SDPA.  EPL_ATTENTION=epl makes an unsupported input an error, =sdpa forces the library path.
_IMPL = os.environ.get("EPL_ATTENTION", "auto")


def key_padding_mask(kv_len: torch.Tensor, S: int, causal: bool, device=None) -> torch.Tensor:
  """Boolean ``[B, 1, S, S]`` SDPA mask (True = attend) of key lengths ``kv_len`` (clamped to ``[1, S]``, like the kernels)."""
  keys = torch.arange(S, device=device if device is not None else kv_len.device)
  lens = kv_len.to(keys.device).long().clamp(1, S)
  mask = (keys < lens[:, None])[:, None, None, :]
  if causal:
    mask = mask & torch.ones(S, S, dtype=torch.bool, device=keys.device).tril()
  return mask


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, causal: bool = True, dropout_p: float = 0.0,
              kv_len: torch.Tensor = None) -> torch.Tensor:
  """``[B, H, S, D]`` q, k, v -> ``[B, H, S, D]``.  The hand-written kernel takes the packed layout only (``attention_packed``),
  so this is the SDPA path on every device (an error under ``EPL_ATTENTION=epl``)."""
  if _IMPL == "epl" and q.is_cuda:
    raise RuntimeError("EPL_ATTENTION=epl: the hand-written attention kernel takes the packed [B, S, 3, H, 64] layout "
                       "(attention_packed), not separate q, k, v")
  if kv_len is None:
    return torch.nn.functional.scaled_dot_product_attention(q, k, v, is_causal=causal, dropout_p=dropout_p)
  mask = key_padding_mask(kv_len, k.shape[-2], causal, device=q.device)
  return torch.nn.functional.scaled_dot_product_attention(q, k, v, attn_mask=mask, dropout_p=dropout_p)


def attention_packed(qkv: torch.Tensor, causal: bool = True, kv_len: torch.Tensor = None) -> torch.Tensor:
  """``qkv``: ``[B, S, 3, H, D]`` (output of a fused QKV projection) -> ``[B, S, H*D]``.  ``kv_len``: key lengths, see above."""
  from easyparallellibrary_b200.runtime import amp
  if amp.o1_active():
    qkv = amp.cast_args("attention", qkv)
  if _IMPL != "sdpa" and qkv.is_cuda:
    from easyparallellibrary_b200.ops import attention_kernel
    if attention_kernel.supported_packed(qkv):
      return attention_kernel.flash_attention_packed(qkv, causal, kv_len)
    if _IMPL == "epl":
      raise RuntimeError("hand-written attention kernel does not support this input (needs bf16, head dim 64, contiguous; "
                         "optional key lengths as int32 [B] on the same device)")
  B, S, _, H, D = qkv.shape
  q, k, v = qkv.permute(2, 0, 3, 1, 4).unbind(0)
  if kv_len is None:
    y = torch.nn.functional.scaled_dot_product_attention(q, k, v, is_causal=causal)
  else:
    y = torch.nn.functional.scaled_dot_product_attention(q, k, v, attn_mask=key_padding_mask(kv_len, S, causal, device=qkv.device))
  return y.transpose(1, 2).reshape(B, S, H * D)


def attention_reference(q, k, v, causal: bool = True, kv_len=None) -> torch.Tensor:
  """Plain fp32 softmax(QK^T)V — the numerics reference for kernel tests."""
  qf, kf, vf = q.float(), k.float(), v.float()
  s = qf @ kf.transpose(-1, -2) / math.sqrt(q.shape[-1])
  if causal:
    S, T = s.shape[-2:]
    mask = torch.ones(S, T, dtype=torch.bool, device=q.device).tril(T - S)
    s = s.masked_fill(~mask, float("-inf"))
  if kv_len is not None:
    T = s.shape[-1]
    keys = torch.arange(T, device=q.device)
    s = s.masked_fill(~(keys < kv_len.to(q.device).long().clamp(1, T)[:, None])[:, None, None, :], float("-inf"))
  return (torch.softmax(s, -1) @ vf).to(q.dtype)
