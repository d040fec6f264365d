"""Linear layers on the hand-written tcgen05 GEMM (``csrc/gemm_tcgen05.cu``).

Forward ``y = x @ W^T (+b) (GELU)`` is one kernel (bias / GELU in the TMEM
epilogue).  Backward uses the same kernel with MN-major operand descriptors, so
no transposed copies are ever materialised:

* ``dX = dY @ W``            A = dY (K-major), B = W viewed as [contraction=N, out=K] (MN-major);
* ``dW = dY^T @ X``          A = dY viewed as [contraction=M, out=N] (MN-major), B = X (MN-major);
* the MLP block fuses ``* gelu'(pre)`` into the epilogue of the ``dH`` GEMM.

On CPU (tests, planning) everything routes to ``torch.nn.functional``.
"""
from __future__ import annotations

import math
from typing import Optional

import os

import torch
from torch import nn

from easyparallellibrary_b200.ops import _lib

EPI_NONE, EPI_BIAS, EPI_BIAS_GELU, EPI_DGELU, EPI_BIAS_RESIDUAL = range(5)
_FORCE_BN = 0            # test hook: force a tile width (128 / 160 / 256)
_NUM_SMS = 0             # 0 = all; the overlap engine lowers this to leave SMs for a concurrent collective kernel


def gemm_supported(a: torch.Tensor, b: torch.Tensor) -> bool:
  return (a.is_cuda and a.dtype in (torch.bfloat16, torch.float16) and b.dtype == a.dtype
          and a.dim() == 2 and b.dim() == 2 and a.stride(1) == 1 and b.stride(1) == 1
          and a.stride(0) % 8 == 0 and b.stride(0) % 8 == 0 and a.data_ptr() % 16 == 0 and b.data_ptr() % 16 == 0)


def gemm(a: torch.Tensor, b: torch.Tensor, a_mn_major: bool = False, b_mn_major: bool = False,
         bias: Optional[torch.Tensor] = None, epilogue: int = EPI_NONE, pre: Optional[torch.Tensor] = None,
         aux: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None, accumulate: bool = False,
         out_dtype: Optional[torch.dtype] = None, alpha: float = 1.0) -> torch.Tensor:
  """``D[M,N] = op(a) @ op(b)``.

  ``a``: ``[M,K]`` (K-major) or ``[K,M]`` (``a_mn_major``); ``b``: ``[N,K]`` or ``[K,N]`` (``b_mn_major``).
  """
  lib = _lib.require()
  if a_mn_major:
    K, M = a.shape
  else:
    M, K = a.shape
  if b_mn_major:
    Kb, N = b.shape
  else:
    N, Kb = b.shape
  if K != Kb:
    raise ValueError("gemm: contraction mismatch %d vs %d" % (K, Kb))
  if not gemm_supported(a, b):
    raise ValueError("gemm: operands must be 2-D bf16/fp16 CUDA tensors, unit inner stride, 16-byte aligned rows")
  if out is None:
    out = torch.empty((M, N), dtype=out_dtype or a.dtype, device=a.device)
  elif out.shape != (M, N) or out.stride(1) != 1:
    raise ValueError("gemm: bad output shape/stride")
  if epilogue in (EPI_DGELU, EPI_BIAS_RESIDUAL) and (aux is None or aux.stride(0) != out.stride(0)):
    raise ValueError("gemm: aux must share the output's row stride")
  if pre is not None and pre.stride(0) != out.stride(0):
    raise ValueError("gemm: pre must share the output's row stride")
  rc = lib.epl_gemm(a.data_ptr(), b.data_ptr(), out.data_ptr(), M, N, K, a.stride(0), b.stride(0), out.stride(0),
                    int(a_mn_major), int(b_mn_major), _lib.ptr(bias), _lib.ptr(pre), _lib.ptr(aux), epilogue,
                    int(accumulate), _lib.dtype_code(out.dtype), alpha, int(a.dtype == torch.float16), _FORCE_BN,
                    _NUM_SMS, _lib.stream())
  _lib.check(rc, "gemm")
  return out


def colsum(x2: torch.Tensor) -> torch.Tensor:
  lib = _lib.require()
  rows, D = x2.shape
  out = torch.empty(D, dtype=x2.dtype, device=x2.device)
  scratch = torch.empty(lib.epl_colsum_parts(rows, D, _lib.dtype_code(x2.dtype)), D, dtype=torch.float32, device=x2.device)
  rc = lib.epl_colsum(x2.data_ptr(), out.data_ptr(), scratch.data_ptr(), rows, D, _lib.dtype_code(x2.dtype), 0, _lib.stream())
  _lib.check(rc, "colsum")
  _lib.launches += 1
  return out


def _sink_weight_grad(w: torch.Tensor, a: torch.Tensor, b: torch.Tensor) -> Optional[torch.Tensor]:
  """dW = a^T @ b with a:[M,N] b:[M,K].  When the engine registered a flat gradient view on the
  parameter (``epl_main_grad``) the GEMM accumulates straight into it (no autograd add pass)."""
  sink = getattr(w, "epl_main_grad", None)
  if sink is not None and sink.dtype in (torch.bfloat16, torch.float16, torch.float32):
    # first contribution of the step to a weight with a single use: plain store (no read-modify-write of the bucket)
    fresh = getattr(w, "epl_sink_fresh", False)
    if fresh:
      w.epl_sink_fresh = False
    gemm(a, b, a_mn_major=True, b_mn_major=True, out=sink.view(w.shape), accumulate=not fresh)
    ready = getattr(w, "epl_grad_ready", None)
    if ready is not None:
      ready(w)
    return None
  return gemm(a, b, a_mn_major=True, b_mn_major=True)


def _fwd_gemm(x2: torch.Tensor, w: torch.Tensor):
  """Forward GEMM of a linear layer: the fp8 path (``amp.level = "fp8"``, ops/fp8.py) when enabled and the shape fits it."""
  from easyparallellibrary_b200.ops import fp8
  if fp8.ENABLED and x2.dtype == torch.bfloat16 and w.is_contiguous() and fp8.supported(x2.shape[0], w.shape[0], x2.shape[1]):
    return fp8.gemm_fp8
  return gemm


class _LinearFn(torch.autograd.Function):
  @staticmethod
  def forward(ctx, x, w, bias, gelu, residual=None):
    x2 = x.reshape(-1, x.shape[-1])
    if not x2.is_contiguous():
      x2 = x2.contiguous()
    gemm = _fwd_gemm(x2, w)
    pre = None
    ctx.has_res = residual is not None
    if residual is not None:
      r2 = residual.reshape(-1, w.shape[0])
      if not r2.is_contiguous():
        r2 = r2.contiguous()
      y = gemm(x2, w, bias=bias, epilogue=EPI_BIAS_RESIDUAL, aux=r2)
    elif gelu:
      pre = torch.empty((x2.shape[0], w.shape[0]), dtype=x.dtype, device=x.device)
      y = gemm(x2, w, bias=bias, epilogue=EPI_BIAS_GELU, pre=pre)
    else:
      y = gemm(x2, w, bias=bias, epilogue=EPI_BIAS if bias is not None else EPI_NONE)
    ctx.save_for_backward(x2, w, pre if pre is not None else x2.new_empty(0))
    ctx.has_bias, ctx.gelu, ctx.xshape = bias is not None, gelu, x.shape
    return y.view(*x.shape[:-1], w.shape[0])

  @staticmethod
  def backward(ctx, dy):
    x2, w, pre = ctx.saved_tensors
    dy2 = dy.reshape(-1, dy.shape[-1])
    if not dy2.is_contiguous():
      dy2 = dy2.contiguous()
    if ctx.gelu:
      lib = _lib.require()
      dpre = torch.empty_like(dy2)
      rc = lib.epl_gelu_bwd(pre.data_ptr(), dy2.data_ptr(), dpre.data_ptr(), dy2.numel(), _lib.dtype_code(dy2.dtype), _lib.stream())
      _lib.check(rc, "gelu_bwd")
      dy2 = dpre
    dx = gemm(dy2, w, b_mn_major=True).view(ctx.xshape) if ctx.needs_input_grad[0] else None
    dw = _sink_weight_grad(w, dy2, x2) if ctx.needs_input_grad[1] else None
    db = colsum(dy2) if ctx.has_bias and ctx.needs_input_grad[2] else None
    return dx, dw, db, None, (dy if ctx.has_res else None)


class _MlpFn(torch.autograd.Function):
  """y = gelu(x W1^T + b1) W2^T + b2, four GEMMs in backward, GELU' fused into the dH epilogue."""

  @staticmethod
  def forward(ctx, x, w1, b1, w2, b2, residual=None):
    x2 = x.reshape(-1, x.shape[-1])
    if not x2.is_contiguous():
      x2 = x2.contiguous()
    pre = torch.empty((x2.shape[0], w1.shape[0]), dtype=x.dtype, device=x.device)
    h = _fwd_gemm(x2, w1)(x2, w1, bias=b1, epilogue=EPI_BIAS_GELU, pre=pre)
    gemm2_ = _fwd_gemm(h, w2)
    ctx.has_res = residual is not None
    if residual is not None:
      r2 = residual.reshape(-1, w2.shape[0])
      if not r2.is_contiguous():
        r2 = r2.contiguous()
      y = gemm2_(h, w2, bias=b2, epilogue=EPI_BIAS_RESIDUAL, aux=r2)
    else:
      y = gemm2_(h, w2, bias=b2, epilogue=EPI_BIAS if b2 is not None else EPI_NONE)
    ctx.save_for_backward(x2, w1, w2, pre, h)
    ctx.has_b1, ctx.has_b2, ctx.xshape = b1 is not None, b2 is not None, x.shape
    return y.view(*x.shape[:-1], w2.shape[0])

  @staticmethod
  def backward(ctx, dy):
    x2, w1, w2, pre, h = ctx.saved_tensors
    dy2 = dy.reshape(-1, dy.shape[-1])
    if not dy2.is_contiguous():
      dy2 = dy2.contiguous()
    dpre = gemm(dy2, w2, b_mn_major=True, epilogue=EPI_DGELU, aux=pre)
    dw2 = _sink_weight_grad(w2, dy2, h)
    db2 = colsum(dy2) if ctx.has_b2 else None
    dx = gemm(dpre, w1, b_mn_major=True).view(ctx.xshape) if ctx.needs_input_grad[0] else None
    dw1 = _sink_weight_grad(w1, dpre, x2)
    db1 = colsum(dpre) if ctx.has_b1 else None
    return dx, dw1, db1, dw2, db2, (dy if ctx.has_res else None)


_AB_TORCH = os.environ.get("EPL_LINEAR", "") == "torch"    # measurement aid: A/B the whole step against cuBLAS + unfused epilogues


def _use_kernel(x: torch.Tensor, w: torch.Tensor) -> bool:
  if _AB_TORCH:
    return False
  return (x.is_cuda and x.dtype in (torch.bfloat16, torch.float16) and w.dtype == x.dtype
          and x.shape[-1] % 8 == 0 and w.shape[0] % 8 == 0 and w.is_contiguous())


class _GatherLinearFn(torch.autograd.Function):
  """``linear`` whose weight is a ZeRO-3 shard with a deferred all-gather (``parallel/zero3.py::PendingGather``): the forward
  GEMM gathers the weight over NVLink while it multiplies (K2, ``ops/tp_kernels.ag_weight_gemm``); backward is the ordinary
  pair of GEMMs on the weight the ZeRO-3 engine re-gathers before the layer's backward."""

  @staticmethod
  def forward(ctx, x, w, bias, gelu, pend):
    x2 = x.reshape(-1, x.shape[-1])
    if not x2.is_contiguous():
      x2 = x2.contiguous()
    y, pre = pend.gemm(x2, bias, gelu)                      # fills w's storage as a side effect
    ctx.save_for_backward(x2, w, pre if pre is not None else x2.new_empty(0))
    ctx.has_bias, ctx.gelu, ctx.xshape, ctx.has_res = bias is not None, gelu, x.shape, False
    return y.view(*x.shape[:-1], w.shape[0])

  @staticmethod
  def backward(ctx, dy):
    x2, w, pre = ctx.saved_tensors
    if x2.is_cuda and _lib.available():
      return _LinearFn.backward(ctx, dy)
    dy2 = dy.reshape(-1, dy.shape[-1])                      # reference math (CPU tests of the protocol)
    if ctx.gelu:
      with torch.enable_grad():
        pr = pre.detach().requires_grad_()
        torch.nn.functional.gelu(pr, approximate="tanh").backward(dy2)
      dy2 = pr.grad
    dx = (dy2 @ w).view(ctx.xshape) if ctx.needs_input_grad[0] else None
    dw = dy2.t() @ x2 if ctx.needs_input_grad[1] else None
    db = dy2.sum(0) if ctx.has_bias and ctx.needs_input_grad[2] else None
    return dx, dw, db, None, None


def _resolve_pending(x: torch.Tensor, w: torch.Tensor, fusable: bool):
  """ZeRO-3 deferred gather: returns the pending object if the fused weight-gather GEMM should run, else gathers now."""
  pend = getattr(w, "epl_pending_gather", None)
  if pend is None:
    return None
  if fusable and pend.can_fuse(x):
    return pend
  pend.materialize()
  return None


def linear(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, gelu: bool = False,
           residual: Optional[torch.Tensor] = None) -> torch.Tensor:
  """``y = x @ w^T (+ bias) (GELU)`` or, with ``residual``, ``y = residual + x @ w^T + bias`` — one kernel either way."""
  from easyparallellibrary_b200.runtime import amp
  if amp.o1_active():                            # O1 allow-list op: fp16 inputs, fp32 weights cast just in time
    x, w, bias, residual = amp.cast_args("linear", x, w, bias, residual)
  pend = _resolve_pending(x, w, fusable=residual is None)
  if pend is not None:
    return _GatherLinearFn.apply(x, w, bias, gelu, pend)
  if _use_kernel(x, w):
    return _LinearFn.apply(x, w, bias, gelu, residual)
  y = torch.nn.functional.linear(x, w, bias)
  if residual is not None:
    return residual + y
  return torch.nn.functional.gelu(y, approximate="tanh") if gelu else y


def mlp(x, w1, b1, w2, b2, residual: Optional[torch.Tensor] = None) -> torch.Tensor:
  from easyparallellibrary_b200.runtime import amp
  if amp.o1_active():
    x, w1, b1, w2, b2, residual = amp.cast_args("mlp", x, w1, b1, w2, b2, residual)
  _resolve_pending(x, w1, fusable=False)          # the fused MLP block keeps its own kernels: gather a deferred weight first
  if _use_kernel(x, w1) and w2.shape[0] % 8 == 0:
    return _MlpFn.apply(x, w1, b1, w2, b2, residual)
  h = torch.nn.functional.gelu(torch.nn.functional.linear(x, w1, b1), approximate="tanh")
  y = torch.nn.functional.linear(h, w2, b2)
  return y if residual is None else residual + y


class Linear(nn.Module):
  """Drop-in ``nn.Linear`` (weight ``[out, in]``) running on the tcgen05 GEMM."""

  def __init__(self, in_features: int, out_features: int, bias: bool = True, gelu: bool = False, init_std: Optional[float] = None):
    super().__init__()
    self.in_features, self.out_features, self.gelu, self.init_std = in_features, out_features, gelu, init_std
    self.weight = nn.Parameter(torch.empty(out_features, in_features))
    self.bias = nn.Parameter(torch.empty(out_features)) if bias else None
    self.reset_parameters()

  def reset_parameters(self):
    if self.weight.is_meta:
      return
    if self.init_std is not None:
      nn.init.normal_(self.weight, std=self.init_std)
    else:
      nn.init.kaiming_uniform_(self.weight, a=math.sqrt(5))
    if self.bias is not None:
      nn.init.zeros_(self.bias)

  def epl_flops(self, inputs, output):
    x = inputs[0]
    return 2.0 * (x.numel() // x.shape[-1]) * self.in_features * self.out_features

  def forward(self, x):
    return linear(x, self.weight, self.bias, self.gelu)
