"""Numerics of every sm_100a kernel against a plain PyTorch fp32 reference of the same op."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _close(a, b, rtol, atol, what=""):
  a, b = a.float(), b.float()
  err = (a - b).abs()
  tol = atol + rtol * b.abs()
  bad = (err > tol).float().mean().item()
  assert bad < 1e-3, "%s: %.4f%% elements out of tolerance, max err %.4g (ref max %.4g)" % (
      what, bad * 100, err.max().item(), b.abs().max().item())


@pytest.mark.parametrize("gdt,odt", [(torch.bfloat16, torch.bfloat16), (torch.float32, None), (torch.float16, torch.float16)])
def test_adamw(gdt, odt):
  from easyparallellibrary_b200.ops import fused_optim
  from easyparallellibrary_b200.runtime.optimizer import AdamHyper, adamw_reference
  torch.manual_seed(0)
  n = 1_000_003 if gdt == torch.float32 else 1 << 20
  master = torch.randn(n, device=DEV)
  grad = (torch.randn(n, device=DEV) * 3).to(gdt)
  m, v = torch.rand(n, device=DEV) * 0.1, torch.rand(n, device=DEV) * 0.1
  mask = (torch.rand(n, device=DEV) > 0.3).float()
  out = torch.empty(n, device=DEV, dtype=odt) if odt else None
  h = AdamHyper(lr=1e-2, weight_decay=0.1)
  rm, rmm, rv = master.clone(), m.clone(), v.clone()
  rout = torch.empty(n, device=DEV, dtype=odt) if odt else None
  adamw_reference(rm, grad, rmm, rv, 3, h, 0.5, mask, rout)
  fused_optim.adamw_step(master, grad, m, v, 3, h, 0.5, mask, out)
  _close(master, rm, 1e-5, 1e-6, "master")
  _close(m, rmm, 1e-5, 1e-6, "m")
  _close(v, rv, 1e-5, 1e-6, "v")
  if odt:
    _close(out, rout, 1e-2, 1e-3, "out")


def test_sgd_and_sumsq():
  from easyparallellibrary_b200.ops import fused_optim
  from easyparallellibrary_b200.runtime.optimizer import SGDHyper, sgd_reference
  n = 100_001
  master, grad, mom = torch.randn(n, device=DEV), torch.randn(n, device=DEV).bfloat16(), torch.randn(n, device=DEV)
  rm, rmom = master.clone(), mom.clone()
  h = SGDHyper(lr=0.1, momentum=0.9, weight_decay=0.01)
  out, rout = torch.empty(n, device=DEV, dtype=torch.bfloat16), torch.empty(n, device=DEV, dtype=torch.bfloat16)
  sgd_reference(rm, grad, rmom, h, 2.0, rout)
  fused_optim.sgd_step(master, grad, mom, h, 2.0, out)
  _close(master, rm, 1e-5, 1e-6, "sgd")
  s = fused_optim.sumsq_and_finite(grad)
  assert abs(s[0].item() - grad.float().pow(2).sum().item()) / s[0].item() < 1e-3 and s[1].item() == 0
  grad[7] = float("inf")
  assert fused_optim.sumsq_and_finite(grad)[1].item() == 1.0


@pytest.mark.parametrize("D", [768, 1600, 4096])
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float32])
def test_layernorm(D, dt):
  from easyparallellibrary_b200.ops.layernorm import layer_norm, rms_norm
  torch.manual_seed(0)
  rows = 1000
  x = (torch.randn(rows, D, device=DEV) * 2 + 0.5).to(dt).requires_grad_()
  g = (torch.rand(D, device=DEV) + 0.5).to(dt).requires_grad_()
  b = torch.randn(D, device=DEV).to(dt).requires_grad_()
  dy = torch.randn(rows, D, device=DEV).to(dt)
  y = layer_norm(x, g, b)
  y.backward(dy)
  xf, gf, bf = x.detach().float().requires_grad_(), g.detach().float().requires_grad_(), b.detach().float().requires_grad_()
  yr = torch.nn.functional.layer_norm(xf, (D,), gf, bf)
  yr.backward(dy.float())
  tol = (2e-2, 2e-2) if dt == torch.bfloat16 else (1e-4, 1e-4)
  _close(y, yr, *tol, "ln y")
  _close(x.grad, xf.grad, *tol, "ln dx")
  _close(g.grad, gf.grad, tol[0], tol[1] * 30, "ln dgamma")
  _close(b.grad, bf.grad, tol[0], tol[1] * 30, "ln dbeta")
  x.grad = None
  y2 = rms_norm(x, g)
  y2.backward(dy)
  xf.grad = None
  yr2 = xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + 1e-6) * gf
  yr2.backward(dy.float())
  _close(y2, yr2, *tol, "rms y")
  _close(x.grad, xf.grad, *tol, "rms dx")


def test_xent():
  from easyparallellibrary_b200.ops.cross_entropy import softmax_cross_entropy
  torch.manual_seed(0)
  rows, V = 300, 50304
  logits = (torch.randn(rows, V, device=DEV) * 3).bfloat16()
  labels = torch.randint(0, V, (rows,), device=DEV)
  labels[5] = -100
  ref_in = logits.float().requires_grad_()
  ref = torch.nn.functional.cross_entropy(ref_in, labels, ignore_index=-100)
  (ref * 2).backward()
  mine_in = logits.clone().requires_grad_()
  loss = softmax_cross_entropy(mine_in, labels)
  (loss * 2).backward()
  assert abs(loss.item() - ref.item()) < 2e-3 * abs(ref.item())
  _close(mine_in.grad, ref_in.grad, 2e-2, 1e-6, "dlogits")


CASES = [  # (M, N, K)
    (256, 256, 128), (128, 160, 64), (384, 512, 320), (1000, 1600, 1600), (2048, 6400, 1600), (333, 264, 200),
]


@pytest.mark.parametrize("M,N,K", CASES)
@pytest.mark.parametrize("layout", ["nt", "nn", "tn"])
def test_gemm_layouts(M, N, K, layout):
  from easyparallellibrary_b200.ops.linear import gemm
  torch.manual_seed(0)
  K = (K + 7) // 8 * 8
  if layout == "nt":      # D = A[M,K] @ B[N,K]^T
    a, b = torch.randn(M, K, device=DEV).bfloat16(), torch.randn(N, K, device=DEV).bfloat16()
    ref = a.float() @ b.float().t()
    out = gemm(a, b)
  elif layout == "nn":    # D = A[M,K] @ B[K,N]
    N = (N + 7) // 8 * 8
    a, b = torch.randn(M, K, device=DEV).bfloat16(), torch.randn(K, N, device=DEV).bfloat16()
    ref = a.float() @ b.float()
    out = gemm(a, b, b_mn_major=True)
  else:                   # D = A[K,M]^T @ B[K,N]
    M, N = (M + 7) // 8 * 8, (N + 7) // 8 * 8
    a, b = torch.randn(K, M, device=DEV).bfloat16(), torch.randn(K, N, device=DEV).bfloat16()
    ref = a.float().t() @ b.float()
    out = gemm(a, b, a_mn_major=True, b_mn_major=True)
  _close(out, ref, 1e-2, 1e-2 * math.sqrt(K), "gemm %s" % layout)


@pytest.mark.parametrize("bn", [128, 160, 256, 512])       # 512 = the 2-CTA (cta_group::2) 256x256 kernel
def test_gemm_tile_widths_and_epilogues(bn):
  from easyparallellibrary_b200.ops import linear as L
  torch.manual_seed(1)
  M, N, K = 512, 1280, 512
  a, b = torch.randn(M, K, device=DEV).bfloat16(), (torch.randn(N, K, device=DEV) * 0.05).bfloat16()
  bias = torch.randn(N, device=DEV).bfloat16()
  L._FORCE_BN = bn
  try:
    ref = a.float() @ b.float().t() + bias.float()
    _close(L.gemm(a, b, bias=bias, epilogue=L.EPI_BIAS), ref, 1e-2, 5e-2, "bias")
    pre = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    act = L.gemm(a, b, bias=bias, epilogue=L.EPI_BIAS_GELU, pre=pre)
    _close(pre, ref, 1e-2, 5e-2, "pre")
    _close(act, torch.nn.functional.gelu(pre.float(), approximate="tanh"), 1e-2, 2e-2, "gelu")
    res = torch.randn(M, N, device=DEV).bfloat16()
    _close(L.gemm(a, b, bias=bias, epilogue=L.EPI_BIAS_RESIDUAL, aux=res), ref + res.float(), 1e-2, 5e-2, "residual")
    x = pre.float().requires_grad_()
    torch.nn.functional.gelu(x, approximate="tanh").sum().backward()
    _close(L.gemm(a, b, epilogue=L.EPI_DGELU, aux=pre), (a.float() @ b.float().t()) * x.grad, 1e-2, 5e-2, "dgelu")
    acc = torch.randn(M, N, device=DEV)
    expect = acc + a.float() @ b.float().t()
    _close(L.gemm(a, b, out=acc, accumulate=True), expect, 1e-2, 5e-2, "accumulate fp32")
  finally:
    L._FORCE_BN = 0


def test_linear_and_mlp_autograd():
  from easyparallellibrary_b200.ops.linear import linear, mlp
  torch.manual_seed(2)
  B, S, d = 4, 96, 256
  x = torch.randn(B, S, d, device=DEV).bfloat16().requires_grad_()
  w1 = (torch.randn(4 * d, d, device=DEV) * 0.05).bfloat16().requires_grad_()
  b1 = torch.randn(4 * d, device=DEV).bfloat16().requires_grad_()
  w2 = (torch.randn(d, 4 * d, device=DEV) * 0.05).bfloat16().requires_grad_()
  b2 = torch.randn(d, device=DEV).bfloat16().requires_grad_()
  dy = torch.randn(B, S, d, device=DEV).bfloat16()
  y = mlp(x, w1, b1, w2, b2)
  y.backward(dy)
  f = [t.detach().float().requires_grad_() for t in (x, w1, b1, w2, b2)]
  yr = torch.nn.functional.linear(torch.nn.functional.gelu(torch.nn.functional.linear(f[0], f[1], f[2]), approximate="tanh"), f[3], f[4])
  yr.backward(dy.float())
  _close(y, yr, 2e-2, 5e-2, "mlp y")
  for name, t, r in zip(("dx", "dw1", "db1", "dw2", "db2"), (x, w1, b1, w2, b2), f):
    _close(t.grad, r.grad, 3e-2, 3e-2 * r.grad.abs().max().item(), "mlp " + name)
  x.grad = None
  w = (torch.randn(3 * d, d, device=DEV) * 0.05).bfloat16().requires_grad_()
  y = linear(x, w, None)
  y.backward(torch.ones_like(y))
  _close(w.grad, (torch.ones(B * S, 3 * d, device=DEV).t() @ x.detach().float().view(-1, d)), 2e-2, 0.5, "linear dw")


def test_gpt2_tiny_step_matches_torch():
  """One training step of GPT-2-tiny through the engine on the kernels vs the same model on torch fp32 ops."""
  import easyparallellibrary_b200 as epl
  from easyparallellibrary_b200.models.gpt2 import GPT2, GPT2Config
  torch.manual_seed(0)
  epl.init(epl.Config({"amp.level": "bf16"}))
  with epl.replicate(1):
    model = GPT2(GPT2Config.named("tiny"))
  ref = GPT2(GPT2Config.named("tiny"))
  ref.load_state_dict(model.state_dict())
  tr = epl.Trainer(model, "adamw", lr=1e-3)
  idx = torch.randint(0, 512, (8, 128), device=DEV)
  losses = [tr.step(idx, idx).item() for _ in range(5)]
  opt = torch.optim.AdamW(ref.parameters(), lr=1e-3, weight_decay=0.01)
  ref_losses = []
  for _ in range(5):
    loss = ref(idx.cpu(), idx.cpu())
    opt.zero_grad()
    loss.backward()
    opt.step()
    ref_losses.append(loss.item())
  assert losses[-1] < losses[0]
  for a, b in zip(losses, ref_losses):
    assert abs(a - b) < 0.05 * abs(b) + 0.05, (losses, ref_losses)


def test_layernorm_fork_and_residual_linear():
  """Pre-LN residual block pieces: LN fork (skip gradient joined inside the LN backward kernel) and the
  residual-add GEMM epilogue, against plain fp32 autograd."""
  from easyparallellibrary_b200.ops.layernorm import layer_norm_fork
  from easyparallellibrary_b200.ops.linear import linear, mlp
  torch.manual_seed(3)
  B, S, d = 2, 64, 256
  x = torch.randn(B, S, d, device=DEV).bfloat16().requires_grad_()
  g = (torch.rand(d, device=DEV) + 0.5).bfloat16().requires_grad_()
  b = torch.randn(d, device=DEV).bfloat16().requires_grad_()
  w = (torch.randn(d, d, device=DEV) * 0.05).bfloat16().requires_grad_()
  wb = torch.randn(d, device=DEV).bfloat16().requires_grad_()
  w1 = (torch.randn(4 * d, d, device=DEV) * 0.05).bfloat16().requires_grad_()
  b1 = torch.zeros(4 * d, device=DEV).bfloat16().requires_grad_()
  w2 = (torch.randn(d, 4 * d, device=DEV) * 0.05).bfloat16().requires_grad_()
  b2 = torch.zeros(d, device=DEV).bfloat16().requires_grad_()
  dy = torch.randn(B, S, d, device=DEV).bfloat16()

  def block(x, g, b, w, wb, w1, b1, w2, b2, fused):
    F = torch.nn.functional
    if fused:
      skip, h = layer_norm_fork(x, g, b)
      x2 = linear(h, w, wb, residual=skip)
      skip, h = layer_norm_fork(x2, g, b)
      return mlp(h, w1, b1, w2, b2, residual=skip)
    h = F.layer_norm(x, (d,), g, b)
    x2 = x + F.linear(h, w, wb)
    h = F.layer_norm(x2, (d,), g, b)
    return x2 + F.linear(F.gelu(F.linear(h, w1, b1), approximate="tanh"), w2, b2)

  params = (x, g, b, w, wb, w1, b1, w2, b2)
  y = block(*params, True)
  y.backward(dy)
  ref = [t.detach().float().requires_grad_() for t in params]
  yr = block(*ref, False)
  yr.backward(dy.float())
  _close(y, yr, 3e-2, 5e-2, "block y")
  for name, t, r in zip("x g b w wb w1 b1 w2 b2".split(), params, ref):
    _close(t.grad, r.grad, 4e-2, 4e-2 * r.grad.abs().max().item(), "block d" + name)


@pytest.mark.parametrize("causal", [True, False])
@pytest.mark.parametrize("B,S,H", [(2, 256, 3), (1, 1024, 2), (2, 200, 2), (1, 384, 4), (1, 4160, 2)])  # 4160: 3 launches
def test_flash_attention_packed(B, S, H, causal):
  """tcgen05 flash attention fwd + bwd vs fp32 softmax(QK^T)V autograd."""
  from easyparallellibrary_b200.ops.attention_kernel import flash_attention_packed
  torch.manual_seed(0)
  D = 64
  qkv = (torch.randn(B, S, 3, H, D, device=DEV) * 0.8).bfloat16().requires_grad_()
  dout = torch.randn(B, S, H * D, device=DEV).bfloat16()
  out = flash_attention_packed(qkv, causal)
  out.backward(dout)
  ref_in = qkv.detach().float().requires_grad_()
  q, k, v = ref_in.permute(2, 0, 3, 1, 4).unbind(0)
  s = q @ k.transpose(-1, -2) / math.sqrt(D)
  if causal:
    s = s.masked_fill(~torch.ones(S, S, dtype=torch.bool, device=DEV).tril(), float("-inf"))
  ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B, S, H * D)
  ref.backward(dout.float())
  _close(out, ref, 2e-2, 2e-2, "attn out")
  g, gr = qkv.grad.float(), ref_in.grad
  for idx, name in enumerate(("dq", "dk", "dv")):
    _close(g[:, :, idx], gr[:, :, idx], 3e-2, 3e-2 * gr[:, :, idx].abs().max().item(), "attn " + name)


@pytest.mark.parametrize("causal", [True, False])
def test_backward_gradients_are_bitwise_reproducible(causal):
  """Same inputs, same bits: the attention backward's dQ (slot-ordered sums, in one launch and in several) and the bias-gradient
  column sums (partial rows added in a fixed order) do not depend on which CTA finishes first."""
  from easyparallellibrary_b200.ops.attention_kernel import flash_attention_packed
  from easyparallellibrary_b200.ops.linear import colsum
  torch.manual_seed(0)
  for B, S, H in ((8, 1024, 4), (1, 4160, 2)):
    qkv = (torch.randn(B, S, 3, H, 64, device=DEV) * 0.8).bfloat16()
    dout = torch.randn(B, S, H * 64, device=DEV).bfloat16()
    grads = []
    for _ in range(3):
      x = qkv.clone().requires_grad_()
      flash_attention_packed(x, causal).backward(dout)
      grads.append(x.grad)
    assert all(torch.equal(grads[0], g) for g in grads[1:]), (B, S, H)
  x = torch.randn(8192, 1600, device=DEV).bfloat16()
  sums = [colsum(x) for _ in range(3)]
  assert all(torch.equal(sums[0], t) for t in sums[1:])


@pytest.mark.parametrize("causal", [True, False])
def test_flash_attention_rescale_path(causal):
  """Large logits: the running row maximum keeps moving by more than 2^8 in later key tiles, which exercises the lazy
  in-TMEM rescale of the output accumulator (csrc/attention.cu) and the two-half row-max exchange."""
  from easyparallellibrary_b200.ops.attention_kernel import flash_attention_packed
  torch.manual_seed(1)
  B, S, H, D = 2, 640, 2, 64
  qkv = torch.randn(B, S, 3, H, D, device=DEV)
  qkv[:, :, :2] *= 3.0                                     # scores ~ N(0, 9^2): log2 range of several tens
  qkv = qkv.bfloat16().requires_grad_()
  dout = torch.randn(B, S, H * D, device=DEV).bfloat16()
  out = flash_attention_packed(qkv, causal)
  out.backward(dout)
  ref_in = qkv.detach().float().requires_grad_()
  q, k, v = ref_in.permute(2, 0, 3, 1, 4).unbind(0)
  s = q @ k.transpose(-1, -2) / math.sqrt(D)
  if causal:
    s = s.masked_fill(~torch.ones(S, S, dtype=torch.bool, device=DEV).tril(), float("-inf"))
  ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B, S, H * D)
  ref.backward(dout.float())
  _close(out, ref, 3e-2, 3e-2, "attn out (large logits)")
  g, gr = qkv.grad.float(), ref_in.grad
  for idx, name in enumerate(("dq", "dk", "dv")):
    _close(g[:, :, idx], gr[:, :, idx], 4e-2, 4e-2 * gr[:, :, idx].abs().max().item(), "attn large " + name)


def test_vocab_parallel_xent_kernel_modes():
  """K4 on one GPU: split the classes into two shards, run the statistics / gradient kernels per shard and combine
  exactly like the distributed op does; compare with the unsharded fp32 cross-entropy."""
  from easyparallellibrary_b200.ops.tensor_parallel import _VocabParallelXent

  class FakeComm:
    size, rank = 1, 0

  torch.manual_seed(0)
  rows, V = 64, 4096
  logits = (torch.randn(rows, V, device=DEV) * 2).bfloat16()
  labels = torch.randint(0, V, (rows,), device=DEV)
  ref_in = logits.float().requires_grad_()
  ref = torch.nn.functional.cross_entropy(ref_in, labels, reduction="none")
  ref.sum().backward()
  half = V // 2
  shards = [logits[:, :half].contiguous().requires_grad_(), logits[:, half:].contiguous().requires_grad_()]
  lib = __import__("easyparallellibrary_b200.ops._lib", fromlist=["require"]).require()
  from easyparallellibrary_b200.ops import _lib
  stats = []
  for i, sh in enumerate(shards):
    st = torch.empty(rows, 3, dtype=torch.float32, device=DEV)
    rc = lib.epl_xent(sh.data_ptr(), labels.data_ptr(), None, None, st.data_ptr(), None, rows, half, sh.stride(0), 1.0, -100, i * half, 1,
                      _lib.BF16, _lib.stream())
    assert rc == 0
    stats.append(st)
  allst = torch.stack(stats)
  gmax = allst[:, :, 0].max(0).values
  gsum = (allst[:, :, 1] * (allst[:, :, 0] - gmax).exp()).sum(0)
  loss = gsum.log() + gmax - allst[:, :, 2].sum(0)
  _close(loss, ref, 1e-2, 2e-2, "vocab-parallel loss")
  gst = torch.stack([gmax, gsum], 1).contiguous()
  for i, sh in enumerate(shards):
    g = torch.empty_like(sh)
    rc = lib.epl_xent(sh.data_ptr(), labels.data_ptr(), None, g.data_ptr(), None, gst.data_ptr(), rows, half, sh.stride(0), 1.0, -100,
                      i * half, 2, _lib.BF16, _lib.stream())
    assert rc == 0
    _close(g, ref_in.grad[:, i * half:(i + 1) * half], 2e-2, 1e-4, "vocab-parallel grad shard %d" % i)


@pytest.mark.parametrize("width", [512, 448, 384, 1024])
@pytest.mark.parametrize("layout", ["nt", "nn", "tn"])
@pytest.mark.parametrize("M,N,K", [(512, 512, 256), (1000, 1600, 1600), (8192, 6400, 1600), (300, 264, 200)])
def test_gemm_two_cta_layouts(M, N, K, layout, width):
  """cta_group::2 kernel, every tile width (256 / 192 / 128 = force codes 512 / 448 / 384), on all three operand layouts
  incl. ragged edges (the 192-wide tile reads 1.5 swizzle atoms of an MN-major B per CTA); 1024 = the 4-CTA cluster
  kernel that multicasts the B tile across two CTA pairs."""
  from easyparallellibrary_b200.ops import linear as L
  torch.manual_seed(0)
  M, N, K = (M + 7) // 8 * 8, (N + 7) // 8 * 8, (K + 7) // 8 * 8
  L._FORCE_BN = width
  try:
    if layout == "nt":
      a, b = torch.randn(M, K, device=DEV).bfloat16(), torch.randn(N, K, device=DEV).bfloat16()
      ref, out = a.float() @ b.float().t(), L.gemm(a, b)
    elif layout == "nn":
      a, b = torch.randn(M, K, device=DEV).bfloat16(), torch.randn(K, N, device=DEV).bfloat16()
      ref, out = a.float() @ b.float(), L.gemm(a, b, b_mn_major=True)
    else:
      a, b = torch.randn(K, M, device=DEV).bfloat16(), torch.randn(K, N, device=DEV).bfloat16()
      ref, out = a.float().t() @ b.float(), L.gemm(a, b, a_mn_major=True, b_mn_major=True)
  finally:
    L._FORCE_BN = 0
  _close(out, ref, 1e-2, 1e-2 * math.sqrt(K), "2cta gemm %s" % layout)


def test_rope_kernel():
  from easyparallellibrary_b200.ops.rope import apply_rope, rope_reference
  torch.manual_seed(0)
  qkv = torch.randn(2, 96, 3, 4, 64, device=DEV).bfloat16().requires_grad_()
  out = apply_rope(qkv, 10000.0, 3)
  ref_in = qkv.detach().float().requires_grad_()
  ref = rope_reference(ref_in, 10000.0, 3)
  _close(out, ref, 2e-2, 2e-2, "rope fwd")
  g = torch.randn_like(out)
  out.backward(g)
  ref.backward(g.float())
  _close(qkv.grad, ref_in.grad, 2e-2, 3e-2, "rope bwd")
  assert torch.equal(out[:, :, 2], qkv[:, :, 2])          # V untouched


def test_cuda_graph_step_matches_eager_step():
  """The whole training step captured in a CUDA graph (parallel/graph_step.py) follows the eager trajectory: same kernels,
  per-step optimizer values read from device memory; and it really replays (no eager launches after the capture)."""
  import easyparallellibrary_b200 as epl
  from easyparallellibrary_b200.models.gpt2 import GPT2, GPT2Config
  from easyparallellibrary_b200.ops import _lib
  runs = {}
  for graph in (False, True):
    torch.manual_seed(0)
    epl.init(epl.Config({"amp.level": "bf16"}))
    with epl.replicate(1):
      model = GPT2(GPT2Config.named("tiny"))
    tr = epl.Trainer(model, "adamw", lr=1e-3, cuda_graph=graph)
    g = torch.Generator().manual_seed(1)
    toks = [torch.randint(0, 512, (8, 128), generator=g).to(DEV) for _ in range(8)]
    runs[graph] = [tr.step(t, t).item() for t in toks]
    if graph:
      assert tr._graphed is not None and tr._graphed.graph is not None and not tr._graphed.failed
      assert tr._graphed.launches_per_replay > 20
      assert tr.optimizers[0][0].step_count == 8
  for a, b in zip(runs[False], runs[True]):
    assert abs(a - b) < 2e-3 * abs(a) + 1e-3, (runs[False], runs[True])


def test_fp8_quantize_and_gemm():
  """e4m3 path: the quantiser against torch's float8_e4m3fn cast, the UTCQMMA GEMM against an fp32 matmul of the SAME quantised
  operands (tight: only accumulation order and the bf16 output rounding differ) and against the unquantised product (loose: e4m3
  has 3 mantissa bits)."""
  from easyparallellibrary_b200.ops import fp8
  from easyparallellibrary_b200.ops import linear as L
  torch.manual_seed(0)
  x = (torch.randn(512, 768, device=DEV) * 2).bfloat16()
  q, inv = fp8.quantize_e4m3(x)
  amax = x.float().abs().max()
  assert abs(inv.item() - amax.item() / 448.0) < 1e-6 * amax.item()
  ref_q = (x.float() * (448.0 / amax)).to(torch.float8_e4m3fn)
  assert torch.equal(q.view(torch.float8_e4m3fn).float(), ref_q.float())
  for (M, N, K) in ((512, 768, 1024), (1024, 1600, 1600), (300, 520, 272)):
    a = torch.randn(M, K, device=DEV).bfloat16()
    w = (torch.randn(N, K, device=DEV) * 0.05).bfloat16()
    b = torch.randn(N, device=DEV).bfloat16()
    y = fp8.gemm_fp8(a, w, bias=b, epilogue=L.EPI_BIAS)
    aq, sa = fp8.quantize_e4m3(a)
    wq, sw = fp8.quantize_e4m3(w)
    exact = (aq.view(torch.float8_e4m3fn).float() @ wq.view(torch.float8_e4m3fn).float().t()) * (sa * sw) + b.float()
    full = a.float() @ w.float().t() + b.float()
    scale = full.abs().max().item()
    assert (y.float() - exact).abs().max().item() < 8e-3 * scale, (M, N, K)
    assert (y.float() - full).abs().max().item() < 0.08 * scale, (M, N, K)


def test_fp8_training_follows_bf16():
  """amp.level = fp8 (forward GEMMs in e4m3, backward bf16): same loss curve as bf16 within a few percent over 40 steps."""
  import easyparallellibrary_b200 as epl
  from easyparallellibrary_b200.models.gpt2 import GPT2, GPT2Config
  curves = {}
  for level in ("bf16", "fp8"):
    torch.manual_seed(0)
    epl.init(epl.Config({"amp.level": level}))
    with epl.replicate(1):
      model = GPT2(GPT2Config(vocab_size=2048, n_positions=128, n_embd=512, n_layer=2, n_head=8))
    tr = epl.Trainer(model, "adamw", lr=1e-3)
    g = torch.Generator().manual_seed(1)
    toks = torch.randint(0, 2048, (8, 128), generator=g).to(DEV)
    curves[level] = [tr.step(toks, toks).item() for _ in range(40)]
  from easyparallellibrary_b200.ops import fp8
  fp8.ENABLED = False
  assert curves["fp8"][-1] < 0.7 * curves["fp8"][0]
  import math
  for a, b in zip(curves["bf16"], curves["fp8"]):       # the curve falls by 3 orders of magnitude: compare on a log scale
    assert abs(math.log(max(a, 1e-3)) - math.log(max(b, 1e-3))) < 0.35, (curves["bf16"][::8], curves["fp8"][::8])


@pytest.mark.parametrize("layout", ["nt", "tn"])
def test_gemm_bf16_accumulate_matches_fp32(layout):
  """D += A B for a bf16 D (weight-gradient GEMMs of micro-batches 2..M): the old values are prefetched through the epilogue's
  aux path; must equal the fp32 sum rounded once."""
  from easyparallellibrary_b200.ops import linear as L
  torch.manual_seed(3)
  M, N, K = 1600, 768, 2048
  if layout == "nt":
    a, b = torch.randn(M, K, device=DEV).bfloat16(), (torch.randn(N, K, device=DEV) * 0.05).bfloat16()
    ref = a.float() @ b.float().t()
    kw = {}
  else:
    a, b = torch.randn(K, M, device=DEV).bfloat16(), (torch.randn(K, N, device=DEV) * 0.05).bfloat16()
    ref = a.float().t() @ b.float()
    kw = dict(a_mn_major=True, b_mn_major=True)
  old = torch.randn(M, N, device=DEV).bfloat16()
  out = old.clone()
  L.gemm(a, b, out=out, accumulate=True, **kw)
  expect = (ref + old.float())
  err = (out.float() - expect).abs().max().item()
  assert err < 2e-2 * expect.abs().max().item(), err
