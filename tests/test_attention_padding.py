"""Key-padding lengths (``kv_len``) in the attention kernels and BERT's ``(input_ids, input_mask, segment_ids)`` features.

GPU tests check the tcgen05 kernels (csrc/attention.cu) against an fp32 reference, the no-length path bit for bit, and the
CUDA-graph / pipeline-graph replays; CPU tests check the SDPA path, BERT's masking and the multi-process engines."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from dist_utils import run_distributed

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "bert_tiny_ids_only.npz")
DEV = "cuda"
gpu = pytest.mark.gpu


def _close(a, b, rtol, atol, what=""):
  a, b = a.float(), b.float()
  err = (a - b).abs()
  tol = atol + rtol * b.abs()
  bad = (err > tol).float().mean().item()
  assert bad < 1e-3, "%s: %.4f%% elements out of tolerance, max err %.4g (ref max %.4g)" % (
      what, bad * 100, err.max().item(), b.abs().max().item())


def _padded_qkv(B, S, H, lens, seed=0):
  """bf16 [B, S, 3, H, 64] with large finite garbage in every row at or past the batch row's length."""
  g = torch.Generator(device=DEV).manual_seed(seed)
  qkv = torch.randn(B, S, 3, H, 64, device=DEV, generator=g) * 0.8
  garbage = (torch.rand(B, S, 3, H, 64, device=DEV, generator=g) * 2 - 1) * 1e3
  pad = torch.arange(S, device=DEV)[None, :] >= lens.to(DEV)[:, None]
  qkv = torch.where(pad[:, :, None, None, None], garbage, qkv)
  return qkv.bfloat16()


def _reference(qkv, dout, lens, causal):
  B, S, _, H, D = qkv.shape
  ref_in = qkv.detach().float().requires_grad_()
  q, k, v = ref_in.permute(2, 0, 3, 1, 4).unbind(0)
  s = q @ k.transpose(-1, -2) / math.sqrt(D)
  keys = torch.arange(S, device=qkv.device)
  vis = (keys[None, :] < lens.to(qkv.device).long()[:, None])[:, None, None, :]
  if causal:
    vis = vis & torch.ones(S, S, dtype=torch.bool, device=qkv.device).tril()
  s = s.masked_fill(~vis, float("-inf"))
  ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B, S, H * D)
  ref.backward(dout.float())
  return ref.detach(), ref_in.grad


def _fwd_bwd(qkv, dout, causal, kv_len):
  from easyparallellibrary_b200.ops.attention_kernel import flash_attention_packed
  x = qkv.detach().clone().requires_grad_()
  out = flash_attention_packed(x, causal, kv_len)
  out.backward(dout)
  return out.detach(), x.grad


# ------------------------------------------------------------------------------------------------ kernels (GPU)
@gpu
@pytest.mark.parametrize("causal", [True, False])
@pytest.mark.parametrize("B,S,H", [(4, 384, 4), (3, 1024, 2), (2, 4160, 2)])   # 4160: the backward takes three launches
def test_padded_attention_matches_fp32_reference(B, S, H, causal):
  """Forward and backward with key lengths 1, 127, 128, 129, a random one and S (in batches of B) vs fp32 softmax(QK^T)V with
  the same key mask; the padded Q/K/V rows hold large finite garbage, and the padded keys get exactly zero dK / dV."""
  r = int(torch.randint(2, S, (1,), generator=torch.Generator().manual_seed(S)))
  all_lens = [1, 127, 128, 129, r, S]
  for i in range(0, len(all_lens), B):
    lens = torch.tensor((all_lens[i:i + B] + [S] * B)[:B], dtype=torch.int32, device=DEV)
    qkv = _padded_qkv(B, S, H, lens, seed=i)
    dout = torch.randn(B, S, H * 64, device=DEV).bfloat16()
    out, grad = _fwd_bwd(qkv, dout, causal, lens)
    ref, gr = _reference(qkv, dout, lens, causal)
    what = "S=%d lens=%s causal=%d " % (S, lens.tolist(), causal)
    _close(out, ref, 2e-2, 2e-2, what + "out")
    for idx, name in enumerate(("dq", "dk", "dv")):
      _close(grad[:, :, idx], gr[:, :, idx], 3e-2, 3e-2 * gr[:, :, idx].abs().max().item(), what + name)
    for b, n in enumerate(lens.tolist()):
      assert bool((grad[b, n:, 1:] == 0).all()), what + "dK/dV of padded keys of row %d" % b


@gpu
@pytest.mark.parametrize("causal", [True, False])
@pytest.mark.parametrize("B,S,H", [(2, 1000, 3), (1, 4160, 2)])
def test_no_lengths_is_bitwise_unchanged(B, S, H, causal):
  """kv_len=None, kv_len all = S and the original epl_attn_fwd / epl_attn_bwd entry points give the same bits."""
  from easyparallellibrary_b200.ops import _lib
  from easyparallellibrary_b200.ops.attention_kernel import _lib_attn
  torch.manual_seed(0)
  qkv = (torch.randn(B, S, 3, H, 64, device=DEV) * 0.8).bfloat16()
  dout = torch.randn(B, S, H * 64, device=DEV).bfloat16()
  o_none, g_none = _fwd_bwd(qkv, dout, causal, None)
  o_full, g_full = _fwd_bwd(qkv, dout, causal, torch.full((B,), S, dtype=torch.int32, device=DEV))
  lib = _lib_attn()
  scale = 1.0 / math.sqrt(64)
  out = torch.empty(B, S, H, 64, dtype=torch.bfloat16, device=DEV)
  lse = torch.empty(B, H, S, dtype=torch.float32, device=DEV)
  _lib.check(lib.epl_attn_fwd(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), B, S, H, scale, int(causal), _lib.stream()), "fwd")
  dqkv = torch.empty_like(qkv)
  delta = torch.empty(B, H, S, dtype=torch.float32, device=DEV)
  dq_acc = torch.empty(lib.epl_attn_dq_slots(S), B, S, H, 64, dtype=torch.float32, device=DEV)
  _lib.check(lib.epl_attn_bwd(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), delta.data_ptr(), dq_acc.data_ptr(),
                              dqkv.data_ptr(), B, S, H, scale, int(causal), _lib.stream()), "bwd")
  torch.cuda.synchronize()
  assert torch.equal(o_none, o_full) and torch.equal(g_none, g_full)
  assert torch.equal(o_none, out.view(B, S, H * 64)) and torch.equal(g_none, dqkv)


@gpu
@pytest.mark.parametrize("causal", [True, False])
def test_padded_backward_is_bitwise_reproducible(causal):
  """Dead key tiles add nothing to their dQ slot: the backward with lengths still gives the same bits run after run."""
  for B, S, H in ((8, 1024, 4), (2, 4160, 2)):
    lens = torch.tensor(([1, 129, S, 700, 128, 1000, 3, S] if S == 1024 else [1500, S])[:B], dtype=torch.int32, device=DEV)
    qkv = _padded_qkv(B, S, H, lens)
    dout = torch.randn(B, S, H * 64, device=DEV).bfloat16()
    grads = [_fwd_bwd(qkv, dout, causal, lens)[1] for _ in range(3)]
    assert all(torch.equal(grads[0], g) for g in grads[1:]), (B, S, H)


@gpu
def test_cuda_graph_replays_with_refreshed_lengths():
  """fwd + bwd captured once; new contents of the length tensor between replays are honoured (no host read of the lengths)."""
  from easyparallellibrary_b200.ops.attention_kernel import flash_attention_packed
  B, S, H = 3, 640, 2
  torch.manual_seed(0)
  qkv = (torch.randn(B, S, 3, H, 64, device=DEV) * 0.8).bfloat16()
  dout = torch.randn(B, S, H * 64, device=DEV).bfloat16()
  kv_len = torch.tensor([S, 200, 1], dtype=torch.int32, device=DEV)
  x = qkv.clone().requires_grad_()

  def body():
    x.grad = None
    out = flash_attention_packed(x, False, kv_len)
    out.backward(dout)
    return out

  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(side):
    body()
  torch.cuda.current_stream().wait_stream(side)
  g = torch.cuda.CUDAGraph()
  with torch.cuda.graph(g):
    out_static = body()
  grad_static = x.grad
  for lens in ([S, 200, 1], [129, S, 640 - 1], [1, 1, 128]):
    kv_len.copy_(torch.tensor(lens, dtype=torch.int32))
    g.replay()
    torch.cuda.synchronize()
    o_ref, g_ref = _fwd_bwd(qkv, dout, False, torch.tensor(lens, dtype=torch.int32, device=DEV))
    assert torch.equal(out_static, o_ref) and torch.equal(grad_static, g_ref), lens


@gpu
def test_unpacked_attention_falls_back_to_sdpa_on_gpu():
  from easyparallellibrary_b200.ops import attention as A
  torch.manual_seed(0)
  q, k, v = (torch.randn(2, 3, 50, 64, device=DEV) for _ in range(3))
  lens = torch.tensor([50, 7], dtype=torch.int32, device=DEV)
  if A._IMPL == "epl":
    pytest.skip("EPL_ATTENTION=epl makes the unpacked call an error")
  for causal in (True, False):
    _close(A.attention(q, k, v, causal, kv_len=lens), A.attention_reference(q, k, v, causal, kv_len=lens), 1e-3, 1e-3, "sdpa")


def _tiny64(**kw):
  from easyparallellibrary_b200.models.bert import BertConfig
  return BertConfig.named("tiny", hidden_size=256, num_attention_heads=4, intermediate_size=512, **kw)


def _masked_batch(g, B, S, vocab=1000, garbage=None):
  lens = torch.randint(S // 4, S + 1, (B,), generator=g)
  lens[0] = min(129, S)
  mask = (torch.arange(S)[None] < lens[:, None]).long()
  seg = (torch.arange(S)[None] >= (lens[:, None] // 3)).long() * mask
  ids = torch.randint(0, vocab, (B, S), generator=g)
  ids = torch.where(mask.bool(), ids, torch.zeros_like(ids) if garbage is None else garbage)
  start = torch.minimum(torch.randint(0, S, (B,), generator=g), lens - 1)
  end = torch.minimum(start + 2, lens - 1)
  return torch.stack([ids, mask, seg], 1), start, end


@gpu
def test_bert_kernel_path_matches_sdpa_path(monkeypatch):
  """A BERT step on masked [B, 3, S] features: the tcgen05 kernel with key lengths vs torch SDPA with the same mask."""
  import easyparallellibrary_b200 as epl
  from easyparallellibrary_b200.models.bert import Bert, squad_loss
  from easyparallellibrary_b200.ops import attention as A
  from easyparallellibrary_b200.ops import attention_kernel
  calls = []
  real = attention_kernel.flash_attention_packed
  monkeypatch.setattr(attention_kernel, "flash_attention_packed", lambda qkv, causal=True, kv_len=None: (
      calls.append(kv_len is not None), real(qkv, causal, kv_len))[1])
  res = {}
  for impl in ("auto", "sdpa"):
    monkeypatch.setattr(A, "_IMPL", impl)
    torch.manual_seed(0)
    epl.init(epl.Config({"amp.level": "bf16"}))
    with epl.replicate(1):
      model = Bert(_tiny64())
    tr = epl.Trainer(model, "adamw", lr=1e-3, loss_fn=squad_loss)
    g = torch.Generator().manual_seed(1)
    batches = [_masked_batch(g, 4, 384) for _ in range(3)]
    losses = [tr.step(*b).item() for b in batches]
    logits = tr.eval_step(batches[0][0]).float()
    res[impl] = (losses, logits, batches[0][0][:, 1].bool().to(DEV))
  assert calls and all(calls)
  for a, b in zip(res["auto"][0], res["sdpa"][0]):
    assert abs(a - b) < 2e-2 * abs(b) + 1e-2, (res["auto"][0], res["sdpa"][0])
  valid = res["auto"][2]
  _close(res["auto"][1][valid], res["sdpa"][1][valid], 5e-2, 5e-2, "bert logits")


@gpu
def test_bert_whole_step_graph_follows_each_batch_mask():
  """The whole-step CUDA graph replays two differently masked batches like the eager step does."""
  import easyparallellibrary_b200 as epl
  from easyparallellibrary_b200.models.bert import Bert, squad_loss
  runs = {}
  for graph in (False, True):
    torch.manual_seed(0)
    epl.init(epl.Config({"amp.level": "bf16"}))
    with epl.replicate(1):
      model = Bert(_tiny64())
    tr = epl.Trainer(model, "adamw", lr=1e-3, loss_fn=squad_loss, cuda_graph=graph)
    g = torch.Generator().manual_seed(1)
    two = [_masked_batch(g, 4, 256) for _ in range(2)]
    runs[graph] = [tr.step(*two[i % 2]).item() for i in range(6)]
    if graph:
      assert tr._graphed is not None and tr._graphed.graph is not None and not tr._graphed.failed
  for a, b in zip(runs[False], runs[True]):
    assert abs(a - b) < 2e-3 * abs(a) + 1e-3, runs


@gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_pipeline_stage_graphs_replay_each_micro_batch_mask():
  """2-stage 1F1B BERT, two micro-batches with different masks: stage CUDA graphs give the eager losses."""
  out = {}
  for mode in ("1", "0"):
    env = dict(os.environ, EPL_PIPE_GRAPH=mode, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
      env.pop(k, None)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-port", "29641",
                        os.path.join(ROOT, "tests", "scripts", "bert_pipe_masks.py")], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    out[mode] = json.loads([l for l in r.stdout.splitlines() if l.startswith("LOSSES ")][-1][len("LOSSES "):])
  np.testing.assert_allclose(out["1"], out["0"], rtol=2e-3, atol=1e-3)


# ------------------------------------------------------------------------------------------------ SDPA path (CPU)
def _cpu_bert(**kw):
  import easyparallellibrary_b200 as epl
  from easyparallellibrary_b200.models.bert import Bert, BertConfig
  epl.init(epl.Config({}), init_process_group=False)
  torch.manual_seed(0)
  return Bert(BertConfig.named("tiny", **kw))


def test_padded_positions_do_not_reach_valid_outputs_or_weight_gradients():
  """Other ids / segment ids at padded positions: same outputs at valid positions, same weight gradients of a loss over them."""
  model = _cpu_bert()
  g = torch.Generator().manual_seed(3)
  feats, _, _ = _masked_batch(g, 3, 48)
  mask = feats[:, 1].bool()
  other = feats.clone()
  other[:, 0][~mask] = torch.randint(0, 1000, (int((~mask).sum()),), generator=g)
  other[:, 2][~mask] = 1
  w = torch.randn(3, 48, 2, generator=g)
  res = []
  for f in (feats, other):
    model.zero_grad()
    out = model(f)
    (out * w)[mask].sum().backward()
    res.append((out.detach()[mask], {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}))
  assert torch.allclose(res[0][0], res[1][0], rtol=1e-6, atol=1e-6)
  assert res[0][1].keys() == res[1][1].keys()
  for n in res[0][1]:
    assert torch.allclose(res[0][1][n], res[1][1][n], rtol=1e-5, atol=1e-6), n


def test_ids_only_input_is_unchanged():
  """[B, S] ids compute what they computed before features existed (recorded output), and match [B, 3, S] features with an
  all-ones mask and segment 0."""
  model = _cpu_bert()
  gold = np.load(GOLDEN)
  ids = torch.from_numpy(gold["ids"])
  out = model(ids).detach()
  np.testing.assert_allclose(out.numpy(), gold["logits"], rtol=1e-5, atol=1e-6)
  feats = torch.stack([ids, torch.ones_like(ids), torch.zeros_like(ids)], 1)
  assert torch.allclose(model(feats).detach(), out, rtol=1e-6, atol=1e-6)
  ref = model(ids).detach()
  assert torch.equal(out, ref)


def test_attention_with_lengths_matches_reference_on_cpu():
  from easyparallellibrary_b200.ops.attention import attention, attention_packed, attention_reference
  torch.manual_seed(0)
  B, H, S, D = 3, 2, 20, 16
  q, k, v = (torch.randn(B, H, S, D) for _ in range(3))
  lens = torch.tensor([20, 7, 1], dtype=torch.int32)
  for causal in (True, False):
    ref = attention_reference(q, k, v, causal, kv_len=lens)
    assert torch.allclose(attention(q, k, v, causal, kv_len=lens), ref, atol=1e-5)
    packed = torch.stack([q, k, v], 0).permute(1, 3, 0, 2, 4).contiguous()          # [B, S, 3, H, D]
    assert torch.allclose(attention_packed(packed, causal, kv_len=lens), ref.transpose(1, 2).reshape(B, S, H * D), atol=1e-5)
  assert torch.allclose(attention(q, k, v, False), attention_reference(q, k, v, False), atol=1e-5)
  # lengths are clamped to [1, S] like in the kernels
  assert torch.equal(attention(q, k, v, False, kv_len=torch.tensor([99, 0, -3], dtype=torch.int32)),
                     attention(q, k, v, False, kv_len=torch.tensor([20, 1, 1], dtype=torch.int32)))


# ------------------------------------------------------------------------------------------------ engines (CPU, gloo)
def _masked_steps(steps=3, B=4, S=32):
  g = torch.Generator().manual_seed(7)
  return [_masked_batch(g, B, S) for _ in range(steps)]


def _pipe_worker(rank, world, conf):
  import easyparallellibrary_b200 as epl
  from easyparallellibrary_b200.models.bert import Bert, BertConfig, squad_loss
  epl.init(epl.Config(conf))
  torch.manual_seed(0)
  model = Bert(BertConfig.named("tiny", num_hidden_layers=8, num_pipeline_stages=2))   # 4 layers a stage: recomputed
  tr = epl.Trainer(model, "adamw", lr=1e-2, loss_fn=squad_loss).build()
  losses = [tr.step(*b).item() for b in _masked_steps()]      # the two micro-batches of every step have different masks
  params = {}
  for s in tr.plan.local_stages:
    for k, v in tr.stage_modules[s].state_dict().items():
      params["%d.%s" % (s, k)] = v.float().numpy().copy()
  return losses, params, tr.plan.pipeline


def test_pipeline_with_recompute_uses_each_micro_batch_mask():
  """2-stage 1F1B with gradient checkpointing: the recomputed forward of micro-batch 0 runs after micro-batch 1's forward and
  must read micro-batch 0's mask.  Two processes match one process."""
  conf = {"pipeline.num_micro_batch": 2, "gradient_checkpoint.type": "auto"}
  base = run_distributed(_pipe_worker, 1, args=(conf,))[0]
  res = run_distributed(_pipe_worker, 2, args=(conf,))
  assert res[0][2] and res[1][2] and not base[2]
  merged = {}
  for r in res:
    merged.update(r[1])
  assert set(merged) == set(base[1])
  assert max(float(np.abs(merged[k] - base[1][k]).max()) for k in merged) < 1e-6
  np.testing.assert_allclose(res[0][0], base[0], rtol=0, atol=1e-6)


def _tp_worker(rank, world):
  """Bert tiny with split(world) (world = 1: the plain model) from the same full weights: losses of three masked batches."""
  import easyparallellibrary_b200 as epl
  from easyparallellibrary_b200.models.bert import Bert, BertConfig
  epl.init(epl.Config({}), init_process_group=False)
  torch.manual_seed(0)
  full = Bert(BertConfig.named("tiny"))                       # the full weights, built in a graph of their own
  epl.init(epl.Config({"cluster.colocate_split_and_replicate": True}))
  if world == 1:
    torch.manual_seed(0)
    model = Bert(BertConfig.named("tiny"))
  else:
    epl.set_default_strategy(epl.replicate(device_count=1))
    model = Bert(BertConfig.named("tiny", tensor_parallel=world))
    _load_tp_shards(model, full, rank, world)
  tr = epl.Trainer(model, "sgd", lr=0.1)
  return [float(tr.eval_step(*b)) for b in _masked_steps()]


def _load_tp_shards(tp_model, full, r, n):
  """Rank r's shards of the plain model's weights (QKV columns are [3, heads, head_dim] in both, per-rank heads under TP)."""
  with torch.no_grad():
    for name, p in tp_model.named_parameters():
      if not name.startswith("layers."):
        p.copy_(dict(full.named_parameters())[name])
    for lt, lf in zip(tp_model.layers, full.layers):
      d = lf.qkv.weight.shape[1]
      lt.qkv.weight.copy_(lf.qkv.weight.view(3, n, d // n, d)[:, r].reshape(-1, d))
      lt.qkv.bias.copy_(lf.qkv.bias.view(3, n, d // n)[:, r].reshape(-1))
      lt.proj.weight.copy_(lf.proj.weight.chunk(n, 1)[r]); lt.proj.bias.copy_(lf.proj.bias)
      lt.fc.weight.copy_(lf.fc.weight.chunk(n, 0)[r]); lt.fc.bias.copy_(lf.fc.bias.chunk(n, 0)[r])
      lt.out.weight.copy_(lf.out.weight.chunk(n, 1)[r]); lt.out.bias.copy_(lf.out.bias)
      for a in ("ln1", "ln2"):
        getattr(lt, a).load_state_dict(getattr(lf, a).state_dict())


def test_tensor_parallel_bert_with_masks_matches_one_process():
  """split(2): the key lengths apply to the TP group's whole batch (T // S sequences); the losses match the plain model's."""
  base = run_distributed(_tp_worker, 1)[0]
  for r in run_distributed(_tp_worker, 2):
    np.testing.assert_allclose(r, base, rtol=0, atol=1e-6)


def test_squad_example_features_carry_the_input_mask(tmp_path):
  """run_squad.py writes [3, S] (input_ids, input_mask, segment_ids) features, then trains and predicts on them."""
  env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), CUDA_VISIBLE_DEVICES="")
  for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "TF_CONFIG"):
    env.pop(k, None)
  r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "bert", "run_squad.py"), "--model", "tiny", "--do_train",
                      "--do_predict", "--num_train_steps", "3", "--train_batch_size", "4", "--synthetic_paragraphs", "8",
                      "--output_dir", str(tmp_path)], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
  assert r.returncode == 0 and "step 1 loss" in r.stdout and "eval " in r.stdout, r.stdout[-1500:] + r.stderr[-2500:]
  d = torch.load(os.path.join(str(tmp_path), "train_features_rank0", "features-00000.pt"))
  f = d["features"]
  assert f.dim() == 3 and f.shape[1] == 3
  mask = f[:, 1]
  assert set(mask.unique().tolist()) <= {0, 1} and (mask[:, 0] == 1).all()
  assert (mask[:, :-1] >= mask[:, 1:]).all()                     # right-padded
  assert bool((mask == 0).any())                                  # the synthetic windows do have padding
  assert bool((f[:, 0][mask == 0] == 0).all())                    # padded ids are [PAD]
  assert bool((f[:, 2] == 1).any())                               # segment ids of the document part
