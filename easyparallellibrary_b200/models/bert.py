"""BERT encoder (base / large) — the reference's pipeline and tensor-parallel workload
(``examples/bert``: BERT-base DP batch 12 x seq 384; BERT-large 2-stage pipeline, 10 micro-batches;
``BASELINE.json``: BERT-large ``epl.split(8)``).

Post-LN transformer encoder + a span-classification (SQuAD) head.  ``tensor_parallel=True`` builds every layer's
attention and MLP from column/row-parallel pairs with token-sharded activations in between, i.e. the
all-gather->GEMM and GEMM->reduce-scatter fused kernels carry all TP traffic.  ``num_pipeline_stages`` cuts the
layer stack with ``epl.set_default_strategy`` exactly like ``examples/bert/modeling.py:829-834``.

Model input: either token ids ``[B, S]`` (every position is a real token, segment 0 everywhere), or the SQuAD features
``[B, 3, S]`` = ``stack(input_ids, input_mask, segment_ids)`` along dim 1.  ``input_mask`` must be right-padded (ones, then
zeros), as every BERT feature pipeline produces it: attention sees it as a key length per sequence, ``input_mask.sum(-1)``, so
padded keys are masked while padded query rows are still computed (their outputs are ignored by the loss).  The features travel
as ONE tensor, so ``loss_fn(out, start, end)``, ``eval_step(features)`` and micro-batch splitting treat them like the ids.
Layers after the embeddings read the mask from ``epl.current_micro_batch()[0]``.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch
from torch import nn

from easyparallellibrary_b200.ops.attention import attention
from easyparallellibrary_b200.ops.layernorm import LayerNorm
from easyparallellibrary_b200.ops.linear import Linear, mlp


@dataclass
class BertConfig:
  vocab_size: int = 30528
  hidden_size: int = 768
  num_hidden_layers: int = 12
  num_attention_heads: int = 12
  intermediate_size: int = 3072
  max_position_embeddings: int = 512
  type_vocab_size: int = 2
  num_pipeline_stages: int = 1
  tensor_parallel: int = 1

  @staticmethod
  def named(name: str, **kw) -> "BertConfig":
    table = {"tiny": dict(hidden_size=128, num_hidden_layers=2, num_attention_heads=4, intermediate_size=512, vocab_size=1024),
             "base": {}, "large": dict(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096)}
    cfg = dict(table[name])
    cfg.update(kw)
    return BertConfig(**cfg)

  def flops_per_token(self, seq_len: int) -> float:
    d, L, f = self.hidden_size, self.num_hidden_layers, self.intermediate_size
    return 3.0 * L * (8 * d * d + 4 * d * f + 4 * seq_len * d)


def split_features(features: torch.Tensor):
  """``[B, S]`` ids -> ``(ids, None, None)``; ``[B, 3, S]`` features -> ``(input_ids, input_mask, segment_ids)``."""
  if features.dim() == 3:
    if features.shape[1] != 3:
      raise ValueError("BERT features must be [B, S] ids or [B, 3, S] (input_ids, input_mask, segment_ids), got %s"
                       % (tuple(features.shape),))
    return features[:, 0], features[:, 1], features[:, 2]
  return features, None, None


def sequence_and_key_lengths():
  """``(S, kv_len)`` of the micro-batch being executed: ``kv_len`` is the int32 ``[B]`` count of ones in the (right-padded)
  ``input_mask``, or ``None`` for plain ``[B, S]`` ids (no padding)."""
  import easyparallellibrary_b200 as epl
  ids, mask, _ = split_features(epl.current_micro_batch()[0])
  return ids.shape[1], (None if mask is None else mask.sum(-1, dtype=torch.int32))


class BertEmbeddings(nn.Module):
  def __init__(self, cfg: BertConfig):
    super().__init__()
    self.word = nn.Embedding(cfg.vocab_size, cfg.hidden_size)
    self.pos = nn.Embedding(cfg.max_position_embeddings, cfg.hidden_size)
    self.typ = nn.Embedding(cfg.type_vocab_size, cfg.hidden_size)
    self.ln = LayerNorm(cfg.hidden_size, eps=1e-12)
    for e in (self.word, self.pos, self.typ):
      nn.init.normal_(e.weight, std=0.02)

  def forward(self, features):
    ids, _, seg = split_features(features)
    pos = torch.arange(ids.shape[1], device=ids.device)
    if seg is None:
      return self.ln(self.word(ids) + self.pos(pos) + self.typ.weight[0])
    return self.ln(self.word(ids) + self.pos(pos) + self.typ(seg))


class BertLayer(nn.Module):
  def __init__(self, cfg: BertConfig):
    super().__init__()
    d = cfg.hidden_size
    self.heads = cfg.num_attention_heads
    self.qkv = Linear(d, 3 * d, init_std=0.02)
    self.proj = Linear(d, d, init_std=0.02)
    self.ln1 = LayerNorm(d, eps=1e-12)
    self.fc = Linear(d, cfg.intermediate_size, init_std=0.02)
    self.out = Linear(cfg.intermediate_size, d, init_std=0.02)
    self.ln2 = LayerNorm(d, eps=1e-12)

  def forward(self, x):
    B, S, d = x.shape
    from easyparallellibrary_b200.ops.attention import attention_packed
    from easyparallellibrary_b200.ops.linear import linear
    _, kv_len = sequence_and_key_lengths()
    a = attention_packed(self.qkv(x).view(B, S, 3, self.heads, d // self.heads), causal=False, kv_len=kv_len)
    x = self.ln1(linear(a, self.proj.weight, self.proj.bias, residual=x))
    return self.ln2(mlp(x, self.fc.weight, self.fc.bias, self.out.weight, self.out.bias, residual=x))


class BertLayerTP(nn.Module):
  """Tensor-parallel layer on token shards ``[T/N, d]`` (T = batch x seq tokens of the whole TP group)."""

  def __init__(self, cfg: BertConfig, split):
    super().__init__()
    from easyparallellibrary_b200.ops import tensor_parallel as tp
    d, n = cfg.hidden_size, cfg.tensor_parallel
    self.split = split
    self.heads_local = cfg.num_attention_heads // n
    self.head_dim = d // cfg.num_attention_heads
    with split:
      self.qkv = tp.ColumnParallelLinear(d, 3 * d, init_std=0.02)
      self.proj = tp.RowParallelLinear(d, d, init_std=0.02)
      self.fc = tp.ColumnParallelLinear(d, cfg.intermediate_size, gelu=True, init_std=0.02)
      self.out = tp.RowParallelLinear(cfg.intermediate_size, d, init_std=0.02)
    self.ln1 = LayerNorm(d, eps=1e-12)
    self.ln2 = LayerNorm(d, eps=1e-12)
    self.seq_len = None

  def forward(self, x_shard):                      # [T/N, d]
    S, kv_len = sequence_and_key_lengths()         # token shards carry no sequence shape: it comes from the micro-batch
    if self.seq_len is not None:
      S = self.seq_len
    qkv = self.qkv(x_shard)                        # [T, 3d/N]  (all-gather -> GEMM)
    T = qkv.shape[0]                               # the TP group's whole batch: T // S sequences, one length each
    from easyparallellibrary_b200.ops.attention import attention_packed
    a = attention_packed(qkv.view(T // S, S, 3, self.heads_local, self.head_dim), causal=False, kv_len=kv_len).reshape(T, -1)
    x_shard = self.ln1(x_shard + self.proj(a))     # GEMM -> reduce-scatter
    return self.ln2(x_shard + self.out(self.fc(x_shard)))


class _TokenShard(nn.Module):
  """[B, S, d] -> this TP rank's token shard [B*S/N, d] (every rank of the split group holds the same batch)."""

  def __init__(self, split):
    super().__init__()
    self.split = split

  def forward(self, x):
    from easyparallellibrary_b200.ops.tensor_parallel import current_tp_group
    g = current_tp_group(self.split)
    B, S, d = x.shape
    return x.reshape(B * S, d).chunk(g.size, 0)[g.rank].contiguous()


class _TokenGather(nn.Module):
  """Token shard [B*S/N, d] -> [B, S, d] (all-gather forward, reduce-scatter backward)."""
  epl_collective = True

  def __init__(self, split):
    super().__init__()
    self.split = split

  def forward(self, x):
    from easyparallellibrary_b200.ops.tensor_parallel import current_tp_group
    g = current_tp_group(self.split)
    S, _ = sequence_and_key_lengths()
    full = _gather_tokens(x, g) if x.requires_grad else g.comm.allgather(x)
    return full.view(-1, S, full.shape[-1])


class SquadHead(nn.Module):
  def __init__(self, cfg: BertConfig):
    super().__init__()
    self.qa = nn.Linear(cfg.hidden_size, 2)

  def forward(self, x):
    return self.qa(x.float() if x.dtype != self.qa.weight.dtype else x)


def squad_loss(logits: torch.Tensor, start: torch.Tensor, end: torch.Tensor) -> torch.Tensor:
  s, e = logits.float().unbind(-1)
  ce = torch.nn.functional.cross_entropy
  return 0.5 * (ce(s, start) + ce(e, end))


class Bert(nn.Module):
  def __init__(self, cfg: BertConfig):
    super().__init__()
    import easyparallellibrary_b200 as epl
    self.cfg = cfg
    stages = max(cfg.num_pipeline_stages, 1)
    per = (cfg.num_hidden_layers + stages - 1) // stages
    if stages > 1:
      epl.set_default_strategy(epl.replicate(1, name="stage_0"))
    self.embed = BertEmbeddings(cfg)
    layers = []
    self._split = epl.split(device_count=cfg.tensor_parallel) if cfg.tensor_parallel > 1 else None
    # tensor parallel: the token sharding / gathering are blocks of their own, so a pipeline cut can fall anywhere between
    # layers and every stage still sees [tokens/N, d] activations (stage 0 owns the shard block, the last stage the gather)
    self.shard = _TokenShard(self._split) if self._split is not None else None
    for i in range(cfg.num_hidden_layers):
      if stages > 1 and i > 0 and i % per == 0:
        epl.set_default_strategy(epl.replicate(1, name="stage_%d" % (i // per)))
      layers.append(BertLayerTP(cfg, self._split) if self._split is not None else BertLayer(cfg))
    self.layers = nn.ModuleList(layers)
    self.gather = _TokenGather(self._split) if self._split is not None else None
    self.head = SquadHead(cfg)

  def epl_sequential(self):
    tp_in = [self.shard] if self.shard is not None else []
    tp_out = [self.gather] if self.gather is not None else []
    return [self.embed] + tp_in + list(self.layers) + tp_out + [self.head]

  def forward(self, features, start=None, end=None):
    """``features``: ``[B, S]`` token ids or ``[B, 3, S]`` (input_ids, input_mask, segment_ids), see the module docstring."""
    import easyparallellibrary_b200 as epl
    from easyparallellibrary_b200.ir.graph import Graph
    cur = epl.current_micro_batch()
    if cur is None or cur[0] is not features:               # called outside a Trainer step (plain module use)
      Graph.get().current_micro_batch = (features, start, end)
    x = features
    for block in self.epl_sequential():
      x = block(x)
    if start is None:
      return x
    return squad_loss(x, start, end)


def _gather_tokens(x, g):
  from easyparallellibrary_b200.communicators import functional as CF
  return CF.all_gather(x.contiguous(), g.comm)
