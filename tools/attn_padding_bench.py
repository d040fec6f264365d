"""Cost of key-padding lengths (``kv_len``) on one GPU: attention fwd + bwd (csrc/attention.cu) and BERT-large training steps.

  python tools/attn_padding_bench.py [--iters 50] [--steps 10]

Attention at the BERT-large shape (B 32, S 384, H 16) and the GPT-2-XL shape (B 8, S 1024, H 25), non-causal, three cases: no
lengths, all lengths = S, seeded lengths uniform in [S/4, S].  BERT-large training steps (bf16, whole-step CUDA graph) at the
same two (B, S), with [B, S] ids and with [B, 3, S] features whose masks have the seeded lengths.  Times are CUDA events over
many launches after a warm-up; the card name and power limit are printed with them.  Prints one JSON line per measurement.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch


def card():
  try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                       timeout=30).stdout.strip().splitlines()[0]
  except Exception as e:  # pragma: no cover - reported, not hidden
    q = "nvidia-smi unavailable (%s)" % e
  return q


def lengths(B, S, seed):
  g = torch.Generator().manual_seed(seed)
  return torch.randint(S // 4, S + 1, (B,), generator=g, dtype=torch.int64).to(torch.int32)


def time_ms(fn, iters, warmup=5):
  for _ in range(warmup):
    fn()
  torch.cuda.synchronize()
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  a.record()
  for _ in range(iters):
    fn()
  b.record()
  torch.cuda.synchronize()
  return a.elapsed_time(b) / iters


def bench_attention(B, S, H, iters):
  from easyparallellibrary_b200.ops.attention_kernel import flash_attention_packed
  torch.manual_seed(0)
  qkv = (torch.randn(B, S, 3, H, 64, device="cuda") * 0.8).bfloat16().requires_grad_()
  dout = torch.randn(B, S, H * 64, device="cuda").bfloat16()
  seeded = lengths(B, S, 0).cuda()
  cases = {"none": None, "all_S": torch.full((B,), S, dtype=torch.int32, device="cuda"), "uniform_S/4_S": seeded}
  live = sum((int(n) + 127) // 128 for n in seeded.tolist()) / (B * ((S + 127) // 128))
  rows = []
  for name, kv_len in cases.items():
    def step():
      qkv.grad = None
      flash_attention_packed(qkv, False, kv_len).backward(dout)
    rows.append({"bench": "attention_fwd_bwd", "B": B, "S": S, "H": H, "lengths": name, "ms": round(time_ms(step, iters), 4),
                 "live_key_tile_share": round(live, 3) if name.startswith("uniform") else 1.0})
  return rows


def bench_bert(B, S, steps):
  import easyparallellibrary_b200 as epl
  from easyparallellibrary_b200.models.bert import Bert, BertConfig, squad_loss
  rows = []
  for masked in (False, True):
    epl.init(epl.Config({"amp.level": "bf16"}), init_process_group=False)
    torch.manual_seed(1234)
    with torch.device("cuda"):
      model = Bert(BertConfig.named("large", max_position_embeddings=max(512, S)))
    tr = epl.Trainer(model, "adamw", lr=1e-4, weight_decay=0.01, loss_fn=squad_loss, cuda_graph=True).build()
    g = torch.Generator().manual_seed(5)
    ids = torch.randint(0, 30000, (B, S), generator=g)
    start, end = torch.randint(0, S // 4, (B,), generator=g), torch.randint(0, S // 4, (B,), generator=g)
    if masked:
      mask = (torch.arange(S)[None] < lengths(B, S, 0).long()[:, None]).long()
      x = torch.stack([ids * mask, mask, torch.zeros_like(ids)], 1)
    else:
      x = ids
    batch = [t.cuda() for t in (x, start, end)]
    ms = time_ms(lambda: tr.step(*batch), steps, warmup=3)
    rows.append({"bench": "bert_large_train_step", "B": B, "S": S, "masked": masked, "ms": round(ms, 3),
                 "graphed": tr._graphed is not None and tr._graphed.graph is not None and not tr._graphed.failed})
    del tr, model
    torch.cuda.empty_cache()
  return rows


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--iters", type=int, default=50)
  ap.add_argument("--steps", type=int, default=10)
  ap.add_argument("--no-bert", action="store_true")
  args = ap.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit("attn_padding_bench.py needs a GPU")
  from easyparallellibrary_b200.ops import _lib
  _lib.require()
  print(json.dumps({"card": card(), "torch": torch.__version__}), flush=True)
  for B, S, H in ((32, 384, 16), (8, 1024, 25)):
    for row in bench_attention(B, S, H, args.iters):
      print(json.dumps(row), flush=True)
  if not args.no_bert:
    for B, S in ((32, 384), (8, 1024)):
      for row in bench_bert(B, S, args.steps):
        print(json.dumps(row), flush=True)
  print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
  main()
