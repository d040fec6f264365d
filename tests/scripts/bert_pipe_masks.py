"""2-stage 1F1B BERT (head dim 64, bf16) on 2 GPUs whose two micro-batches carry different key-padding masks; prints the
losses as JSON on rank 0.  Run once with EPL_PIPE_GRAPH=1 (stage CUDA graphs) and once with EPL_PIPE_GRAPH=0 (eager): the
graphs must replay each micro-batch's own mask, so both runs print the same losses."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch

import easyparallellibrary_b200 as epl
from easyparallellibrary_b200.models.bert import Bert, BertConfig, squad_loss


def main():
  epl.init(epl.Config({"pipeline.num_micro_batch": 2, "amp.level": "bf16"}))
  torch.manual_seed(0)
  model = Bert(BertConfig.named("tiny", hidden_size=256, num_attention_heads=4, intermediate_size=512, num_pipeline_stages=2))
  tr = epl.Trainer(model, "adamw", lr=1e-3, loss_fn=squad_loss).build()
  g = torch.Generator().manual_seed(1)
  B, S = 4, 256
  losses = []
  for step in range(4):
    ids = torch.randint(0, 1000, (B, S), generator=g)
    lens = torch.randint(S // 4, S + 1, (B,), generator=g)
    lens[step % B] = 1 + 127 * step                      # per micro-batch: different masks, including tile-boundary lengths
    mask = (torch.arange(S)[None] < lens[:, None]).long()
    seg = (torch.arange(S)[None] >= (lens[:, None] // 3)).long() * mask
    feats = torch.stack([ids * mask + 5 * (1 - mask), mask, seg], 1)
    start = torch.minimum(torch.randint(0, S, (B,), generator=g), lens - 1)
    end = torch.minimum(start + 3, lens - 1)
    losses.append(float(tr.step(feats, start, end).loss))
  if int(os.environ.get("RANK", "0")) == 0:
    print("LOSSES " + json.dumps(losses), flush=True)
  epl.shutdown()


if __name__ == "__main__":
  main()
