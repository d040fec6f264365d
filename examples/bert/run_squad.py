"""BERT question answering (SQuAD-style) fine-tuning — the reference's flagship example (``examples/bert/run_squad.py``:
data pipeline, flags <-> EPL config keys, training, prediction and EM / F1 evaluation), rebuilt on EPL-B200.

There is no network in the sandbox, so ``--train_file`` / ``--predict_file`` are optional: without them a synthetic SQuAD-v1.1
shaped corpus (JSON in the official schema, written under ``--output_dir``) stands in; the real files work unchanged.  The
tokenizer is a self-contained lower-casing word-piece tokenizer whose vocabulary is built from the training corpus (or read
from ``--vocab_file``).

  python examples/bert/run_squad.py --model tiny --do_train --do_predict --num_train_steps 30
  torchrun --nproc-per-node 8 examples/bert/run_squad.py --model base --do_train --train_batch_size 12 --max_seq_length 384
  torchrun --nproc-per-node 8 examples/bert/run_squad.py --model large --num_pipe_stages 2 --num_micro_batch 10 --do_train
  torchrun --nproc-per-node 8 examples/bert/run_squad.py --model large --tensor_parallel 8 --do_train

Flags that are EPL config keys (reference run_squad.py:1171-1252): ``--num_micro_batch`` (pipeline.num_micro_batch),
``--num_pipe_stages``, ``--gc`` (gradient_checkpoint.type), ``--amp`` (amp.level), ``--zero`` (zero.level), ``--offload``,
``--io_slicing`` (io.slicing: every data-parallel replica reads its own shard of the feature files).
"""
import argparse
import collections
import json
import os
import random
import re
import string
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
import easyparallellibrary_b200 as epl
from easyparallellibrary_b200.models.bert import Bert, BertConfig, squad_loss
from easyparallellibrary_b200.runtime.saver import load_checkpoint, save_checkpoint
from easyparallellibrary_b200.utils.dataset import ShardedFileDataset


# ------------------------------------------------------------------------------------------------ data
SquadExample = collections.namedtuple("SquadExample", "qas_id question doc_tokens answer_text start_word end_word")
Features = collections.namedtuple("Features", "unique_id example_index tokens token_to_word input_ids input_mask segment_ids start end")


def synthetic_squad(path: str, n_paragraphs: int, seed: int) -> str:
  """A SQuAD-v1.1 shaped JSON file: paragraphs of pseudo-words, questions that quote the words around the answer span."""
  rnd = random.Random(seed)
  vocab = ["".join(rnd.choice(string.ascii_lowercase) for _ in range(rnd.randint(3, 8))) for _ in range(600)]
  data = []
  for pi in range(n_paragraphs):
    words = [rnd.choice(vocab) for _ in range(rnd.randint(60, 140))]
    context = " ".join(words)
    qas = []
    for qi in range(3):
      s = rnd.randint(3, len(words) - 6)
      e = s + rnd.randint(0, 2)
      answer = " ".join(words[s:e + 1])
      start_char = len(" ".join(words[:s])) + 1
      question = "which words follow " + " ".join(words[s - 3:s]) + " ?"
      qas.append({"id": "q%d_%d" % (pi, qi), "question": question, "answers": [{"text": answer, "answer_start": start_char}]})
    data.append({"title": "doc%d" % pi, "paragraphs": [{"context": context, "qas": qas}]})
  os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
  with open(path, "w") as f:
    json.dump({"version": "1.1", "data": data}, f)
  return path


def read_squad_examples(path: str):
  examples = []
  for article in json.load(open(path))["data"]:
    for para in article["paragraphs"]:
      text = para["context"]
      doc_tokens, char_to_word, prev_space = [], [], True
      for c in text:
        if c.isspace():
          prev_space = True
        else:
          if prev_space:
            doc_tokens.append(c)
          else:
            doc_tokens[-1] += c
          prev_space = False
        char_to_word.append(len(doc_tokens) - 1)
      for qa in para["qas"]:
        ans = qa["answers"][0]
        s = char_to_word[ans["answer_start"]]
        e = char_to_word[min(ans["answer_start"] + len(ans["text"]) - 1, len(char_to_word) - 1)]
        examples.append(SquadExample(qa["id"], qa["question"], doc_tokens, ans["text"], s, e))
  return examples


class WordPieceTokenizer(object):
  """Lower-case, split on whitespace / punctuation, greedy longest-match word pieces over ``vocab``."""
  SPECIAL = ["[PAD]", "[UNK]", "[CLS]", "[SEP]"]

  def __init__(self, vocab):
    self.vocab = {t: i for i, t in enumerate(vocab)}

  @classmethod
  def build(cls, texts, size: int):
    counts = collections.Counter()
    for t in texts:
      for w in cls.basic(t):
        counts[w] += 1
        for k in range(1, len(w)):                      # suffix pieces so unseen words still decompose
          counts["##" + w[k:]] += 0.01
    chars = sorted({c for w in counts for c in w.replace("##", "")})
    vocab = cls.SPECIAL + chars + ["##" + c for c in chars]
    vocab += [w for w, _ in counts.most_common(max(size - len(vocab), 0)) if w not in set(vocab)]
    return cls(vocab[:max(size, len(cls.SPECIAL) + 2 * len(chars))])

  @staticmethod
  def basic(text):
    return re.findall(r"[a-z0-9]+|[^\sa-z0-9]", text.lower())

  def tokenize_word(self, w):
    out, i = [], 0
    while i < len(w):
      j = len(w)
      while j > i and ((w[i:j] if i == 0 else "##" + w[i:j]) not in self.vocab):
        j -= 1
      if j == i:
        return ["[UNK]"]
      out.append(w[i:j] if i == 0 else "##" + w[i:j])
      i = j
    return out

  def tokenize(self, text):
    return [p for w in self.basic(text) for p in self.tokenize_word(w)]

  def ids(self, tokens):
    return [self.vocab.get(t, 1) for t in tokens]


def convert_examples_to_features(examples, tok, max_seq_length, doc_stride, max_query_length, training):
  """Sliding windows over the document (reference run_squad.py convert_examples_to_features): every window is one feature."""
  feats, uid = [], 1000000000
  for ei, ex in enumerate(examples):
    q = tok.tokenize(ex.question)[:max_query_length]
    word_to_tok, tok_to_word, doc = [], [], []
    for wi, w in enumerate(ex.doc_tokens):
      word_to_tok.append(len(doc))
      for p in tok.tokenize(w):
        tok_to_word.append(wi)
        doc.append(p)
    ts = word_to_tok[ex.start_word]
    te = (word_to_tok[ex.end_word + 1] - 1) if ex.end_word + 1 < len(ex.doc_tokens) else len(doc) - 1
    room = max_seq_length - len(q) - 3
    start = 0
    while start < len(doc):
      length = min(room, len(doc) - start)
      tokens = ["[CLS]"] + q + ["[SEP]"] + doc[start:start + length] + ["[SEP]"]
      seg = [0] * (len(q) + 2) + [1] * (length + 1)
      off = len(q) + 2
      t2w = {off + i: tok_to_word[start + i] for i in range(length)}
      if training:
        inside = ts >= start and te < start + length
        s_pos, e_pos = (ts - start + off, te - start + off) if inside else (0, 0)
      else:
        s_pos = e_pos = -1
      ids = tok.ids(tokens)
      pad = max_seq_length - len(ids)
      # input_mask: 1 for real tokens, 0 for padding (right-padded, as models/bert.py requires)
      feats.append(Features(uid, ei, tokens, t2w, ids + [0] * pad, [1] * len(ids) + [0] * pad, seg + [0] * pad, s_pos, e_pos))
      uid += 1
      if start + length >= len(doc):
        break
      start += min(length, doc_stride)
  return feats


def stack_features(chunk):
  """The model input of a list of features: ``[N, 3, S]`` = (input_ids, input_mask, segment_ids), see models/bert.py."""
  return torch.tensor([[f.input_ids, f.input_mask, f.segment_ids] for f in chunk])


def write_feature_files(feats, directory, per_file):
  """Features are written as several files so ``io.slicing`` has something to shard (the reference shards TFRecords)."""
  os.makedirs(directory, exist_ok=True)
  files = []
  for i in range(0, len(feats), per_file):
    path = os.path.join(directory, "features-%05d.pt" % (i // per_file))
    chunk = feats[i:i + per_file]
    torch.save({"features": stack_features(chunk), "start": torch.tensor([f.start for f in chunk]),
                "end": torch.tensor([f.end for f in chunk])}, path)
    files.append(path)
  return files


def read_feature_file(path):
  """Yields ``([3, S] features, start, end)`` per feature."""
  d = torch.load(path)
  for i in range(d["features"].shape[0]):
    yield d["features"][i], d["start"][i], d["end"][i]


# ------------------------------------------------------------------------------------------------ evaluation
def normalize_answer(s):
  s = "".join(ch for ch in s.lower() if ch not in set(string.punctuation))
  return " ".join(re.sub(r"\b(a|an|the)\b", " ", s).split())


def f1_score(pred, truth):
  p, t = normalize_answer(pred).split(), normalize_answer(truth).split()
  common = collections.Counter(p) & collections.Counter(t)
  same = sum(common.values())
  if same == 0:
    return 0.0
  prec, rec = same / len(p), same / len(t)
  return 2 * prec * rec / (prec + rec)


def predict(trainer, examples, feats, batch_size, max_answer_length=30):
  """Best (start, end) span per example over all of its windows -> answer text -> EM / F1 (official SQuAD-v1.1 metrics)."""
  best = {}
  for i in range(0, len(feats), batch_size):
    chunk = feats[i:i + batch_size]
    logits = trainer.eval_step(stack_features(chunk))
    if logits is None:                                   # pipeline: only the last stage sees the logits
      continue
    logits = logits.float().cpu()
    for f, lg in zip(chunk, logits):
      s_log, e_log = lg[:, 0], lg[:, 1]
      cand = sorted(f.token_to_word)
      for s in sorted(cand, key=lambda k: -s_log[k])[:10]:
        for e in sorted(cand, key=lambda k: -e_log[k])[:10]:
          if s <= e < s + max_answer_length:
            score = float(s_log[s] + e_log[e])
            if score > best.get(f.example_index, (-1e30,))[0]:
              best[f.example_index] = (score, f.token_to_word[s], f.token_to_word[e])
  import torch.distributed as dist
  if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
    # under pipeline parallelism only the last stage of a replica sees the logits: merge every rank's best spans
    parts = [None] * dist.get_world_size()
    dist.all_gather_object(parts, best)
    best = {}
    for part in parts:
      for k, v in part.items():
        if v[0] > best.get(k, (-1e30,))[0]:
          best[k] = v
  em = f1 = 0.0
  for ei, ex in enumerate(examples):
    if ei in best:
      _, ws, we = best[ei]
      pred = " ".join(ex.doc_tokens[ws:we + 1])
      em += float(normalize_answer(pred) == normalize_answer(ex.answer_text))
      f1 += f1_score(pred, ex.answer_text)
  n = max(len(examples), 1)
  return {"exact_match": 100.0 * em / n, "f1": 100.0 * f1 / n, "examples": len(examples), "predicted": len(best)}


# ------------------------------------------------------------------------------------------------ main
def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--model", default="base", help="tiny | base | large")
  ap.add_argument("--train_file", default="")
  ap.add_argument("--predict_file", default="")
  ap.add_argument("--vocab_file", default="")
  ap.add_argument("--output_dir", default="/tmp/epl_squad")
  ap.add_argument("--do_train", action="store_true")
  ap.add_argument("--do_predict", action="store_true")
  ap.add_argument("--max_seq_length", type=int, default=384)
  ap.add_argument("--doc_stride", type=int, default=128)
  ap.add_argument("--max_query_length", type=int, default=64)
  ap.add_argument("--train_batch_size", type=int, default=12)
  ap.add_argument("--predict_batch_size", type=int, default=8)
  ap.add_argument("--learning_rate", type=float, default=3e-5)
  ap.add_argument("--num_train_steps", type=int, default=100)
  ap.add_argument("--warmup_proportion", type=float, default=0.1, help="linear warm-up over this share of the steps, then linear decay to 0")
  ap.add_argument("--save_checkpoints_steps", type=int, default=0)
  ap.add_argument("--resume", action="store_true")
  ap.add_argument("--synthetic_paragraphs", type=int, default=60)
  # EPL config keys
  ap.add_argument("--num_micro_batch", type=int, default=1)
  ap.add_argument("--num_pipe_stages", type=int, default=1)
  ap.add_argument("--tensor_parallel", type=int, default=1)
  ap.add_argument("--gc", default="", help="'' | collection | auto")
  ap.add_argument("--amp", default="bf16", help="'' | O1 | bf16 | fp8")
  ap.add_argument("--zero", default="")
  ap.add_argument("--offload", default="")
  ap.add_argument("--io_slicing", action="store_true")
  ap.add_argument("--auto_parallel", action="store_true",
                  help="let the planner cut the layer stack into --num_pipe_stages stages (reference run_squad_auto_pipe.py)")
  args = ap.parse_args()
  rank = int(os.environ.get("RANK", 0))
  if args.model == "tiny":
    args.max_seq_length, args.doc_stride, args.max_query_length = min(args.max_seq_length, 96), 32, 24

  epl.init(epl.Config({"pipeline.num_micro_batch": args.num_micro_batch, "gradient_checkpoint.type": args.gc,
                       "amp.level": args.amp if torch.cuda.is_available() else "", "zero.level": args.zero,
                       "offload.level": args.offload, "io.slicing": args.io_slicing,
                       "auto.auto_parallel": args.auto_parallel,
                       "pipeline.num_stages": args.num_pipe_stages if args.auto_parallel else -1,
                       "cluster.colocate_split_and_replicate": args.tensor_parallel > 1}))
  if args.tensor_parallel > 1:
    epl.set_default_strategy(epl.replicate(device_count=1))

  train_file = args.train_file or synthetic_squad(os.path.join(args.output_dir, "train-synthetic.json"), args.synthetic_paragraphs, 0)
  predict_file = args.predict_file or synthetic_squad(os.path.join(args.output_dir, "dev-synthetic.json"), max(args.synthetic_paragraphs // 6, 4), 1)
  train_examples = read_squad_examples(train_file)
  bcfg = BertConfig.named(args.model, num_pipeline_stages=1 if args.auto_parallel else args.num_pipe_stages,
                          tensor_parallel=args.tensor_parallel,
                          max_position_embeddings=max(512, args.max_seq_length))
  if args.vocab_file:
    tok = WordPieceTokenizer([l.rstrip("\n") for l in open(args.vocab_file)])
  else:
    tok = WordPieceTokenizer.build([" ".join(e.doc_tokens) + " " + e.question for e in train_examples], min(bcfg.vocab_size, 8000))
  assert len(tok.vocab) <= bcfg.vocab_size

  model = Bert(bcfg)
  loss_fn = squad_loss if (args.num_pipe_stages > 1 or args.auto_parallel) else None
  from easyparallellibrary_b200.runtime.lr_schedule import warmup_linear_decay
  schedule = warmup_linear_decay(args.learning_rate, args.num_train_steps, int(args.warmup_proportion * args.num_train_steps))
  trainer = epl.Trainer(model, "adamw", lr=schedule, weight_decay=0.01, loss_fn=loss_fn).build()   # reference optimization.py:29-58
  if args.resume and os.path.exists(os.path.join(args.output_dir, "ckpt")):
    step0 = load_checkpoint(trainer, os.path.join(args.output_dir, "ckpt"))
    if rank == 0:
      print("resumed from step %d" % step0, flush=True)

  if args.do_train:
    feats = convert_examples_to_features(train_examples, tok, args.max_seq_length, args.doc_stride, args.max_query_length, True)
    random.Random(12345).shuffle(feats)
    files = write_feature_files(feats, os.path.join(args.output_dir, "train_features_rank%d" % rank), per_file=64)
    ds = ShardedFileDataset(files, read_feature_file, shuffle=True, seed=rank if not args.io_slicing else 0)
    batch = args.train_batch_size * args.num_micro_batch
    step, epoch = trainer.global_step, 0
    while step < args.num_train_steps:
      ds.set_epoch(epoch)
      loader = torch.utils.data.DataLoader(ds, batch_size=batch, drop_last=True)
      for features, s, e in loader:
        out = trainer.step(features, s, e)
        if rank == 0 and (step % 10 == 0 or step < 3):
          print("step %d loss %.4f" % (step, float(out.loss)), flush=True)
        step += 1
        if args.save_checkpoints_steps and step % args.save_checkpoints_steps == 0:
          save_checkpoint(trainer, os.path.join(args.output_dir, "ckpt"))
        if step >= args.num_train_steps:
          break
      epoch += 1
    save_checkpoint(trainer, os.path.join(args.output_dir, "ckpt"))

  if args.do_predict:
    dev_examples = read_squad_examples(predict_file)
    dev_feats = convert_examples_to_features(dev_examples, tok, args.max_seq_length, args.doc_stride, args.max_query_length, False)
    metrics = predict(trainer, dev_examples, dev_feats, args.predict_batch_size)
    if rank == 0:
      print("eval " + json.dumps(metrics), flush=True)
      with open(os.path.join(args.output_dir, "eval_results.json"), "w") as f:
        json.dump(metrics, f)
  epl.shutdown()


if __name__ == "__main__":
  main()
