"""Spawn ``world`` CPU processes running ``fn(rank, world, *args)`` under a gloo process group."""
import os
import socket
import traceback

import torch.multiprocessing as mp


def _free_port():
  s = socket.socket()
  s.bind(("127.0.0.1", 0))
  port = s.getsockname()[1]
  s.close()
  return port


def _entry(rank, world, port, fn, args, queue, env):
  os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), LOCAL_WORLD_SIZE=str(world),
                    MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
  os.environ.update(env or {})
  try:
    res = fn(rank, world, *args)
    queue.put((rank, "ok", res))
  except Exception:
    queue.put((rank, "err", traceback.format_exc()))
  finally:
    try:
      import torch.distributed as dist
      if dist.is_initialized():
        dist.destroy_process_group()
    except Exception:
      pass


def run_distributed(fn, world, args=(), env=None, timeout=180):
  """One retry for failures of the host rather than of the code under test: a rendezvous port taken between probing and
  binding, or a worker that never reported because the box was overloaded."""
  import queue as _queue
  try:
    return _run_once(fn, world, args, env, timeout)
  except _queue.Empty:
    return _run_once(fn, world, args, env, 2 * timeout)
  except AssertionError as e:
    if "Address already in use" in str(e) or "EADDRINUSE" in str(e):
      return _run_once(fn, world, args, env, timeout)
    raise


def _run_once(fn, world, args, env, timeout):
  ctx = mp.get_context("spawn")
  q = ctx.Queue()
  port = _free_port()
  procs = [ctx.Process(target=_entry, args=(r, world, port, fn, args, q, env)) for r in range(world)]
  # the workers inherit the environment at start: with no visible GPU the library takes its CPU path (gloo, CPU tensors) on any
  # machine, instead of placing every rank on the same device of a one-GPU box
  visible = os.environ.get("CUDA_VISIBLE_DEVICES")
  os.environ["CUDA_VISIBLE_DEVICES"] = ""
  try:
    for p in procs:
      p.start()
  finally:
    if visible is None:
      del os.environ["CUDA_VISIBLE_DEVICES"]
    else:
      os.environ["CUDA_VISIBLE_DEVICES"] = visible
  results = {}
  try:
    for _ in range(world):
      rank, status, payload = q.get(timeout=timeout)
      if status != "ok":
        raise AssertionError("rank %d failed:\n%s" % (rank, payload))
      results[rank] = payload
  finally:
    for p in procs:
      p.join(timeout=20)
      if p.is_alive():
        p.kill()
  return [results[r] for r in range(world)]
