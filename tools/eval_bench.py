"""Evaluation throughput of the AutoInt trainer at the headline geometry: B = 8192, 39 fields, 1 M rows per field,
bf16.  Prints one JSON line (rank 0) with, per layout, three measurements alternated in rounds in this one process:

  eval      AutoIntTrainer.evaluate() over `--eval-batches` device batches: the captured eval step (forward-only
            tcgen05 tower, metrics and loss in the graph) plus the per-batch loss read-back; samples/s, host clock
            around the whole call (it ends in a synchronise);
  predict   the eager path it replaces: predict() + BinaryMetrics.update_state per batch, then result(); samples/s;
  train     the captured train step (CUDA events around graph replays); ms and samples/s.

Layouts: `single` (every field single-valued) and, on one GPU, `bag` (26 single-valued fields and 13 with K = 8, bag
lengths uniform in [0, 8], the layout of tools/bag_bench.py).  `gpu` holds the card's name and power limit, which every
number depends on.  Ids are uniform over each field's 1 M rows; the arenas (7.5 GB) are far larger than the 126 MB L2.

    python tools/eval_bench.py [--rounds 5] [--eval-batches 50] [--steps 100]
    python tools/eval_bench.py --gpus 8          # ShardedAutoIntTrainer, per-rank batch B (torch.distributed.run)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.idmap_bench import gpu_info  # noqa: E402

F, ROWS, B = 39, 1_000_000, 8192
BAG_K = [1] * 26 + [8] * 13


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--eval-batches", type=int, default=50, help="batches per timed evaluate() / predict() pass")
    ap.add_argument("--steps", type=int, default=100, help="captured train steps per round")
    ap.add_argument("--batches", type=int, default=8, help="distinct batches cycled through")
    args = ap.parse_args()
    if args.gpus > 1 and "RANK" not in os.environ:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29911", os.path.abspath(__file__), *sys.argv[1:]]
        raise SystemExit(subprocess.run(cmd).returncode)

    import numpy as np
    import torch
    import torch.distributed as dist
    from recommendsystem_b200.api.metrics import BinaryMetrics
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    if not torch.cuda.is_available():
        raise SystemExit("eval_bench needs a CUDA device")
    world, rank = 1, 0
    if "RANK" in os.environ:
        rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
        dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
        torch.cuda.set_device(dev)
        dist.init_process_group("nccl", device_id=dev)
    else:
        dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(20261022 + rank)

    def batches(K):
        S = sum(K)
        out = []
        for _ in range(args.batches):
            ids = torch.randint(0, ROWS, (B, S), device=dev, generator=g)
            col = 0
            for k in K:
                if k > 1:      # bag length uniform in [0, k]: the slots past it are padding
                    n = torch.randint(0, k + 1, (B, 1), device=dev, generator=g)
                    ids[:, col:col + k] = torch.where(torch.arange(k, device=dev)[None, :] < n, ids[:, col:col + k], -1)
                col += k
            out.append((ids, (torch.rand(B, 1, device=dev, generator=g) < 0.25).float()))
        return out

    def trainer(K):
        cfg = AutoIntConfig(num_fields=F, rows_per_field=ROWS, batch=B, dtype="bf16", bag_size=K)
        if world > 1:
            from recommendsystem_b200.sharded import ShardedAutoIntTrainer
            return ShardedAutoIntTrainer(cfg, dev)
        return AutoIntTrainer(cfg, dev)

    layouts = {"single": [1] * F} if world > 1 else {"single": [1] * F, "bag": BAG_K}
    runs = {}
    for name, K in layouts.items():
        tr = trainer(K)
        tr.capture()
        assert tr.fuse_tower, "the headline configuration runs the tcgen05 tower"
        runs[name] = (tr, batches(K))

    def cycle(bs, n):
        return (bs[i % len(bs)] for i in range(n))

    def t_eval(tr, bs):
        t0 = time.perf_counter()
        tr.evaluate(cycle(bs, args.eval_batches))
        return args.eval_batches * B / (time.perf_counter() - t0)

    def t_predict(tr, bs):
        m = BinaryMetrics(device=dev)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for ids, y in cycle(bs, args.eval_batches):
            m.update_state(y, tr.predict(ids))
        m.result()
        return args.eval_batches * B / (time.perf_counter() - t0)

    def t_train(tr, bs):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for ids, y in cycle(bs, args.steps):
            tr.step(ids, y)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / args.steps

    for tr, bs in runs.values():                              # warm-up: captures the eval graph, loads modules
        t_eval(tr, bs); t_predict(tr, bs); t_train(tr, bs)
    res = {name: {"eval": [], "predict": [], "train_ms": []} for name in runs}
    for _ in range(args.rounds):
        for name, (tr, bs) in runs.items():
            res[name]["eval"].append(t_eval(tr, bs))
            res[name]["predict"].append(t_predict(tr, bs))
            res[name]["train_ms"].append(t_train(tr, bs))
    out = {}
    for name, r in res.items():
        out[name] = {
            "eval_samples_per_s": float(np.median(r["eval"])),
            "predict_metrics_samples_per_s": float(np.median(r["predict"])),
            "train_step_ms": float(np.median(r["train_ms"])),
            "train_samples_per_s": float(B / np.median(r["train_ms"]) * 1e3),
            "eval_spread": [float(np.min(r["eval"])), float(np.max(r["eval"]))],
            "predict_spread": [float(np.min(r["predict"])), float(np.max(r["predict"]))],
            "train_ms_spread": [float(np.min(r["train_ms"])), float(np.max(r["train_ms"]))],
        }
    if rank == 0:
        print(json.dumps({"geometry": {"batch_per_gpu": B, "fields": F, "rows_per_field": ROWS, "dtype": "bf16",
                                       "gpus": world, "bag_fields": "26 x K=1 + 13 x K=8 (lengths uniform in [0, 8])"},
                          "layouts": out, "rounds": args.rounds, "eval_batches": args.eval_batches,
                          "train_steps_per_round": args.steps, "gpu": gpu_info()}), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
