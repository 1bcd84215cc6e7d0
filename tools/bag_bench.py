"""Multi-valued fields in the AutoInt trainer at the headline geometry: B = 8192, 39 fields, 1 M rows per field, bf16.
Prints one JSON line:

  step      captured train-step time (CUDA events around graph replays, ms) of three trainers, alternated in rounds
            in this one process:
              single   the default single-valued configuration (bag_size = 1);
              bag      26 single-valued fields and 13 with K = 8, bag lengths uniform in [0, 8] (so some bags are
                       empty), the bag mean inside the InteractingLayer forward's tile loader;
              unfused  the same bag layout with fuse_embedding=False (rs_embed_bag_fwd_ld, then the forward);
  phases    per-phase times (eager PhaseTimer, ms per step, launches per step) of `bag` and `unfused`, including the
            per-slot gradient pass embed_bag_grad that the sorted-segment update reads;
  gpu       card name and power limit (nvidia-smi), which every number above depends on.

Ids are uniform over each field's 1 M rows; the arenas (7.5 GB each) are far larger than the 126 MB L2.

    python tools/bag_bench.py [--steps 100] [--rounds 5] [--batches 8]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.idmap_bench import gpu_info  # noqa: E402

F, ROWS, B = 39, 1_000_000, 8192
BAG_K = [1] * 26 + [8] * 13


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100, help="captured steps per round and trainer")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batches", type=int, default=8, help="distinct batches cycled through")
    ap.add_argument("--phase-steps", type=int, default=20, help="eager instrumented steps per bag trainer")
    args = ap.parse_args()

    import numpy as np
    import torch
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer, PhaseTimer
    if not torch.cuda.is_available():
        raise SystemExit("bag_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(20261022)

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

    mk = lambda K, fuse: AutoIntConfig(num_fields=F, rows_per_field=ROWS, batch=B, dtype="bf16", bag_size=K,
                                       fuse_embedding=fuse)
    runs = {"single": (mk(1, True), batches([1] * F)), "bag": (mk(BAG_K, True), batches(BAG_K)),
            "unfused": (mk(BAG_K, False), batches(BAG_K))}
    trainers = {}
    for name, (cfg, bs) in runs.items():
        tr = AutoIntTrainer(cfg, dev)
        tr.capture()
        trainers[name] = (tr, bs)
    assert trainers["bag"][0].fused and not trainers["unfused"][0].fused and not trainers["single"][0].bag

    def timed(tr, bs, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            ids, y = bs[i % len(bs)]
            tr.step(ids, y)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / n

    for tr, bs in trainers.values():
        timed(tr, bs, 20)                                     # warm-up
    step = {k: [] for k in trainers}
    for _ in range(args.rounds):
        for name, (tr, bs) in trainers.items():
            step[name].append(timed(tr, bs, args.steps))
    res_step = {k: {"ms_mean": float(np.mean(v)), "ms_min": float(np.min(v)), "ms_max": float(np.max(v))}
                for k, v in step.items()}

    phases = {}
    for name in ("bag", "unfused"):
        tr, bs = trainers[name]
        tr.graph = None                                       # eager, instrumented
        tr.timer = PhaseTimer()
        for i in range(args.phase_steps):
            ids, y = bs[i % len(bs)]
            tr.step(ids, y)
        phases[name] = {k: {"ms": round(v[0], 4), "launches": v[1]} for k, v in tr.timer.summary().items()}
        tr.timer = None

    print(json.dumps({"geometry": {"batch": B, "fields": F, "rows_per_field": ROWS, "dtype": "bf16",
                                   "bag_fields": "26 x K=1 + 13 x K=8 (lengths uniform in [0, 8])"},
                      "step": res_step, "phases": phases, "rounds": args.rounds, "steps_per_round": args.steps,
                      "gpu": gpu_info()}))


if __name__ == "__main__":
    main()
