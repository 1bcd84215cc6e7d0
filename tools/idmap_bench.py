"""Cost of the collision-free id map (id_map="hash") at the headline geometry: 39 fields, 1 M rows per field,
B = 8192, bf16 AutoInt.  Prints one JSON line:

  map       insert and lookup pass times (CUDA events around CUDA-graph replays of each pass, mean over batches) in
            three states: first touch (every key of the batch is new), steady (every key already mapped) and Zipf(1.05)
            ids over the same pool (mostly hits, some new keys);
  step      AutoInt train-step time in mod and hash mode, both captured, alternated in rounds in this one process
            (the hash step includes the show count, a branch off the map lookup);
  evict     IdMap.evict on a full map (every row of the 39 x 1 M owned, Adam [w|m|v] records) with about half the
            keys dropped: random shows in [0, 1), threshold 0.5, decay 0.9 (CUDA events; the map is refilled with
            the same keys and the shows redrawn before each round);
  gpu       card name and power limit (nvidia-smi), which every number above depends on.

Ids are 63-bit signs drawn from a per-field pool of 1 M random keys (uniform, or Zipf(1.05) by rank as bench.py
--ids zipf).  The map's slots (1.25 GB) and the arenas (7.5 GB each) are far larger than the 126 MB L2.

    python tools/idmap_bench.py [--batches 48] [--steps 100] [--rounds 5] [--evict-rounds 3]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

F, ROWS, B, POOL = 39, 1_000_000, 8192, 1_000_000


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:                      # the numbers stay, the card is named by torch alone
        import torch
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unknown ({e.__class__.__name__})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=48, help="batches timed per map state")
    ap.add_argument("--steps", type=int, default=100, help="train steps per round and mode")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warm-steps", type=int, default=500, help="hash-trainer steps before timing (fills the map)")
    ap.add_argument("--evict-rounds", type=int, default=3)
    args = ap.parse_args()

    import numpy as np
    import torch
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    from recommendsystem_b200.idmap import IdMap
    if not torch.cuda.is_available():
        raise SystemExit("idmap_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(20261020)
    pool = torch.randint(0, 2 ** 63 - 1, (F, POOL), device=dev, generator=g)
    fcol = torch.arange(F, device=dev)

    def draw(idx):                               # idx [n, B, F] pool positions -> keys
        return pool[fcol, idx]

    zw = (1.0 / torch.arange(1, POOL + 1, device=dev, dtype=torch.float64) ** 1.05).float()
    zperm = torch.randperm(POOL, device=dev, generator=g)

    def zipf(n):
        r = torch.multinomial(zw, n * B * F, replacement=True, generator=g).view(n, B, F)
        return draw(zperm[r])

    # ---------------------------------------------------------------- map passes
    nb = args.batches
    arena = torch.zeros(F * ROWS, 3, 16, device=dev)
    m = IdMap([ROWS] * F, dev, 1, 0.1, arena[:, 0, :], [(arena[:, 1, :], 0.0), (arena[:, 2, :], 0.0)])
    ids = torch.empty(B, F, dtype=torch.int64, device=dev)
    rows = torch.empty(B, F, dtype=torch.int64, device=dev)
    fields = m.fields(range(F))
    from recommendsystem_b200 import ops
    warm = torch.randint(0, 2 ** 62, (B, F), device=dev, generator=g)

    def ins():
        ops.idmap_insert(m.slots, m.key_of_row, m.counters, m.geom, ids, fields, m.seed, m.scale, m.w, m.states)

    def look():
        ops.idmap_lookup(m.slots, m.counters, m.geom, ids, fields, out=rows, after_insert=True)

    ids.copy_(warm)                              # warm-up launches, then undone
    ins(); look()
    torch.cuda.synchronize()
    m.restore(torch.zeros_like(m.counters))
    graphs = []
    for fn in (ins, look):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            fn()
        graphs.append(gr)
    torch.cuda.synchronize()

    def time_state(batches):
        t_ins, t_look = [], []
        for k in range(batches.shape[0]):
            ids.copy_(batches[k])
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record(); graphs[0].replay(); e[1].record(); graphs[1].replay(); e[2].record()
            e[2].synchronize()
            t_ins.append(e[0].elapsed_time(e[1]) * 1e3)
            t_look.append(e[1].elapsed_time(e[2]) * 1e3)
        return {"insert_us": float(np.mean(t_ins)), "lookup_us": float(np.mean(t_look)),
                "insert_us_min": float(np.min(t_ins)), "lookup_us_min": float(np.min(t_look))}

    # first touch: every key of every batch is new (distinct pool positions per field)
    perm = torch.stack([torch.randperm(POOL, device=dev, generator=g)[:nb * B] for _ in range(F)], 1).view(nb, B, F)
    first = draw(perm)
    res_map = {"first_touch": time_state(first)}
    assert int(m.counters[0].sum()) == nb * B * F, "first-touch batches were not all new keys"
    res_map["steady"] = time_state(first[torch.randperm(nb, device=dev, generator=g)])
    before = int(m.counters[0].sum())
    res_map["zipf"] = time_state(zipf(nb))
    res_map["zipf"]["new_keys_per_batch"] = (int(m.counters[0].sum()) - before) / nb
    res_map["rows_used"] = int(m.counters[0].sum())
    del arena, m, graphs
    torch.cuda.empty_cache()

    # ---------------------------------------------------------------- AutoInt step, mod vs hash
    cfg = lambda mode: AutoIntConfig(dtype="bf16", id_map=mode)
    trs = {"mod": AutoIntTrainer(cfg("mod"), dev), "hash": AutoIntTrainer(cfg("hash"), dev)}
    n_data = 64
    data_ids = draw(torch.randint(0, POOL, (n_data, B, F), device=dev, generator=g))
    data_y = (torch.rand(n_data, B, 1, device=dev, generator=g) < 0.25).float()
    for tr in trs.values():
        tr.ids.copy_(data_ids[0]); tr.labels.copy_(data_y[0])
        tr.capture()
    for s in range(args.warm_steps):
        trs["hash"].step(data_ids[s % n_data], data_y[s % n_data])
        if s < 20:
            trs["mod"].step(data_ids[s % n_data], data_y[s % n_data])
    torch.cuda.synchronize()
    times = {"mod": [], "hash": []}
    for _ in range(args.rounds):
        for mode, tr in trs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for s in range(args.steps):
                tr.ids.copy_(data_ids[s % n_data], non_blocking=True)
                tr.labels.copy_(data_y[s % n_data], non_blocking=True)
                tr.run()
            e1.record()
            e1.synchronize()
            times[mode].append(e0.elapsed_time(e1) / args.steps)
    st = trs["hash"].idmap.stats()
    step = {mode: {"ms_median": float(np.median(v)), "ms_rounds": [round(x, 4) for x in v]} for mode, v in times.items()}
    step["hash_over_mod"] = step["hash"]["ms_median"] / step["mod"]["ms_median"] - 1.0
    step["hash_rows_used"] = int(sum(st["rows_used"]))
    step["hash_overflow"] = int(sum(st["overflow"]))
    del trs
    torch.cuda.empty_cache()

    # ---------------------------------------------------------------- evict on a full map
    arena = torch.zeros(F * ROWS, 3, 16, device=dev)
    m = IdMap([ROWS] * F, dev, 1, 0.1, arena[:, 0, :], [(arena[:, 1, :], 0.0), (arena[:, 2, :], 0.0)])
    fill = pool.t().contiguous()                                  # [1 M, F]: every pool key of every field
    ev = {"ms": [], "dropped": []}
    for _ in range(args.evict_rounds + 1):                        # the first round warms up (workspace, cub)
        m.resolve(fill, m.fields(range(F)), insert=True)
        assert int(m.counters[0].sum()) == F * ROWS, "the map is not full"
        m.show.uniform_(0.0, 1.0, generator=g)
        before = int(m.evicted.sum())
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        m.evict(0.5, 0.9)
        e1.record()
        e1.synchronize()
        ev["ms"].append(e0.elapsed_time(e1))
        ev["dropped"].append(int(m.evicted.sum()) - before)
    ev = {"ms_median": float(np.median(ev["ms"][1:])), "ms_rounds": [round(x, 3) for x in ev["ms"][1:]],
          "dropped_rounds": ev["dropped"][1:], "rows": F * ROWS}
    print(json.dumps({"bench": "idmap", "fields": F, "rows_per_field": ROWS, "batch": B, "dtype": "bf16",
                      "map": res_map, "step": step, "evict": ev, "gpu": gpu_info(),
                      "note": "step times include the ids/labels device copies of each step (both modes)"}))


if __name__ == "__main__":
    main()
