#!/usr/bin/env python
"""bench.py — AutoInt train samples/s on synthetic Criteo-shape batches (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dtype f32|bf16] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): AutoInt (InteractingLayer layer_num=3, unit 16, 2 heads)
+ DNN tower 624->256->128, 39 fields, 1M-row fp32 tables (d=16), batch 8192 per GPU,
forward + backward + sparse Adam on touched rows + dense Adam.  A "step" is one train step on
one fresh batch of uniform ids.

Own arm: `value` = samples/s with ids/labels already resident in HBM (CUDA-graph replay per
step, CUDA events, max over ranks); `e2e` = the same through the public host loop
AutoIntTrainer.fit_host with pinned HOST ids/labels (every step's inputs go H2D and every step's loss
comes back D2H inside the timed region; the loop double-buffers them beside the compute).  `roofline` is the phase
with the largest share of the step; `kernels` lists every phase with its algorithmic
bytes/FLOPs.  `cpu_baseline` / `--impl reference`: the op-for-op torch-CPU restatement of the
reference TF graph (oracle/oracle_torch.py — TensorFlow is not installable offline) on the
box's host cores.

`--dump-outputs DIR` writes what the last timed step computed as DIR/<name>.npy (see timed_outputs), so that two
builds can be compared output for output: the inputs depend on the arguments alone (seeded on the device).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F, D, U, H, L = 39, 16, 16, 2, 3
ROWS = 1_000_000
BATCH = 8192
MLP = (256, 128)
SEED = 20261018


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm_gbs=j["hbm_gbs"], bf16_tflops=j["bf16_tflops"],
                    bf16_tflops_sustained=j.get("bf16_tflops_sustained", j["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------ reference / CPU arm
def cpu_autoint_samples_per_s(batch, steps, warmup, rows_per_field, threads=None):
    """The reference graph restated op-for-op in torch on the CPU (oracle/oracle_torch.py)."""
    import numpy as np
    import torch
    from oracle import oracle_torch as ot
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(SEED)
    total = rows_per_field * F
    table = torch.empty(total, D).normal_(0, 0.1, generator=g)
    rng = np.random.default_rng(SEED)

    def glorot(fi, fo, shape=None):
        lim = (6.0 / (fi + fo)) ** 0.5
        return torch.from_numpy(rng.uniform(-lim, lim, size=shape or (fi, fo)).astype(np.float32))

    params = {"Wqkvr": glorot(D, U, (D, 4 * U)), "bqkvr": torch.zeros(4 * U), "gamma": torch.ones(U),
              "beta": torch.zeros(U)}
    w = [F * D] + list(MLP)
    for i in range(len(MLP)):
        params[f"mlp_W{i}"] = glorot(w[i], w[i + 1]); params[f"mlp_b{i}"] = torch.zeros(w[i + 1])
    params["out_W"] = glorot(MLP[-1] + F * U, 1); params["out_b"] = torch.zeros(1)
    model = ot.AutoIntCPU(table, params, H, L, 1e-3)
    base = (torch.arange(F) * rows_per_field)[None, :]
    times = []
    for i in range(warmup + steps):
        ids = torch.randint(0, rows_per_field, (batch, F), generator=g) + base
        y = (torch.rand(batch, 1, generator=g) < 0.25).float()
        t0 = time.perf_counter()
        model.train_step(ids, y)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return batch * len(times) / sum(times), 1e3 * sum(times) / len(times), threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import psutil
    rows = ROWS if psutil.virtual_memory().available > 14e9 else 100_000
    sps, ms, threads = cpu_autoint_samples_per_s(BATCH, args.steps, args.warmup, rows)
    sample = (f"{args.steps} train steps (after {args.warmup} warm-up) of batch {BATCH}, {rows} rows/field, "
              "torch-CPU op-for-op restatement of the reference TF graph (TensorFlow unavailable offline)")
    print(json.dumps({
        "impl": "reference", "metric": "autoint_train_samples_per_s", "value": sps, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, "cpu"),
        "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(args, dtype):
    return {"workload": "AutoInt(layer_num=3,unit_num=16,head_num=2)+DNN(256,128), 39 fields, 1M-row tables d=16, "
                        f"batch {BATCH}/GPU, fwd+bwd+sparse Adam+dense Adam (BASELINE configs[1])",
            "batch_per_gpu": BATCH, "global_batch": BATCH * args.gpus, "fields": F, "embed_dim": D,
            "rows_per_field": ROWS, "act_dtype": dtype, "ids": ("uniform" if getattr(args, "ids", "uniform") == "uniform" else "Zipf(1.05) over permuted rows") + ", fresh batch every step",
            "l2": "tables+Adam state 7.5 GB per GPU >> 126 MB L2 (inputs larger than L2, no flush needed)",
            "parallelism": f"dp{args.gpus}" + ("+row-sharded tables (all-to-all)" if args.gpus > 1 else "")}


# ------------------------------------------------------------------------------ own arm
# DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the dominant kernels from the committed
# `ncu --set full` capture of THIS workload (profiles/r1d_ncu_full_metrics.csv; batch 8192, bf16, 1 GPU).  ncu
# replays kernels serialised and cold, so these are per-launch byte counts, not timings.
NCU_TRAFFIC_BYTES = {
    "interacting_bwd": 100.531e6 + 5.835e6,     # profiles/r2_ncu_full_metrics.csv (round-2 kernels, inside a real step)
    "interacting_fwd": 23.019e6 + 42.803e6,     # with the fused lookup: ids + table rows read, X + y + saved written
    "embed_gather": 22.937e6 + 0.326e6,         # profiles/r1d_ncu_full_metrics.csv (kernel unchanged)
    "embed_segsum_adam": 73.986e6 + 23.438e6,
}


def algorithmic(phase, B, act_bytes, n_unique):
    """(bytes, flops) per launch of each phase — DESIGN.md §kernels; SURVEY.md §8d."""
    n = B * F
    zw = MLP[-1] + F * U
    gemm = 2 * B * (F * D * MLP[0] + MLP[0] * MLP[1])
    inter_f = L * (2 * 4 * F * D * U + 2 * 2 * H * F * F * (U // H)) * B
    t = {
        "embed_gather": (n * (8 + D * 4 + D * act_bytes + 8), 0),          # + 8 B sort key written
        "embed_gather_peer": (n * (8 + D * 4 + D * act_bytes), 0),          # rows read over NVLink (W-1)/W of them
        "scatter_grads_peer": (n * (4 + 2 * D * act_bytes), 0),             # grads stored over NVLink (W-1)/W of them
        # x in, y out, + per iteration the saved pre-LayerNorm row and the H softmax statistics (fp32) the tcgen05
        # forward writes / backward reads
        "interacting_fwd": (n * (D + U) * act_bytes + L * n * (U + H) * 4, inter_f),
        # + the fused lookup: id 8 B + fp32 table row + sort key 8 B (X is then a WRITE of the kernel, not a read)
        "interacting_fwd_fused": (n * (8 + D * 4 + 8) + n * (D + U) * act_bytes + L * n * (U + H) * 4, inter_f),
        "interacting_bwd": (n * (U + 2 * D) * act_bytes + L * n * (U + H) * 4, 3 * inter_f),
        "mlp_fwd": (B * (F * D + 2 * MLP[0] + MLP[1]) * act_bytes, gemm),
        "mlp_bwd": (B * (2 * MLP[0] + 3 * MLP[1]) * act_bytes, 2 * B * MLP[0] * MLP[1]),     # act_bwd + dgrad (main stream)
        "mlp_wgrad": (B * (F * D + 2 * MLP[0] + MLP[1]) * act_bytes, gemm),                  # x^T dy + colsums (side stream)
        "mlp_dgrad_x": (B * (MLP[0] + 2 * F * D) * act_bytes, 2 * B * F * D * MLP[0]),
        "logits_loss": (B * zw * act_bytes * 5, 6 * B * zw),
        "sort_keys": (n * 8 * 2, 0),
        "embed_segsum_adam": (n * (8 + D * act_bytes) + n_unique * 2 * 3 * D * 4, 0),
        "dense_adam": (0, 0),
    }
    return t.get(phase, (0, 0))


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def _graph_time_us(fn, inner=10, reps=7):
    """median microseconds per call of `fn`, `inner` calls captured in one CUDA graph (CUDA events)."""
    import torch
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    st, gr = torch.cuda.Stream(), torch.cuda.CUDAGraph()
    with torch.cuda.stream(st):
        with torch.cuda.graph(gr, stream=st):
            for _ in range(inner):
                fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); gr.replay(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3 / inner)
    return sorted(ts)[len(ts) // 2]


def bench_cfg1(dev, steps=20, warmup=5):
    """BASELINE configs[0]: AutoInt (L = 3, 2 heads, d = 16), 39 fields, batch 1024, fwd + bwd (+ both optimizers), FP32
    parity-mode kernels (the configuration the reference's CPU path runs)."""
    import torch
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    B = 1024
    cfg = AutoIntConfig(num_fields=F, rows_per_field=ROWS // 10, embed_dim=D, layer_num=L, unit_num=U, head_num=H,
                        mlp_hidden=MLP, batch=B, dtype="f32", seed=SEED)
    tr = AutoIntTrainer(cfg, dev)
    g = torch.Generator(device=dev).manual_seed(SEED)
    ids = torch.randint(0, ROWS // 10, (steps + warmup, B, F), device=dev, generator=g)
    y = (torch.rand(steps + warmup, B, 1, device=dev, generator=g) < 0.25).float()
    tr.capture()
    for i in range(warmup):
        tr.step(ids[i], y[i])
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(warmup, warmup + steps):
        tr.step(ids[i], y[i])
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    return {"workload": "AutoInt(L=3,U=16,H=2)+DNN(256,128), 39 fields, batch 1024, fp32 (BASELINE configs[0])",
            "ms_per_step": ms, "samples_per_s": B / ms * 1e3, "dtype": "f32", "loss": float(tr.loss.item())}


def bench_cfg3(dev, pk, B=4096, T=100):
    """BASELINE configs[2]: DIN attention unit + sum pooling over a behaviour sequence of length 100, batch 4096 (variant
    A = din.py, B = staytime/layer.py), forward and backward, against the HBM roofline (SURVEY 8d bytes)."""
    import torch
    from recommendsystem_b200 import cabi, ops
    g = torch.Generator(device=dev).manual_seed(3)
    Hd = 16
    out = {"workload": f"DIN attention unit, T={T}, B={B}, H=16 (BASELINE configs[2])"}
    for dt, sz, dn in ((torch.float32, 4, "f32"), (torch.bfloat16, 2, "bf16")):
        q = torch.randn(B, Hd, device=dev, generator=g).to(dt)
        keys = torch.randn(B, T, Hd, device=dev, generator=g).to(dt)
        lens = torch.randint(1, T + 1, (B,), device=dev, generator=g, dtype=torch.int32)
        lens[0] = T
        mask = (torch.arange(T, device=dev)[None, :] < lens[:, None]).to(torch.uint8).contiguous()
        dout = torch.randn(B, Hd, device=dev, generator=g).to(dt)
        for mode, name, win in ((cabi.DIN_A, "A", 3 * Hd), (cabi.DIN_B, "B", 4 * Hd)):
            W1 = torch.randn(win, Hd, device=dev, generator=g) * 0.2
            b1 = torch.zeros(Hd, device=dev)
            W2 = torch.randn(Hd, 1, device=dev, generator=g) * 0.2
            b2 = torch.zeros(1, device=dev)
            vals, sl, mk = (keys, lens, None) if mode == cabi.DIN_A else (None, None, mask)
            tf = _graph_time_us(lambda: ops.din_fwd(mode, q, keys, vals, sl, mk, W1, b1, W2, b2))
            tb = _graph_time_us(lambda: ops.din_bwd(mode, q, keys, vals, sl, mk, W1, b1, W2, b2, dout))
            fb = B * (T * Hd * sz + Hd * sz + T) + B * Hd * sz
            bb = fb + B * T * Hd * sz + B * Hd * sz
            out[f"{name}_{dn}"] = {"fwd_us": round(tf, 2), "bwd_us": round(tb, 2),
                                   "fwd_GBps": round(fb / tf / 1e3, 1), "bwd_GBps": round(bb / tb / 1e3, 1),
                                   "fwd_frac_of_measured_hbm": round(fb / tf / 1e3 / pk["hbm_gbs"], 4),
                                   "bwd_frac_of_measured_hbm": round(bb / tb / 1e3 / pk["hbm_gbs"], 4),
                                   "samples_per_s_fwd_bwd": round(B / (tf + tb) * 1e6, 1)}
    return out


def run_config(args):
    """--config cfg1 | cfg3 (| cfg4 | cfg5, see run_models): one JSON line for a BASELINE config other than the headline."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if args.config in ("cfg4", "cfg5"):
        from tools import models_multi_bench
        return models_multi_bench.main(args)
    if rank != 0:
        return
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    pk = peaks()
    if args.config == "cfg1":
        r = bench_cfg1(dev, args.steps, args.warmup)
        line = {"metric": "autoint_train_samples_per_s", "value": r["samples_per_s"], "unit": "samples/s", "n_gpus": 1,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": r["workload"]}, "loss": r["loss"]}
    else:
        r = bench_cfg3(dev, pk)
        best = r["A_f32"]
        line = {"metric": "din_fwd_bwd_samples_per_s", "value": best["samples_per_s_fwd_bwd"], "unit": "samples/s",
                "n_gpus": 1, "steps": 70, "warmup": 3, "ms_per_step": (best["fwd_us"] + best["bwd_us"]) / 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": r["workload"]},
                "roofline": {"bound": "hbm", "achieved": best["fwd_GBps"], "peak": pk["hbm_gbs"], "unit": "GB/s",
                             "frac": best["fwd_frac_of_measured_hbm"], "traffic": None, "kernel": "din_fwd (variant A, fp32)"},
                "din": r}
    print(json.dumps(line), flush=True)


def _finish(world, dist):
    """Multi-rank teardown: tearing the NCCL communicator down while captured graphs still
    reference it can block, so synchronise, flush and leave without running destructors."""
    import torch
    torch.cuda.synchronize()
    if world > 1:
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


DUMP_MAX_ROWS = 1 << 19      # 32 MiB of fp32 table rows: a dump stays under 64 MB


def timed_outputs(tr):
    """What the trainer's last step computed, as float32 / float64 host arrays: the loss, the clipped predictions,
    every dense parameter after the update, and the embedding rows the step updated (`table_rows`: arena row indices,
    this rank's own rows when sharded; `table`: their values), a fixed seeded sample if there are more than
    DUMP_MAX_ROWS of them.  Collective when sharded: every rank calls it."""
    import torch
    rows = tr._touched_rows()
    if rows.numel() > DUMP_MAX_ROWS:
        g = torch.Generator(device=rows.device).manual_seed(SEED)
        rows = rows[torch.randperm(rows.numel(), device=rows.device, generator=g)[:DUMP_MAX_ROWS]].sort().values
    out = {"loss": tr.loss, "pred": tr.p_raw.float().clamp(1e-6, 1.0), "table_rows": rows.double(), "table": tr.table[rows]}
    out.update({f"dense_{k}": v for k, v in tr.P.items()})
    return {k: (v if v.dtype == torch.float64 else v.float()).cpu().numpy() for k, v in out.items()}


def run_own(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from recommendsystem_b200 import cabi
    from recommendsystem_b200 import ops as ops_mod
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer, PhaseTimer

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        from recommendsystem_b200.sharded import ShardedAutoIntTrainer as Trainer
    else:
        Trainer = AutoIntTrainer
    cfg = AutoIntConfig(num_fields=F, rows_per_field=ROWS, embed_dim=D, layer_num=L, unit_num=U, head_num=H,
                        mlp_hidden=MLP, batch=BATCH, dtype=args.dtype, seed=SEED)
    tr = Trainer(cfg, dev)
    K, W = args.steps, args.warmup
    g = torch.Generator(device=dev).manual_seed(SEED + rank)
    nb = K + W
    if args.ids == "zipf":
        # secondary workload (SURVEY §8d): Zipf(s = 1.05) popularity over a random permutation of each field's rows
        # -> many duplicate rows per batch (long sorted-segment runs, L2-resident hot rows)
        w = 1.0 / torch.arange(1, ROWS + 1, device=dev, dtype=torch.float64) ** 1.05
        rank_of = torch.multinomial(w.float(), nb * BATCH * F, replacement=True, generator=g).view(nb, BATCH, F)
        perm = torch.randperm(ROWS, device=dev, generator=g)
        ids_dev = perm[rank_of]
    else:
        ids_dev = torch.randint(0, ROWS, (nb, BATCH, F), device=dev, generator=g)
    y_dev = (torch.rand(nb, BATCH, 1, device=dev, generator=g) < 0.25).float()
    act_bytes = 4 if args.dtype == "f32" else 2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- instrumented eager pass: per-phase CUDA-event times + launches per step (rank 0 reports)
    tr.step(ids_dev[0], y_dev[0])
    torch.cuda.synchronize()
    n0 = cabi.launch_count()
    tr.timer = PhaseTimer()
    for i in range(min(K, 20)):
        tr.step(ids_dev[i % nb], y_dev[i % nb])
    phases = tr.timer.summary()
    launches_per_step = (cabi.launch_count() - n0) // min(K, 20)
    tr.timer = None
    n_unique = int(torch.unique(ids_dev[0] + torch.arange(F, device=dev)[None, :] * ROWS).numel())

    # ---- device-resident timing (CUDA graph replay)
    tr.capture()
    for i in range(W):
        tr.step(ids_dev[i], y_dev[i])
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(W, W + K):
        tr.step(ids_dev[i], y_dev[i])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clk = clocks.stop() if rank == 0 else None
    loss_dev = float(tr.loss.item())
    # taken now: the end-to-end loop below trains the same trainer further
    dump = timed_outputs(tr) if args.dump_outputs else None

    # ---- end to end: pinned host inputs, H2D + step + loss D2H every step
    ids_host = ids_dev.cpu().pin_memory()
    y_host = y_dev.cpu().pin_memory()
    for _ in tr.fit_host((ids_host[i], y_host[i]) for i in range(W)):
        pass
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    # the public end-to-end loop: every step uploads its own pinned-host batch and returns its own loss
    # to the host; the loader overlaps batch n+1's H2D and step n-1's loss D2H with step n's compute
    for last in tr.fit_host((ids_host[i], y_host[i]) for i in range(W, W + K)):
        pass
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)

    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        _finish(world, dist)
        return

    pk = peaks()
    step_ms_sum = sum(v[0] for v in phases.values())
    kernels = []
    fused = bool(getattr(tr, "fused", False))
    for name, (pms, nl) in sorted(phases.items(), key=lambda kv: -kv[1][0]):
        by, fl = algorithmic(name + "_fused" if (fused and name == "interacting_fwd") else name, BATCH, act_bytes, n_unique)
        kernels.append({"phase": name, "ms": round(pms, 4), "share": round(pms / step_ms_sum, 4), "launches": nl,
                        "alg_bytes": by, "alg_flops": fl,
                        "GBps": round(by / pms / 1e6, 1) if by else None,
                        "TFLOPps": round(fl / pms / 1e9, 2) if fl else None})
    # The eager per-phase times above include the host launch gaps of multi-launch phases (the eager pass is
    # host-bound; the headline replays a CUDA graph).  The roofline kernel is therefore chosen and timed from
    # SINGLE-kernel launches replayed ten times inside one CUDA graph with CUDA events around the replay (1 GPU).
    iso = {}
    if world == 1:
        T_ = ops_mod._DT[tr.act_dtype]
        st_ = lambda: ops_mod._stream()
        nW_ = D * 4 * U
        singles = {
            "interacting_fwd": lambda: cabi.call(
                "rs_interacting_fwd", tr.X.data_ptr(), D, 0, T_, tr.P["Wqkvr"].data_ptr(), tr.P["bqkvr"].data_ptr(),
                tr.P["gamma"].data_ptr(), tr.P["beta"].data_ptr(), cfg.ln_eps, tr.Z[:, tr.n_deep:].data_ptr(), U, tr.zw,
                tr.saved.data_ptr(), BATCH, F, D, U, H, L, 1, int(args.dtype == "bf16"), st_()),
            "interacting_bwd": lambda: tr._interacting_bwd(tr.flat_g[tr.spec[0][2]:], st_(), T_),
            "embed_gather": lambda: tr._embed_forward(lambda name: _NullCtx(), st_(), T_),
            "embed_segsum_adam": lambda: ops_mod.segsum_adam(tr.table, tr.table_m, tr.table_v, tr.dX.view(-1, D), tr.keys_sorted,
                                                             cfg.lr_sparse, cfg.beta1, cfg.beta2, cfg.eps, tr.adam_scalars),
        }
        if fused:
            tabs_, w_, lb_, keys_ = tr._lookup_args()
            singles["interacting_fwd"] = lambda: cabi.call(
                "rs_interacting_fwd_gather", tabs_, tr.table_ld, w_, tr.ids.data_ptr(), lb_.data_ptr(), tr.rows_t.data_ptr(),
                tr.X.data_ptr(), D, 0, keys_, T_, tr.P["Wqkvr"].data_ptr(), tr.P["bqkvr"].data_ptr(), tr.P["gamma"].data_ptr(),
                tr.P["beta"].data_ptr(), cfg.ln_eps, tr.Z[:, tr.n_deep:].data_ptr(), U, tr.zw, tr.saved.data_ptr(), BATCH, F, D,
                U, H, L, 1, st_())
            # the kernel itself, as the step launches it (its 1120-float partial reduction runs on the side stream)
            singles["interacting_bwd"] = lambda: tr._interacting_bwd_fused(None, st_(), T_, None)
        for name, fn in singles.items():
            try:
                iso[name] = _graph_time_us(fn) / 1e3
            except Exception as e:
                iso[name + "_error"] = repr(e)[:120]
        if "embed_gather" in iso and not any(k["phase"] == "embed_gather" for k in kernels):
            by_, _ = algorithmic("embed_gather", BATCH, act_bytes, n_unique)
            embed_alone = {"gather_alone_ms": round(iso["embed_gather"], 4), "gather_alone_GBps": round(by_ / iso["embed_gather"] / 1e6, 1),
                           "note": "the separate gather kernel, NOT part of the fused step; timed for reference"}
        else:
            embed_alone = None
        for k in kernels:
            if k["phase"] in iso:
                by, fl = k["alg_bytes"], k["alg_flops"]
                k["ms_alone_in_graph"] = round(iso[k["phase"]], 4)
                k["GBps_alone"] = round(by / iso[k["phase"]] / 1e6, 1) if by else None
                k["TFLOPps_alone"] = round(fl / iso[k["phase"]] / 1e9, 2) if fl else None
        ranked = sorted((k for k in kernels if k["phase"] in iso), key=lambda k: -iso[k["phase"]])
        if ranked:
            top = dict(ranked[0])
            top["ms"], top["GBps"], top["TFLOPps"] = top["ms_alone_in_graph"], top["GBps_alone"], top["TFLOPps_alone"]
        else:
            top = kernels[0]
    else:
        top = kernels[0]
    if top["phase"].startswith("mlp") and args.dtype == "bf16":
        roof = {"bound": "tensor", "achieved": top["TFLOPps"], "peak": pk["bf16_tflops_sustained"],
                "unit": "TFLOP/s", "frac": top["TFLOPps"] / pk["bf16_tflops_sustained"], "traffic": None}
    else:
        roof = {"bound": "hbm", "achieved": top["GBps"], "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": (top["GBps"] or 0) / pk["hbm_gbs"], "traffic": None}
    if world == 1 and args.dtype == "bf16" and BATCH == 8192:
        roof["traffic"] = NCU_TRAFFIC_BYTES.get(top["phase"])
        roof["traffic_source"] = "profiles/r2_ncu_full_metrics.csv (dram__bytes_read + write per launch)"
    # share of the STEP: the kernel's event-timed duration over the graph-replayed step time the headline is made of
    roof.update({"kernel": top["phase"], "peak_source": pk["source"] + " (sustained: kernel timed inside the step)",
                 "share_of_step": round(top["ms"] / (ms / K), 4), "share_of_phase_sum": top["share"]})
    gk = next((k for k in kernels if k["phase"] in ("embed_gather", "embed_gather_peer")), None)
    sk = next(k for k in kernels if k["phase"] == "embed_segsum_adam")
    # eager, instrumented pass: one CUDA-event pair around a single ~30 us launch (the pair and the host launch gap are in
    # the number); the in-graph figures below are the ones to read
    embed = {"scatter_adam_GBps_eager_phase": sk["GBps"],
             "scatter_adam_frac_of_measured_hbm_eager_phase": sk["GBps"] / pk["hbm_gbs"], "unique_rows": n_unique}
    if gk is not None:
        embed.update({"gather_GBps": gk["GBps"], "gather_frac_of_measured_hbm": gk["GBps"] / pk["hbm_gbs"],
                      "gather_frac_of_8TBps": gk["GBps"] / 8000.0, "gather_kernel": gk["phase"]})
    else:
        embed["gather_kernel"] = ("fused into interacting_fwd (rs_interacting_fwd_gather): no gather launch in the step; "
                                  "its ids + rows + X + keys bytes are counted in interacting_fwd's algorithmic bytes")
    if world == 1 and "embed_segsum_adam" in iso:
        by_s, _ = algorithmic("embed_segsum_adam", BATCH, act_bytes, n_unique)
        embed.update({"scatter_adam_ms_in_graph": round(iso["embed_segsum_adam"], 4),
                      "scatter_adam_GBps": round(by_s / iso["embed_segsum_adam"] / 1e6, 1),
                      "scatter_adam_frac_of_measured_hbm": round(by_s / iso["embed_segsum_adam"] / 1e6 / pk["hbm_gbs"], 4),
                      "scatter_adam_GBps_in_graph": round(by_s / iso["embed_segsum_adam"] / 1e6, 1),
                      "scatter_adam_frac_of_measured_hbm_in_graph": round(by_s / iso["embed_segsum_adam"] / 1e6 / pk["hbm_gbs"], 4)})
    if world == 1 and embed_alone is not None:
        embed["separate_gather_kernel"] = embed_alone
    if world == 1 and gk is not None:
        # The per-phase times above come from an eager pass with one CUDA-event pair per phase: for a 13 us kernel
        # the pair itself adds several us.  Time the same gather launch (this batch's ids, the trainer's table)
        # ten times inside one CUDA graph as well.
        try:
            from recommendsystem_b200 import ops as _ops

            def _gather():
                return _ops.embed_gather(tr.table, tr.ids, tr.base_t, tr.rows_t, out_dtype=tr.act_dtype, want_keys=True)
            for _ in range(3):
                _gather()
            torch.cuda.synchronize()
            gs_, gr_ = torch.cuda.Stream(), torch.cuda.CUDAGraph()
            with torch.cuda.stream(gs_):
                with torch.cuda.graph(gr_, stream=gs_):
                    for _ in range(10):
                        _gather()
            ts_ = []
            for _ in range(7):
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record(); gr_.replay(); b_.record(); torch.cuda.synchronize()
                ts_.append(a_.elapsed_time(b_) / 10)
            t_g = sorted(ts_)[len(ts_) // 2]
            by_g, _ = algorithmic("embed_gather", BATCH, act_bytes, n_unique)
            embed.update({"gather_ms_in_graph": t_g, "gather_GBps_in_graph": by_g / t_g / 1e6,
                          "gather_frac_of_measured_hbm_in_graph": by_g / t_g / 1e6 / pk["hbm_gbs"]})
        except Exception as e:                       # a reporting extra: never fail the bench line over it
            embed["gather_in_graph_error"] = repr(e)[:200]

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        import psutil
        rows = ROWS if psutil.virtual_memory().available > 14e9 else 100_000
        sps, cms, threads = cpu_autoint_samples_per_s(BATCH, 6, 2, rows)
        cpu = {"value": sps, "unit": "samples/s", "cores": threads, "kind": "port",
               "sample": f"6 train steps (after 2 warm-up) of batch {BATCH}, {rows} rows/field; torch-CPU op-for-op "
                         "restatement of the reference TF graph (TensorFlow unavailable offline)",
               "ms_per_step": cms}

    other = None
    if world == 1 and not args.no_other_configs:
        try:
            other = {"cfg1": bench_cfg1(dev, steps=20, warmup=5), "cfg3": bench_cfg3(dev, pk)}
        except Exception as e:                       # reporting extras never fail the headline line
            other = {"error": repr(e)[:300]}

    out = {
        "metric": "autoint_train_samples_per_s", "value": BATCH * world * K / (ms / 1e3), "unit": "samples/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": workload_config(args, args.dtype),
        "e2e": {"value": BATCH * world * K / (ms_e2e / 1e3), "unit": "samples/s",
                "h2d_bytes_per_step": BATCH * F * 8 + BATCH * 4, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / K},
        "gpu_launches": int(launches_per_step * K), "launches_per_step": int(launches_per_step),
        "clocks": clk, "roofline": roof, "embed_roofline": embed, "kernels": kernels,
        "cpu_baseline": cpu, "loss": loss_dev, "loss_e2e_last": last, "other_configs": other,
    }
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(out), flush=True)
    _finish(world, dist)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--dtype", default=os.environ.get("RS_BENCH_DTYPE", "bf16"), choices=["f32", "bf16"])
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the cfg1 / cfg3 extras of the default line")
    ap.add_argument("--config", default="cfg2", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"],
                    help="BASELINE.json configs by SURVEY 8 numbering: cfg1 = configs[0] (B=1024 fp32), cfg2 = configs[1] "
                         "(headline, default), cfg3 = DIN, cfg4 = multi_head AUTOINT 200 M rows / 8 GPUs, cfg5 = VideoDnn")
    ap.add_argument("--ids", default="uniform", choices=["uniform", "zipf"],
                    help="id distribution of the synthetic batches (headline: uniform; zipf = skewed secondary workload)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (headline workload only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "own" or args.config != "cfg2"):
        ap.error("--dump-outputs needs the headline workload (--impl own, --config cfg2)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.config != "cfg2":
        run_config(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
