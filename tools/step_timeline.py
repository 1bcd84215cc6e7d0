"""Where does the headline step's time go INSIDE the CUDA graph?  Timestamp kernels (rs_debug_timestamp, %globaltimer)
at the phase boundaries of AutoIntTrainer._launch_step are captured with the step; one replay then yields the time at
which the main stream (and the side stream's tail) reached each boundary.  Each stamp is a one-thread kernel (~2 us on
its stream), so the instrumented step is a few microseconds longer than the real one; the plain replay time is printed
next to it.  usage: python tools/step_timeline.py [--batch 8192] [--reps 20]"""
import argparse
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer  # noqa: E402


def replay_ms(tr, n=50):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(5):
        tr.graph.replay()
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        tr.graph.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--fuse-tower", type=int, default=1, help="0: the tower as 4 GEMMs + the head pass")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    cfg = AutoIntConfig(num_fields=39, rows_per_field=args.rows, embed_dim=16, unit_num=16, head_num=2, layer_num=3,
                        mlp_hidden=(256, 128), batch=args.batch, dtype="bf16",
                        fuse_tower=bool(args.fuse_tower))
    if world > 1:       # torchrun: the row-sharded trainer (rank 0 prints its own timeline)
        import torch.distributed as dist
        from recommendsystem_b200.sharded import ShardedAutoIntTrainer
        dist.init_process_group("nccl", device_id=dev)
        make = lambda: ShardedAutoIntTrainer(cfg, dev)
    else:
        make = lambda: AutoIntTrainer(cfg, dev)
    g = torch.Generator(device="cpu").manual_seed(rank)
    ids = torch.randint(0, 2 ** 40, (args.batch, 39), generator=g).to(dev)
    y = (torch.rand(args.batch, 1, generator=g) < 0.25).float().to(dev)
    out = {}
    for instrumented in (False, True):
        tr = make()
        if instrumented:
            tr.stamps = torch.zeros(64, dtype=torch.int64, device=dev)
        tr.ids.copy_(ids)
        tr.labels.copy_(y)
        tr.capture()
        out[instrumented] = replay_ms(tr)
        if instrumented:
            names = sorted(tr.stamp_names, key=tr.stamp_names.get)
            rows = []
            for _ in range(args.reps):
                tr.graph.replay()
                torch.cuda.synchronize()
                t = tr.stamps[:len(names)].cpu().numpy().astype(np.int64)
                rows.append((t - t[tr.stamp_names["step_begin"]]) / 1e3)
            med = np.median(np.stack(rows), 0)
            if rank == 0:
                print(f"graph replay: {out[False] * 1e3:.1f} us plain, {out[True] * 1e3:.1f} us with {len(names)} stamps")
                print("median time (us after step_begin) at which the stream reached each boundary:")
                for n, v in sorted(zip(names, med), key=lambda kv: kv[1]):
                    print(f"  {v:8.1f}  {n}")
        del tr
        torch.cuda.empty_cache()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
