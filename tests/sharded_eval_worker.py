"""Worker for tests/test_gpu_sharded_eval.py (launched with torch.distributed.run, one rank per GPU): the sharded
evaluate() on per-rank streams of unequal length against the single-GPU evaluate() of the concatenated stream, with
the single-GPU trainer loaded from the sharded trainer's checkpoint."""
import os
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    """argv: mode (eager | graph)  dtype (f32 | bf16)  b (per-rank batch)"""
    from recommendsystem_b200 import checkpoint as ck
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    from recommendsystem_b200.sharded import ShardedAutoIntTrainer
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    use_graph, dtype, b = sys.argv[1] == "graph", sys.argv[2], int(sys.argv[3])
    F = 39
    kw = dict(num_fields=F, rows_per_field=700, batch=b, lr_dense=1e-3, lr_sparse=1e-2, dtype=dtype)
    rng = np.random.default_rng(17)                        # identical on every rank

    def batch(n):
        ids = rng.integers(0, 2 ** 40, size=(n, F)).astype(np.int64)
        ids[rng.random(ids.shape) < 0.05] = -1
        return torch.from_numpy(ids), torch.from_numpy((rng.random((n, 1)) < 0.3).astype(np.float32))

    train = [[batch(b) for _ in range(world)] for _ in range(3)]
    # rank r evaluates r mod 3 full batches (rank 0: none), odd ranks one partial batch more
    streams = [[batch(b) for _ in range(r % 3)] + ([batch(b // 3 + r)] if r % 2 else []) for r in range(world)]

    sh = ShardedAutoIntTrainer(AutoIntConfig(**kw), dev)
    if use_graph:
        sh.capture()
    for step in train:
        sh.step(step[rank][0].to(dev), step[rank][1].to(dev))
    sh.check_overflow()
    box = [tempfile.mkdtemp(prefix="rs_eval_") if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    ck.save_checkpoint(sh, os.path.join(box[0], "w"), step=3)
    dist.barrier()

    mine = [(i.to(dev), y.to(dev)) if rank % 2 else (i.pin_memory(), y.pin_memory()) for i, y in streams[rank]]
    got = sh.evaluate(mine)
    everyone = [None] * world
    dist.all_gather_object(everyone, got)
    sh.step(train[0][rank][0].to(dev), train[0][rank][1].to(dev))       # training goes on after an evaluation
    sh.check_overflow()
    torch.cuda.synchronize()

    ok = True

    def check(name, cond, info=""):
        nonlocal ok
        print(f"[rank {rank}] " + ("PASS " if cond else "FAIL ") + name + (f" {info}" if info else ""), flush=True)
        ok = ok and bool(cond)

    check("every rank returns the same dict", all(e == got for e in everyone))
    if rank == 0:
        one = AutoIntTrainer(AutoIntConfig(**kw), dev)
        ck.load_checkpoint(one, os.path.join(box[0], "w"))
        want = one.evaluate([(i.to(dev), y.to(dev)) for s in streams for i, y in s])
        n_all = sum(i.shape[0] for s in streams for i, _ in s)
        check("count", got["count"] == want["count"] == n_all, f"{got['count']} {want['count']} {n_all}")
        check("auc", got["auc"] == want["auc"], f"{got['auc']!r} {want['auc']!r}")
        check("binary_accuracy", got["binary_accuracy"] == want["binary_accuracy"])
        for k in ("ctr", "copc", "mean_prediction"):
            check(k, abs(got[k] - want[k]) <= 1e-12 * abs(want[k]), f"{got[k]!r} {want[k]!r}")
        check("loss", abs(got["loss"] - want["loss"]) <= 1e-6, f"{got['loss']!r} {want['loss']!r}")
        print(f"[rank 0] sharded {got}\n[rank 0] single {want}", flush=True)
        import shutil
        shutil.rmtree(box[0], ignore_errors=True)
    flag = torch.tensor([0 if ok else 1], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    dist.destroy_process_group()
    sys.exit(int(flag.item()))


if __name__ == "__main__":
    main()
