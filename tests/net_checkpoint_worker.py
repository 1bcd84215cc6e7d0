"""Worker for tests/test_gpu_net_checkpoint.py::test_sharded_round_trips (torch.distributed.run, one rank per GPU):
checkpoints of composed nets over the row-sharded ShardedEmbeddingFeatures.  A W-way net trained two steps is saved
and loaded back into a W-way net (W -> W), into an unsharded net on rank 0 (W -> 1), and the unsharded net's save into
a W-way net (1 -> W); each load must give every record of the global arena, the dense weights and the dense Adam
state back bit for bit."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from recommendsystem_b200 import checkpoint as ck
    from recommendsystem_b200.api.builders import AUTOINT, AUTOINT_LABELS
    from recommendsystem_b200.api.sharded_embedding import ShardedEmbeddingFeatures
    from recommendsystem_b200.api.staytime_config import Config as C
    from recommendsystem_b200.api.video_dnn import TASK_KEYS, mtl_net
    from recommendsystem_b200.arena import field_slices
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    which, root = sys.argv[1], sys.argv[2]
    ok = True

    def check(name, cond):
        nonlocal ok
        if rank == 0:
            print(("PASS " if cond else "FAIL ") + name, flush=True)
        ok = ok and bool(cond)

    g = torch.Generator().manual_seed(17 + rank)             # every rank trains on its own batch
    b = 64
    ids = lambda keys: {k: torch.randint(0, 10 ** 9, (b,), generator=g).to(dev) for k in keys}
    flag = lambda: (torch.rand(b, 1, generator=g) < 0.3).float().to(dev)
    if which == "autoint":
        slots = [str(3000 + i) for i in range(13)]
        inp, lab = ids(slots), {k: flag() for k in AUTOINT_LABELS}

        def build(sharded, seed):
            kw = dict(embedding_cls=ShardedEmbeddingFeatures, group=None) if sharded else {}
            return AUTOINT(slots, [], True, dnn_hidden_units=(32, 16), bucket_size=997, device=str(dev), seed=seed,
                           **kw).model
    else:
        T = 6
        inp = ids(C.SLOTS)
        for s in C.SEQ_SLOTS:
            x = torch.randint(0, 10 ** 9, (b, T), generator=g)
            x[torch.arange(T)[None, :] >= torch.randint(0, T + 1, (b,), generator=g)[:, None]] = -1
            inp[s] = x.to(dev)
        y0 = torch.softmax(torch.randn(b, 400, generator=g), -1)
        lab = {TASK_KEYS[0]: torch.cat([y0, torch.zeros(b, 1)], 1).to(dev), TASK_KEYS[1]: flag(), TASK_KEYS[2]: flag()}

        def build(sharded, seed):
            kw = dict(embedding_cls=ShardedEmbeddingFeatures, group=None) if sharded else {}
            return mtl_net(C.SLOTS, C.SEQ_SLOTS, T, dnn_hidden_units=(64, 32), bucket_size=499, device=str(dev),
                           seed=seed, **kw)["net"]

    def made(sharded, seed):
        net = build(sharded, seed)
        torch.manual_seed(seed)
        net.predict(inp)                                       # lazy build
        return net

    def global_records(net):
        """[total rows, record_floats] in the unsharded arena order (collective for a sharded net)."""
        st = net.emb.store
        mine = st.pack(slice(0, st.n_local)).contiguous()
        if st.world == 1:
            return mine
        shards = [torch.empty_like(mine) for _ in range(st.world)]
        dist.all_gather(shards, mine)
        out = torch.empty(st.total_rows, st.record_floats, device=dev)
        for r in range(st.world):
            for gl, loc in field_slices(st.rows, st.world, r):
                out[gl] = shards[r][loc]
        return out

    def dense(net):
        return [net.opt.flat.clone(), net.opt.flat_m.clone(), net.opt.flat_v.clone(), net.opt.scalars.clone()] + \
            ([net.emb.scalars.clone()] if getattr(net.emb, "scalars", None) is not None else [])

    def same(x, y):
        return len(x) == len(y) and all(torch.equal(p, q) for p, q in zip(x, y))

    src = made(True, 3)
    for _ in range(2):
        src.train_step(inp, lab)
    ck.save_checkpoint(src, os.path.join(root, "w"), step=2)
    torch.cuda.synchronize()
    dist.barrier()
    want_rec, want_dense = global_records(src), dense(src)

    back = made(True, 5)                                       # W -> W
    ck.load_checkpoint(back, os.path.join(root, "w"))
    check(f"{which}: W -> W records", torch.equal(global_records(back), want_rec))
    check(f"{which}: W -> W dense state", same(dense(back), want_dense))

    if rank == 0:                                              # W -> 1, then its save for 1 -> W
        one = made(False, 7)
        ck.load_checkpoint(one, os.path.join(root, "w"))
        check(f"{which}: W -> 1 records", torch.equal(global_records(one), want_rec))
        check(f"{which}: W -> 1 dense state", same(dense(one), want_dense))
        ck.save_checkpoint(one, os.path.join(root, "one"), step=2)
    dist.barrier()
    again = made(True, 9)                                      # 1 -> W
    meta = ck.load_checkpoint(again, os.path.join(root, "one"))
    check(f"{which}: 1 -> W records", meta["world"] == 1 and torch.equal(global_records(again), want_rec))
    check(f"{which}: 1 -> W dense state", same(dense(again), want_dense))

    flag_t = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag_t, op=dist.ReduceOp.MIN)
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0 if int(flag_t.item()) == 1 else 1)


if __name__ == "__main__":
    main()
