"""Multi-valued fields in the AutoInt trainer (AutoIntConfig.bag_size): the bag mean inside the tcgen05 forward's tile
loader (rs_interacting_fwd_gather_bag) bit for bit against rs_embed_bag_fwd_ld + rs_interacting_fwd, the bag trainer
against the single-valued one on collapsed bags, against the oracle, and its state (capture, fit_host, checkpoints)."""
import numpy as np
import pytest

from util import REL_BF16, REL_F32, assert_close, interacting_params

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

f64 = lambda a: np.asarray(a, np.float64)


def _bag_ids(rng, B, K, hi=2 ** 40, kinds=("full", "padded", "empty", "dup")):
    """[B, sum K] ids: every bag full, partly padded, empty or with a repeated id (fields with K = 1: full or empty)."""
    S = int(sum(K))
    ids = np.full((B, S), -1, np.int64)
    off = np.concatenate([[0], np.cumsum(K)])
    for f, k in enumerate(K):
        kind = rng.choice(kinds, size=B)
        vals = rng.integers(0, hi, size=(B, k))
        for b in range(B):
            row = vals[b].copy()
            if kind[b] == "padded" and k > 1:
                row[rng.random(k) < 0.5] = -1
            elif kind[b] == "empty":
                row[:] = -1
            elif kind[b] == "dup" and k > 1:
                row[rng.integers(0, k, size=k // 2 + 1)] = row[0]
            ids[b, off[f]:off[f + 1]] = row
    return ids


def _bag_mean_np(table, ids, K, rows, base):
    """fp32 sum of the valid rows in slot order, times float32(1 / count): embed_bag_fwd_kernel's arithmetic."""
    B, F, d = ids.shape[0], len(K), table.shape[1]
    off = np.concatenate([[0], np.cumsum(K)])
    X = np.zeros((B, F, d), np.float32)
    inv = np.zeros((B, F), np.float32)
    occ_rows, occ_bag = [], []
    for f in range(F):
        acc = np.zeros((B, d), np.float32)
        cnt = np.zeros(B, np.int64)
        for k in range(off[f], off[f + 1]):
            i = ids[:, k]
            ok = i >= 0
            r = base[f] + np.where(ok, i, 0) % rows[f]
            acc = np.where(ok[:, None], acc + table[r], acc)
            cnt += ok
            occ_rows.append(np.where(ok, r, -1)); occ_bag.append(np.arange(B) * F + f)
        inv[:, f] = np.where(cnt > 0, np.float32(1) / np.maximum(cnt, 1).astype(np.float32), np.float32(0))
        X[:, f] = acc * inv[:, f:f + 1]
    return X, inv, np.stack(occ_rows, 1).reshape(-1), np.stack(occ_bag, 1).reshape(-1)


LAYOUTS = {"k1": lambda rng, F: [1] * F, "mixed": lambda rng, F: [int(k) for k in rng.integers(1, 9, size=F)],
           "k32": lambda rng, F: [32 if f == F // 2 else 1 for f in range(F)]}


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("F", [13, 39, 48])
@pytest.mark.parametrize("B", [1, 3, 1000, 8192])
def test_fwd_gather_bag_bit_exact(cuda_dev, B, F, layout):
    from recommendsystem_b200 import cabi, ops
    rng = np.random.default_rng(B * 100 + F)
    K = LAYOUTS[layout](rng, F)
    S, D, U, H, L = sum(K), 16, 16, 2, 3
    rows = rng.integers(3, 5000, size=F).astype(np.int64)
    base = np.concatenate([[0], np.cumsum(rows)[:-1]]).astype(np.int64)
    rec = torch.randn(int(rows.sum()), 3, D, device=cuda_dev) * 0.3
    table = rec[:, 0, :]                                      # [w | m | v] records: row stride 3 D
    ids = torch.from_numpy(_bag_ids(rng, B, K)).to(cuda_dev)
    t = lambda a: torch.from_numpy(np.asarray(a)).to(cuda_dev)
    off, base_t, rows_t = t(np.concatenate([[0], np.cumsum(K)]).astype(np.int64)), t(base), t(rows)
    offsets = t(np.append((np.arange(B, dtype=np.int64)[:, None] * S + np.asarray(off.cpu())[None, :F]).reshape(-1), B * S))
    W, b, g, be = (t(a) for a in interacting_params(rng, D, U))
    p = lambda x: x.data_ptr()

    def outs():
        return (torch.empty(B, F, D, dtype=torch.bfloat16, device=cuda_dev), torch.empty(B * S, dtype=torch.int64,
                device=cuda_dev).fill_(7), torch.full((B * F,), 5.0, device=cuda_dev),
                torch.empty(B, F, U, dtype=torch.bfloat16, device=cuda_dev),
                torch.zeros(L * B * F * (U + 4), device=cuda_dev))      # activations, then the softmax statistics
    X1, k1, i1, y1, s1 = outs()
    cabi.call("rs_embed_bag_fwd_ld", p(table), table.stride(0), p(ids), p(offsets), p(base_t), p(rows_t), B * F, F, D,
              p(X1), cabi.RS_BF16, p(k1), p(i1), ops._stream())
    cabi.call("rs_interacting_fwd", p(X1), D, 0, cabi.RS_BF16, p(W), p(b), p(g), p(be), 1e-3, p(y1), U, 0, p(s1), B, F, D,
              U, H, L, 1, 1, ops._stream())
    X2, k2, i2, y2, s2 = outs()
    cabi.call("rs_interacting_fwd_gather_bag", p(table), table.stride(0), p(ids), p(off), p(base_t), p(rows_t), p(X2), D,
              0, p(k2), p(i2), cabi.RS_BF16, p(W), p(b), p(g), p(be), 1e-3, p(y2), U, 0, p(s2), B, F, S, D, U, H, L, 1,
              ops._stream())
    torch.cuda.synchronize()
    for a, c, what in ((X1, X2, "X"), (k1, k2, "keys"), (i1, i2, "inv_cnt"), (y1, y2, "y"), (s1, s2, "saved")):
        assert torch.equal(a.view(torch.int16) if a.dtype == torch.bfloat16 else a,
                           c.view(torch.int16) if c.dtype == torch.bfloat16 else c), what
    # and the bag mean itself against numpy (fp32 sum in slot order, times 1 / count, RNE to bf16)
    Xr, inv, _, _ = _bag_mean_np(table.cpu().numpy(), ids.cpu().numpy(), K, rows, base)
    assert torch.equal(X2.cpu(), torch.from_numpy(Xr).to(torch.bfloat16))
    assert np.array_equal(i2.cpu().numpy(), inv.reshape(-1))


def _cfg(dtype, K, id_map="mod", B=512, **kw):
    from recommendsystem_b200.autoint import AutoIntConfig
    rng = np.random.default_rng(5)
    F = len(K)
    return AutoIntConfig(num_fields=F, rows_per_field=[int(r) for r in rng.integers(2000, 6000, size=F)], embed_dim=16,
                         unit_num=16, head_num=2, layer_num=3, mlp_hidden=(256, 128), batch=B, dtype=dtype,
                         lr_dense=1e-3, lr_sparse=1e-2, bag_size=K, id_map=id_map, **kw)


def cfg_fields(K):
    return [f for f, k in enumerate(K) for _ in range(k)]


def _mixed_K(F=39, seed=3):
    return [int(k) for k in np.random.default_rng(seed).integers(1, 9, size=F)]


def _records_by_key(tr, keys, fields):
    """(mapped?, [w|m|v] records, show counts) of the (field, id) pairs of `keys` ([N, len(fields)] ids), through the
    trainer's own row numbers (hash mode: a row's number depends on the order the insert threads won their atomics)."""
    if tr.idmap is None:
        rows = torch.from_numpy(tr.base_host[None, fields] + keys % tr.rows_host[None, fields]).to(tr.dev).reshape(-1)
        return np.ones(rows.numel(), bool), tr.arena[rows].cpu().numpy(), None
    r = tr.idmap.resolve(torch.from_numpy(keys).to(tr.dev).contiguous(), tr.idmap.fields(fields), insert=False).reshape(-1)
    ok = r >= 0
    return ok.cpu().numpy(), tr.arena[r[ok]].cpu().numpy(), tr.idmap.show[r[ok]].cpu().numpy()


@pytest.mark.parametrize("id_map", ["mod", "hash"])
@pytest.mark.parametrize("mode", ["bf16_fused_graph", "bf16_unfused", "f32"])
def test_collapsed_bags_equal_single_valued(cuda_dev, mode, id_map):
    """Every bag holds exactly one valid id at a random slot: the bag trainer equals the single-valued trainer on the
    collapsed [B, F] ids bit for bit (the mean of one row is the row, inv = 1, and slot positions order like b F + f)."""
    from recommendsystem_b200.autoint import AutoIntTrainer
    K = _mixed_K()
    F, B = len(K), 512
    kw = {"fuse_embedding": mode != "bf16_unfused"}
    a = AutoIntTrainer(_cfg("f32" if mode == "f32" else "bf16", [1] * F, id_map, B, **kw), cuda_dev)
    b = AutoIntTrainer(_cfg("f32" if mode == "f32" else "bf16", K, id_map, B, **kw), cuda_dev)
    assert b.bag and not a.bag
    if mode == "bf16_fused_graph":
        assert b.fused and b.fuse_tower
        a.capture(); b.capture()
    rng = np.random.default_rng(17)
    off = np.concatenate([[0], np.cumsum(K)])
    seen = []
    for _ in range(3):
        one = rng.integers(0, 2 ** 40, size=(B, F)).astype(np.int64)
        bags = np.full((B, sum(K)), -1, np.int64)
        for f in range(F):
            bags[np.arange(B), off[f] + rng.integers(0, K[f], size=B)] = one[:, f]
        y = (rng.random((B, 1)) < 0.25).astype(np.float32)
        la = float(a.step(torch.from_numpy(one).to(cuda_dev), torch.from_numpy(y).to(cuda_dev)))
        lb = float(b.step(torch.from_numpy(bags).to(cuda_dev), torch.from_numpy(y).to(cuda_dev)))
        assert la == lb
        seen.append(one)
    torch.cuda.synchronize()
    seen = np.concatenate(seen)
    oka, ra, sa = _records_by_key(a, seen, list(range(F)))
    okb, rb, sb = _records_by_key(b, seen, list(range(F)))
    assert oka.all() and okb.all() and np.array_equal(ra, rb)
    if id_map == "hash":
        assert np.array_equal(sa, sb)
        assert torch.equal(a.idmap.counters, b.idmap.counters)
    else:
        assert torch.equal(a.arena, b.arena)
    for n in ("flat", "flat_m", "flat_v", "flat_bf16", "adam_scalars"):
        assert torch.equal(getattr(a, n), getattr(b, n)), n


def _oracle_params(P):
    return dict(Wqkvr=f64(P["Wqkvr"]), bqkvr=f64(P["bqkvr"]), gamma=f64(P["gamma"]), beta=f64(P["beta"]),
                mlp_W=[f64(P["mlp_W0"]), f64(P["mlp_W1"])], mlp_b=[f64(P["mlp_b0"]), f64(P["mlp_b1"])],
                out_W=f64(P["out_W"]), out_b=f64(P["out_b"]))


def test_bag_step_fp32_against_oracle(cuda_dev):
    from oracle import oracle_np as onp
    from recommendsystem_b200.autoint import AutoIntTrainer
    K = [1, 4, 2, 8, 1, 3, 1, 6, 2, 1, 5, 1, 2]
    B, F, d = 96, len(K), 16
    tr = AutoIntTrainer(_cfg("f32", K, B=B), cuda_dev)
    rng = np.random.default_rng(23)
    P0 = tr.dense_state()
    w0, m0, v0 = (t.cpu().numpy().copy() for t in (tr.table, tr.table_m, tr.table_v))
    step0 = int(tr.adam_scalars[0].item())
    ids = _bag_ids(rng, B, K)
    y = (rng.random((B, 1)) < 0.25).astype(np.float32)
    loss = float(tr.step(torch.from_numpy(ids).to(cuda_dev), torch.from_numpy(y).to(cuda_dev)))
    torch.cuda.synchronize()
    X, inv, occ_rows, occ_bag = _bag_mean_np(w0, ids, K, tr.rows_host, tr.base_host)
    assert np.array_equal(tr.X.cpu().numpy(), X)
    res = onp.autoint_fwd_bwd(f64(X), _oracle_params(P0), f64(y), 2, 3, 1e-3)
    assert abs(loss - res["loss"]) <= REL_F32 * abs(res["loss"])
    assert_close(tr.dX.cpu().numpy(), res["dX"], REL_F32, "dX")
    # sparse Adam over one gradient row per valid occurrence: dX[b, f] / count
    ok = occ_rows >= 0
    dX = tr.dX.cpu().numpy().reshape(B * F, d)
    g = dX[occ_bag[ok]] * inv.reshape(-1)[occ_bag[ok], None]
    _, _, corr = onp.adam_scalars(step0 + 1, 0.9, 0.999)
    w2, _, _ = onp.sparse_adam(f64(w0), f64(m0), f64(v0), occ_rows[ok], g, 1e-2, 0.9, 0.999, 1e-8, float(corr))
    assert_close(tr.table.cpu().numpy(), w2, REL_F32, "table after sparse Adam")
    untouched = np.ones(len(w0), bool)
    untouched[occ_rows[ok]] = False
    assert np.array_equal(tr.table.cpu().numpy()[untouched], w0[untouched])
    # predict: the oracle forward on the bag means of the updated tables
    ids2 = _bag_ids(rng, B, K)
    p = tr.predict(torch.from_numpy(ids2).to(cuda_dev)).cpu().numpy()
    X2, _, _, _ = _bag_mean_np(tr.table.cpu().numpy(), ids2, K, tr.rows_host, tr.base_host)
    res2 = onp.autoint_fwd_bwd(f64(X2), _oracle_params(tr.dense_state()), f64(y), 2, 3, 1e-3)
    assert_close(p, np.clip(res2["p_raw"], 1e-6, 1.0), REL_F32, "predict")


def test_bag_step_bf16_bench_size(cuda_dev):
    """B = 8192, 26 single-valued fields and 13 with K = 8 (lengths uniform in [0, 8]), fused loader: X bit-exact, loss
    and logits within 1e-2 of the fp64 oracle on the same tables, dX direction."""
    from oracle import oracle_np as onp
    from recommendsystem_b200.autoint import AutoIntTrainer
    K = [1] * 26 + [8] * 13
    B = 8192
    tr = AutoIntTrainer(_cfg("bf16", K, B=B), cuda_dev)
    assert tr.fused
    rng = np.random.default_rng(29)
    ids = rng.integers(0, 2 ** 40, size=(B, sum(K))).astype(np.int64)
    n = rng.integers(0, 9, size=(B, 13))
    ids[:, 26:] = np.where(np.arange(8)[None, None, :] < n[:, :, None], ids[:, 26:].reshape(B, 13, 8), -1).reshape(B, -1)
    y = (rng.random((B, 1)) < 0.25).astype(np.float32)
    P0 = tr.dense_state()
    w0 = tr.table.cpu().numpy().copy()
    loss = float(tr.step(torch.from_numpy(ids).to(cuda_dev), torch.from_numpy(y).to(cuda_dev)))
    torch.cuda.synchronize()
    X, _, _, _ = _bag_mean_np(w0, ids, K, tr.rows_host, tr.base_host)
    Xb = tr.X.float().cpu().numpy()
    assert np.array_equal(Xb, torch.from_numpy(X).to(torch.bfloat16).float().numpy())
    res = onp.autoint_fwd_bwd(f64(Xb), _oracle_params(P0), f64(y), 2, 3, 1e-3)
    assert abs(loss - res["loss"]) <= REL_BF16 * abs(res["loss"])
    assert_close(tr.p_raw.float().cpu().numpy(), res["p_raw"], REL_BF16, "bf16 logits")
    a, r = f64(tr.dX.float().cpu().numpy()).ravel(), f64(res["dX"]).ravel()
    assert float(a @ r / (np.linalg.norm(a) * np.linalg.norm(r))) >= 0.99


def test_bag_predict_hash_unseen_ids_are_padding(cuda_dev):
    from recommendsystem_b200.autoint import AutoIntTrainer
    K = [2, 3, 1]
    B = 8
    tr = AutoIntTrainer(_cfg("f32", K, "hash", B=B), cuda_dev)
    rng = np.random.default_rng(31)
    ids = rng.integers(0, 2 ** 40, size=(B, 6)).astype(np.int64)
    tr.step(torch.from_numpy(ids).to(cuda_dev), torch.zeros(B, 1, device=cuda_dev))
    q = ids.copy()
    q[:, 1] = 2 ** 41 + np.arange(B)                         # field 0: one seen id, one unseen
    q[:, 2:5] = 2 ** 42 + np.arange(B * 3).reshape(B, 3)     # field 1: nothing seen -> zeros
    tr.predict(torch.from_numpy(q).to(cuda_dev))
    torch.cuda.synchronize()
    r = tr.idmap.resolve(torch.from_numpy(ids[:, [0]]).to(cuda_dev).contiguous(), tr.idmap.fields([0]), insert=False)
    assert torch.equal(tr.X[:, 0], tr.table[r.reshape(-1)])
    assert not bool(tr.X[:, 1].any())


def test_bag_capture_fit_host_and_resume(cuda_dev, tmp_path):
    """capture() undoes its warm-up step exactly; fit_host equals sequential steps; train(2) -> save -> load ->
    train(2) equals train(4), in hash mode with an evict in between."""
    from recommendsystem_b200.autoint import AutoIntTrainer
    from recommendsystem_b200 import checkpoint as ck
    K = _mixed_K(seed=7)
    B = 256
    cfg = _cfg("bf16", K, "hash", B=B)
    rng = np.random.default_rng(37)
    # (ids below every field's capacity: which ids would overflow a full field depends on the insert order)
    batches = [(torch.from_numpy(_bag_ids(rng, B, K, hi=1000)).pin_memory(),
                torch.from_numpy((rng.random((B, 1)) < 0.25).astype(np.float32)).pin_memory()) for _ in range(4)]
    state = lambda t: (t.arena.clone(), t.idmap.show.clone(), t.idmap.counters.clone(), t.flat.clone(),
                       t.flat_m.clone(), t.flat_v.clone(), t.adam_scalars.clone())
    slots = np.concatenate([bt[0].numpy() for bt in batches])
    slot_fields = cfg_fields(K)
    a = AutoIntTrainer(cfg, cuda_dev)
    a.step(batches[0][0].to(cuda_dev), batches[0][1].to(cuda_dev))
    a.ids.copy_(batches[1][0])                               # the warm-up trains on these (new ids too)
    s0 = state(a)
    a.capture()
    for x, y in zip(s0, state(a)):
        assert torch.equal(x, y)
    a2 = AutoIntTrainer(cfg, cuda_dev)
    a2.step(batches[0][0].to(cuda_dev), batches[0][1].to(cuda_dev))
    seq = [a.step_from_host(*bt) for bt in batches[1:3]]
    a.evict(1.5, 0.9)
    seq += [a.step_from_host(*batches[3])]
    pipe = list(a2.fit_host(iter(batches[1:3])))
    assert seq[:2] == pipe
    ck.save_checkpoint(a2, tmp_path / "ck", step=3)
    assert ck.read_meta(tmp_path / "ck")["config"]["bag_size"] == K
    c = AutoIntTrainer(cfg, cuda_dev)
    c.capture()
    ck.load_checkpoint(c, tmp_path / "ck")
    c.evict(1.5, 0.9)
    assert [c.step_from_host(*batches[3])] == seq[2:]
    # per key: the same ids mapped, with the same records and shows; the same dense state
    for x, y in zip(_records_by_key(a, slots, slot_fields), _records_by_key(c, slots, slot_fields)):
        assert np.array_equal(x, y)
    assert torch.equal(a.idmap.counters, c.idmap.counters) and torch.equal(a.idmap.evicted, c.idmap.evicted)
    for n in ("flat", "flat_m", "flat_v", "flat_bf16", "adam_scalars"):
        assert torch.equal(getattr(a, n), getattr(c, n)), n


def test_bag_shape_refusals(cuda_dev):
    from recommendsystem_b200.autoint import AutoIntTrainer
    tr = AutoIntTrainer(_cfg("f32", [1, 3, 2], B=4), cuda_dev)
    bad = torch.zeros(4, 3, dtype=torch.int64, device=cuda_dev)
    with pytest.raises(ValueError, match="sum\\(bag_size\\)"):
        tr.step(bad, torch.zeros(4, 1, device=cuda_dev))
    with pytest.raises(ValueError, match="sum\\(bag_size\\)"):
        tr.predict(bad)
    with pytest.raises(ValueError, match="sum\\(bag_size\\)"):
        list(tr.fit_host([(bad.cpu(), torch.zeros(4, 1))]))
