"""The collision-free id map (recommendsystem_b200.idmap, rs_idmap_* in include/rs_b200.h) and the id_map="hash" mode
of EmbeddingFeatures / AutoIntTrainer.

Method of the parity tests: hash mode is run against mod mode on the same batches, the mod side seeing the ids
remapped on the host to dense indices 0..n-1 per field and its table rows seeded, at those indices, with the records
the hash map's init rule produces for the same keys.  Row numbers differ between the two; everything computed must
not: outputs, losses, dense parameters and every key's [w | m | v] record are compared bit for bit."""
import numpy as np
import pytest
import torch

M64 = (1 << 64) - 1
GOLDEN = 0x9E3779B97F4A7C15


def mix64(z):
    z &= M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def init_rule(seed, field, key, d, scale):
    """numpy restatement of the init rule of a new row (float64)."""
    base = mix64(mix64((seed + GOLDEN * (field + 1)) & M64) ^ (key & M64))
    out = np.zeros(d)
    for p in range((d + 1) // 2):
        r = mix64(base + GOLDEN * (p + 1))
        u1 = ((r >> 40) + 1) * 2.0 ** -24
        u2 = ((r & 0xFFFFFFFF) >> 8) * 2.0 ** -24
        rad = np.sqrt(-2.0 * np.log(u1))
        out[2 * p] = scale * rad * np.cos(2 * np.pi * u2)
        if 2 * p + 1 < d:
            out[2 * p + 1] = scale * rad * np.sin(2 * np.pi * u2)
    return out


def _map(rows, dev, d=4, seed=5, scale=0.1):
    from recommendsystem_b200.idmap import IdMap
    arena = torch.zeros(int(sum(rows)), 3, d, device=dev)
    return IdMap(rows, dev, seed, scale, arena[:, 0, :], [(arena[:, 1, :], 0.0), (arena[:, 2, :], 0.0)]), arena


def _state(m):
    return m.counters.clone(), m.key_of_row.clone(), m.slots.clone()


# ---------------------------------------------------------------------------------------------------- 1. map kernel
@pytest.mark.gpu
def test_map_kernel_distinct_rows_duplicates_padding(cuda_dev):
    rows = [64, 100, 50]
    m, _ = _map(rows, cuda_dev)
    B = 4096
    special = [0, 64, 128, 2 ** 32, 2 ** 32 + 64, 2 ** 40 + 1, 2 ** 62 + 3, 7 + 64]   # congruent mod 64 / >= 2^32
    g = np.random.default_rng(0)
    col = np.full(B, 7, np.int64)                                   # one hot key at thousands of positions
    col[:len(special)] = special
    col[100:130] = g.integers(0, 2 ** 63 - 1, 30)
    col[200:240] = -1                                               # padding
    ids = np.stack([col, col, g.permutation(col)], 1)              # the same ids in every field, shuffled in one
    t = torch.from_numpy(ids).to(cuda_dev)
    fields = m.fields([0, 1, 2])
    r = m.resolve(t, fields, insert=True).cpu().numpy()
    for f in range(3):
        keys, rr = ids[:, f], r[:, f]
        assert (rr[keys < 0] == -1).all()
        distinct = sorted(set(keys[keys >= 0].tolist()))
        rows_of = {}
        for k, x in zip(keys, rr):
            if k >= 0:
                assert rows_of.setdefault(int(k), int(x)) == int(x), "one key, one row"
        got = [rows_of[k] for k in distinct]
        assert len(set(got)) == len(distinct), "distinct keys, distinct rows"
        assert all(m.base[f] <= x < m.base[f] + rows[f] for x in got)
        kor = m.key_of_row.cpu().numpy()
        assert all(kor[rows_of[k]] == k for k in distinct)
    st = m.stats()
    assert st["rows_used"] == [len(set(ids[ids[:, f] >= 0, f].tolist())) for f in range(3)] and st["overflow"] == [0] * 3
    before = _state(m)
    r2 = m.resolve(t, fields, insert=True).cpu().numpy()
    assert (r2 == r).all()
    assert all(torch.equal(a, b) for a, b in zip(before, _state(m))), "a second call allocates nothing"
    unseen = torch.from_numpy(g.integers(2 ** 50, 2 ** 60, (64, 3))).to(cuda_dev)
    assert (m.resolve(unseen, fields, insert=False) == -1).all()
    assert all(torch.equal(a, b) for a, b in zip(before, _state(m))), "lookup-only leaves the map unchanged"


# ---------------------------------------------------------------------------------------------------------- 2. init
@pytest.mark.gpu
@pytest.mark.parametrize("opt", ["adam", "adagrad_row", "adagrad_elem"])
def test_init_rule_and_order_independence(cuda_dev, opt):
    from recommendsystem_b200.idmap import IdMap
    d, rows, seed, scale = 16, [300, 300], 1234567, 0.05
    g = np.random.default_rng(1)
    keys = np.stack([g.integers(0, 2 ** 63 - 1, 256), g.integers(0, 2 ** 20, 256)], 1)

    def build():
        total = sum(rows)
        if opt == "adam":
            rec = torch.full((total, 3, d), float("nan"), device=cuda_dev)        # dirty memory
            w, states = rec[:, 0, :], [(rec[:, 1, :], 0.0), (rec[:, 2, :], 0.0)]
        else:
            w = torch.full((total, d), 7.0, device=cuda_dev)
            g2 = torch.full((total, d) if opt == "adagrad_elem" else (total,), -3.0, device=cuda_dev)
            rec, states = (w, g2), [(g2, 0.1)]
        return IdMap(rows, cuda_dev, seed, scale, w, states), w, rec, states

    def record(rec, r):
        if opt == "adam":
            return rec[r].reshape(-1)
        return torch.cat([rec[0][r].reshape(-1), rec[1][r].reshape(-1)])

    a, wa, reca, sa = build()
    b, wb, recb, sb = build()
    fields = a.fields([0, 1])
    ra = a.resolve(torch.from_numpy(keys).to(cuda_dev), fields, insert=True)
    perm = g.permutation(len(keys))
    kb = torch.from_numpy(keys[perm]).to(cuda_dev)
    b.resolve(kb[:100].contiguous(), fields, insert=True)          # other order, two batches
    b.resolve(kb[100:].contiguous(), fields, insert=True)
    rb = b.resolve(torch.from_numpy(keys).to(cuda_dev), fields, insert=False)
    w_host = wa.cpu().numpy()
    for f in range(2):
        for i in range(0, len(keys), 17):
            k, x = int(keys[i, f]), int(ra[i, f])
            want = init_rule(seed, f, k, d, scale)
            np.testing.assert_allclose(w_host[x], want, rtol=2e-6, atol=1e-9 * scale)
    for i in range(len(keys)):
        for f in range(2):
            assert torch.equal(record(reca, int(ra[i, f])), record(recb, int(rb[i, f]))), "bitwise per key"
    used = ra[ra >= 0].unique()
    for t, v in sa:
        assert (t[used] == v).all(), "optimizer state at its initial value"


# ------------------------------------------------------------------------------------------------------ 3. overflow
@pytest.mark.gpu
def test_overflow(cuda_dev):
    m, _ = _map([64], cuda_dev)
    keys = np.random.default_rng(2).choice(2 ** 40, 200, replace=False).astype(np.int64)
    t = torch.from_numpy(keys).reshape(-1, 1).to(cuda_dev)
    r = m.resolve(t, m.fields([0]), insert=True)
    assert int((r >= 0).sum()) == 64 and m.stats()["rows_used"] == [64]
    assert m.stats()["overflow"] == [136]
    assert sorted(r[r >= 0].tolist()) == list(range(64))
    r2 = m.resolve(t, m.fields([0]), insert=True)
    assert torch.equal(r, r2) and m.stats()["overflow"] == [272] and m.stats()["rows_used"] == [64]
    m.resolve(t, m.fields([0]), insert=False)                      # inference does not count
    assert m.stats()["overflow"] == [272]


# ------------------------------------------------------------------------------------- 4. EmbeddingFeatures parity
def _remap(batches, keys_of):
    """host ids -> dense per-column indices (first appearance order); `keys_of[c]` collects the keys."""
    out = []
    for b in batches:
        o = {}
        for c, v in b.items():
            idx = keys_of.setdefault(c, {})
            if isinstance(v, tuple):
                vals = v[0]
            else:
                vals = v
            flat = vals.reshape(-1)
            mapped = np.array([idx.setdefault(int(k), len(idx)) if k >= 0 else -1 for k in flat], np.int64)
            mapped = mapped.reshape(vals.shape)
            o[c] = (mapped, v[1]) if isinstance(v, tuple) else mapped
        out.append(o)
    return out


def _dev(b, dev):
    return {c: (tuple(torch.from_numpy(x).to(dev) for x in v) if isinstance(v, tuple) else torch.from_numpy(v).to(dev))
            for c, v in b.items()}


def _seed_mod_rows(hash_layer, mod_layer, keys_of, cols):
    """Seed the mod layer's rows 0..n-1 of every column with the records the hash map's init gives the same keys (the
    C-ABI insert on a scratch map of the same geometry)."""
    from recommendsystem_b200.api.embedding import Adam
    from recommendsystem_b200.idmap import IdMap
    dev, d = hash_layer.dev, hash_layer.d
    total = int(hash_layer.rows.sum())
    if isinstance(hash_layer.opt, Adam):
        rec = torch.zeros(total, 3, d, device=dev)
        w, states = rec[:, 0, :], [(rec[:, 1, :], 0.0), (rec[:, 2, :], 0.0)]
    else:
        w = torch.zeros(total, d, device=dev)
        g2 = torch.zeros_like(mod_layer.g2sum)
        states = [(g2, float(hash_layer.opt.initial_g2sum))]
    scratch = IdMap(hash_layer.rows, dev, hash_layer.idmap.seed, hash_layer.idmap.scale, w, states)
    for ci, c in enumerate(cols):
        ks = sorted(keys_of[c].items(), key=lambda kv: kv[1])
        t = torch.tensor([k for k, _ in ks], dtype=torch.int64, device=dev).reshape(-1, 1)
        r = scratch.resolve(t, scratch.fields([ci]), insert=True).reshape(-1)
        dst = int(mod_layer.base[ci]) + torch.arange(len(ks), device=dev)
        mod_layer.table[dst] = w[r]
        if isinstance(hash_layer.opt, Adam):
            mod_layer.m[dst] = 0.0
            mod_layer.v[dst] = 0.0
        else:
            mod_layer.g2sum[dst] = states[0][0][r]


def _records(layer, rows):
    from recommendsystem_b200.api.embedding import Adam
    if isinstance(layer.opt, Adam):
        return layer.arena[rows].reshape(len(rows), -1)
    g2 = layer.g2sum[rows].reshape(len(rows), -1)
    return torch.cat([layer.table[rows], g2], 1)


def _opt(kind):
    from recommendsystem_b200.api.embedding import AdaGrad, Adam
    if kind == "adam":
        return Adam(learning_rate=0.01)
    return AdaGrad(learning_rate=0.05, initial_g2sum=0.1, initial_scale=0.1, per_element=(kind == "adagrad_elem"))


@pytest.mark.gpu
@pytest.mark.parametrize("opt", ["adam", "adagrad_row", "adagrad_elem"])
def test_embedding_features_hash_matches_remapped_mod(cuda_dev, opt):
    from recommendsystem_b200.api.embedding import EmbeddingFeatures, category_column, embedding_column
    d, B, T, bag, cap = 8, 64, 5, 3, 512
    cols = ["a", "b", "s", "bag", "csr"]

    def layer(mode):
        ec = [embedding_column(category_column("a", cap), d), embedding_column(category_column("b", cap), d),
              embedding_column(category_column("s", cap), d, combiner=None, seq_max_len=T),
              embedding_column(category_column("bag", cap), d), embedding_column(category_column("csr", cap), d)]
        return EmbeddingFeatures(ec, _opt(opt), device=str(cuda_dev), seed=42, id_map=mode)

    g = np.random.default_rng(3)
    pools = {c: g.integers(0, 2 ** 63 - 1, 150) for c in cols}
    pools["a"][:4] = [5, 5 + cap, 2 ** 33 + 5, 2 ** 33 + 5 + cap]       # congruent mod the bucket size
    batches = []
    for _ in range(3):
        bt = {"a": g.choice(pools["a"], B), "b": g.choice(pools["b"], B)}
        s = g.choice(pools["s"], (B, T))
        s[g.random((B, T)) < 0.3] = -1
        bt["s"] = s
        bg = g.choice(pools["bag"], (B, bag))
        bg[g.random((B, bag)) < 0.2] = -1
        bt["bag"] = bg
        lens = g.integers(0, 4, B)
        offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        bt["csr"] = (g.choice(pools["csr"], int(offs[-1])).astype(np.int64), offs)
        batches.append(bt)
    grads = []
    for _ in range(3):
        gg = {c: torch.from_numpy(g.standard_normal((B, d)).astype(np.float32)).to(cuda_dev) for c in ("a", "b", "bag", "csr")}
        gg["s"] = torch.from_numpy(g.standard_normal((B, T, d)).astype(np.float32)).to(cuda_dev)
        grads.append(gg)
    keys_of = {}
    remapped = _remap(batches, keys_of)
    h, md = layer("hash"), layer("mod")
    _seed_mod_rows(h, md, keys_of, cols)
    for st in range(3):
        oh, om = h(_dev(batches[st], cuda_dev)), md(_dev(remapped[st], cuda_dev))
        for c in cols:
            if c == "s":
                assert torch.equal(oh[c][0], om[c][0]) and torch.equal(oh[c][1], om[c][1]), (st, c)
            else:
                assert torch.equal(oh[c], om[c]), (st, c)
        h.backward(grads[st])
        md.backward(grads[st])
    for ci, c in enumerate(cols):
        ks = sorted(keys_of[c].items(), key=lambda kv: kv[1])
        t = torch.tensor([k for k, _ in ks], dtype=torch.int64, device=cuda_dev).reshape(-1, 1)
        rh = h.idmap.resolve(t, h.idmap.fields([ci]), insert=False).reshape(-1)
        assert (rh >= 0).all()
        rm = int(md.base[ci]) + torch.arange(len(ks), device=cuda_dev)
        assert torch.equal(_records(h, rh), _records(md, rm)), c
    assert h.idmap.stats()["rows_used"] == [len(keys_of[c]) for c in cols]


@pytest.mark.gpu
def test_overflowed_ids_train_like_padding(cuda_dev):
    """Capacity 64, 200 distinct ids: the overflowed lookups read zeros and update nothing — hash mode equals mod mode
    on the remapped ids with the overflowed ones replaced by padding."""
    from recommendsystem_b200.api.embedding import EmbeddingFeatures, category_column, embedding_column
    d, cap = 8, 64
    ec = lambda: [embedding_column(category_column("a", cap), d), embedding_column(category_column("b", cap), d)]
    h = EmbeddingFeatures(ec(), _opt("adam"), device=str(cuda_dev), seed=1, id_map="hash")
    md = EmbeddingFeatures(ec(), _opt("adam"), device=str(cuda_dev), seed=1)
    g = np.random.default_rng(4)
    a = g.choice(2 ** 40, 200, replace=False).astype(np.int64)
    b = g.choice(a[:20], 200)
    out = h({"a": torch.from_numpy(a).to(cuda_dev), "b": torch.from_numpy(b).to(cuda_dev)})
    rows_a = h.idmap.resolve(torch.from_numpy(a).reshape(-1, 1).to(cuda_dev), h.idmap.fields([0]), insert=False)
    kept = (rows_a.reshape(-1) >= 0).cpu().numpy()
    assert kept.sum() == 64 and h.idmap.stats()["overflow"] == [136, 0]
    assert (out["a"][torch.from_numpy(~kept).to(cuda_dev)] == 0).all()
    # the mod reference: kept ids in first-appearance order, overflowed ones as padding
    keys_of = {}
    a_pad = np.where(kept, a, -1)
    rem = _remap([{"a": a_pad, "b": b}], keys_of)[0]
    _seed_mod_rows(h, md, keys_of, ["a", "b"])
    om = md(_dev(rem, cuda_dev))
    assert torch.equal(out["a"], om["a"]) and torch.equal(out["b"], om["b"])
    gr = {c: torch.from_numpy(g.standard_normal((200, d)).astype(np.float32)).to(cuda_dev) for c in ("a", "b")}
    h.backward(gr)
    md.backward(gr)
    for ci, c in enumerate(["a", "b"]):
        ks = sorted(keys_of[c].items(), key=lambda kv: kv[1])
        t = torch.tensor([k for k, _ in ks], dtype=torch.int64, device=cuda_dev).reshape(-1, 1)
        rh = h.idmap.resolve(t, h.idmap.fields([ci]), insert=False).reshape(-1)
        rm = int(md.base[ci]) + torch.arange(len(ks), device=cuda_dev)
        assert torch.equal(_records(h, rh), _records(md, rm)), c


# ----------------------------------------------------------------------------------------- 5. AutoIntTrainer parity
def _autoint_pair(dev, dtype, fuse, B=256, F=39, cap=600, seed=9):
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    from recommendsystem_b200.idmap import IdMap
    g = np.random.default_rng(seed)
    pools = g.integers(0, 2 ** 63 - 1, (F, 400))
    batches = []
    for _ in range(3):
        ids = np.stack([g.choice(pools[f], B) for f in range(F)], 1)
        ids[g.random((B, F)) < 0.05] = -1
        batches.append((ids, (g.random((B, 1)) < 0.3).astype(np.float32)))
    # tower widths > 32: the bf16 weight-gradient GEMMs read MN-major operands, built for N > 32
    mk = lambda mode: AutoIntConfig(num_fields=F, rows_per_field=cap, batch=B, mlp_hidden=(128, 64), dtype=dtype,
                                    lr_dense=1e-3, lr_sparse=1e-2, seed=seed, fuse_embedding=fuse, id_map=mode)
    keys_of = {}
    rem = []
    for ids, _ in batches:
        r = np.full_like(ids, -1)
        for f in range(F):
            idx = keys_of.setdefault(f, {})
            r[:, f] = [idx.setdefault(int(k), len(idx)) if k >= 0 else -1 for k in ids[:, f]]
        rem.append(r)
    h = AutoIntTrainer(mk("hash"), dev)
    # the mod trainer's rows 0..n-1 of every field hold the records the hash init gives the same keys
    scratch_w = torch.zeros(h.total_rows, 16, device=dev)
    scratch = IdMap(h.rows_host, dev, h.cfg.seed, h.cfg.table_init_scale, scratch_w)
    tables = torch.zeros(h.total_rows, 16, device=dev)
    for f in range(F):
        ks = sorted(keys_of[f].items(), key=lambda kv: kv[1])
        t = torch.tensor([k for k, _ in ks], dtype=torch.int64, device=dev).reshape(-1, 1)
        r = scratch.resolve(t, scratch.fields([f]), insert=True).reshape(-1)
        tables[int(h.base_host[f]) + torch.arange(len(ks), device=dev)] = scratch_w[r]
    md = AutoIntTrainer(mk("mod"), dev, tables=tables)
    return h, md, batches, rem, keys_of


def _per_key(h, md, keys_of):
    for f, idx in keys_of.items():
        ks = sorted(idx.items(), key=lambda kv: kv[1])
        t = torch.tensor([k for k, _ in ks], dtype=torch.int64, device=h.dev).reshape(-1, 1)
        rh = h.idmap.resolve(t, h.idmap.fields([f]), insert=False).reshape(-1)
        assert (rh >= 0).all()
        rm = int(md.base_host[f]) + torch.arange(len(ks), device=h.dev)
        assert torch.equal(h.arena[rh], md.arena[rm]), f


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,fuse", [("bf16", True), ("bf16", False), ("f32", False)])
def test_autoint_hash_matches_remapped_mod(cuda_dev, dtype, fuse):
    h, md, batches, rem, keys_of = _autoint_pair(cuda_dev, dtype, fuse)
    assert h.fused == md.fused == (dtype == "bf16" and fuse)
    dev = cuda_dev
    lh = [float(h.step(torch.from_numpy(batches[0][0]).to(dev), torch.from_numpy(batches[0][1]).to(dev)))]
    lm = [float(md.step(torch.from_numpy(rem[0]).to(dev), torch.from_numpy(batches[0][1]).to(dev)))]
    # capture with step 2's ids in the static buffer: the undone warm-up step inserts new keys
    h.ids.copy_(torch.from_numpy(batches[1][0]).to(dev))
    md.ids.copy_(torch.from_numpy(rem[1]).to(dev))
    torch.cuda.synchronize()
    before = (h.idmap.counters.clone(), h.idmap.key_of_row.clone(), h.arena.clone())
    h.capture()
    md.capture()
    assert torch.equal(before[0], h.idmap.counters) and torch.equal(before[1], h.idmap.key_of_row)
    assert torch.equal(before[2], h.arena), "capture() leaves the records as they were"
    for st in (1, 2):
        lh.append(float(h.step(torch.from_numpy(batches[st][0]).to(dev), torch.from_numpy(batches[st][1]).to(dev))))
        lm.append(float(md.step(torch.from_numpy(rem[st]).to(dev), torch.from_numpy(batches[st][1]).to(dev))))
    assert lh == lm
    assert torch.equal(h.flat, md.flat) and torch.equal(h.flat_m, md.flat_m) and torch.equal(h.flat_v, md.flat_v)
    _per_key(h, md, keys_of)
    assert h.idmap.stats()["rows_used"] == [len(keys_of[f]) for f in range(h.cfg.num_fields)]


# --------------------------------------------------------------------------------------------------- 6. collisions
@pytest.mark.gpu
def test_congruent_ids_train_independently(cuda_dev):
    from recommendsystem_b200.api.embedding import EmbeddingFeatures, category_column, embedding_column
    R, d = 16, 8
    ids = torch.tensor([3, 3 + R], dtype=torch.int64, device=cuda_dev)
    gr = {"a": torch.tensor([[1.0] * d, [-1.0] * d], device=cuda_dev)}
    rows = {}
    for mode in ("hash", "mod"):
        e = EmbeddingFeatures([embedding_column(category_column("a", R), d)], _opt("adam"), device=str(cuda_dev),
                              id_map=mode)
        e({"a": ids})
        rows[mode] = e.touched_rows({"a": ids})
        e.backward(gr)
        if mode == "hash":
            r = e.idmap.resolve(ids.reshape(-1, 1), e.idmap.fields([0]), insert=False).reshape(-1)
            assert int(r[0]) != int(r[1])
            assert not torch.equal(e.table[r[0]], e.table[r[1]])
            with torch.no_grad():
                out = e({"a": ids})["a"]
            assert not torch.equal(out[0], out[1])
    assert rows["mod"].numel() == 1, "mod mode: the two ids share one row"


# ------------------------------------------------------------------------------------------------------- 7. predict
@pytest.mark.gpu
def test_predict_never_inserts(cuda_dev):
    from recommendsystem_b200.api.builders import AUTOINT
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    B, F = 64, 39
    tr = AutoIntTrainer(AutoIntConfig(num_fields=F, rows_per_field=100, batch=B, mlp_hidden=(32, 16), id_map="hash"),
                        cuda_dev)
    ids = torch.randint(0, 2 ** 62, (B, F), device=cuda_dev)
    p = tr.predict(ids)
    assert tr.idmap.stats()["rows_used"] == [0] * F and tr.idmap.stats()["overflow"] == [0] * F
    assert (tr.X == 0).all() and torch.isfinite(p).all()
    slots = [str(3000 + i) for i in range(6)]
    ret = AUTOINT(slots, [], False, dnn_hidden_units=(32, 16), bucket_size=50, device=str(cuda_dev), id_map="hash")
    inp = {s: torch.randint(0, 2 ** 62, (B,), device=cuda_dev) for s in slots}
    y = ret.model.predict(inp)
    assert y.shape == (B, 7) and torch.isfinite(y).all()
    emb = ret.model.emb
    assert emb.idmap.stats()["rows_used"] == [0] * 6
    with torch.no_grad():
        assert all((v == 0).all() for v in emb(inp).values())


# ---------------------------------------------------------------------------------------------------- 8. checkpoint
@pytest.mark.gpu
@pytest.mark.parametrize("capture", [False, True])
def test_checkpoint_resume_is_exact(cuda_dev, tmp_path, capture):
    from recommendsystem_b200 import checkpoint as ck
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    B, F = 128, 39
    cfg = lambda mode="hash": AutoIntConfig(num_fields=F, rows_per_field=300, batch=B, mlp_hidden=(32, 16),
                                            lr_dense=1e-3, lr_sparse=1e-2, id_map=mode, seed=5)
    g = np.random.default_rng(6)
    pool = g.integers(0, 2 ** 63 - 1, (F, 250))
    data = [(torch.from_numpy(np.stack([g.choice(pool[f], B) for f in range(F)], 1)).to(cuda_dev),
             torch.from_numpy((g.random((B, 1)) < 0.3).astype(np.float32)).to(cuda_dev)) for _ in range(4)]
    a = AutoIntTrainer(cfg(), cuda_dev)
    for ids, y in data:
        a.step(ids, y)
    b = AutoIntTrainer(cfg(), cuda_dev)
    for ids, y in data[:2]:
        b.step(ids, y)
    ck.save_checkpoint(b, tmp_path, step=2)
    assert ck.read_meta(tmp_path)["id_map"] == "hash"
    c = AutoIntTrainer(cfg(), cuda_dev)
    ck.load_checkpoint(c, tmp_path)
    assert torch.equal(c.idmap.counters, b.idmap.counters) and torch.equal(c.idmap.key_of_row, b.idmap.key_of_row)
    if capture:
        c.ids.copy_(data[2][0])
        c.capture()
    for ids, y in data[2:]:
        c.step(ids, y)
    assert torch.equal(a.idmap.counters, c.idmap.counters)
    assert torch.equal(a.flat, c.flat)
    ka, kc = a.idmap.key_of_row.cpu().numpy(), c.idmap.key_of_row.cpu().numpy()
    for f in range(F):
        lo, hi = int(a.base_host[f]), int(a.base_host[f] + 300)
        assert set(ka[lo:hi].tolist()) == set(kc[lo:hi].tolist()), f
    allk = torch.from_numpy(pool.T.copy()).to(cuda_dev)
    ra = a.idmap.resolve(allk, a.idmap.fields(range(F)), insert=False)
    rc = c.idmap.resolve(allk, c.idmap.fields(range(F)), insert=False)
    assert torch.equal(ra >= 0, rc >= 0)
    ok = ra >= 0
    assert torch.equal(a.arena[ra[ok]], c.arena[rc[ok]]), "per-key [w|m|v] after train(2)+save+load+train(2)"
    with pytest.raises(ValueError):
        ck.load_checkpoint(AutoIntTrainer(cfg("mod"), cuda_dev), tmp_path)
    ck.save_checkpoint(AutoIntTrainer(cfg("mod"), cuda_dev), tmp_path / "mod")
    with pytest.raises(ValueError):
        ck.load_checkpoint(AutoIntTrainer(cfg(), cuda_dev), tmp_path / "mod")


# ----------------------------------------------------------------------------------------------- 9. GraphedTrainStep
@pytest.mark.gpu
def test_graphed_train_step_autoint_hash(cuda_dev):
    from recommendsystem_b200.api.builders import AUTOINT, AUTOINT_LABELS
    from recommendsystem_b200.api.graph import GraphedTrainStep
    B = 96
    slots = [str(3000 + i) for i in range(8)]
    g = torch.Generator().manual_seed(8)
    pools = torch.randint(0, 2 ** 62, (len(slots), 150), generator=g)
    batches = []
    for _ in range(4):
        inp = {s: pools[i][torch.randint(0, 150, (B,), generator=g)].to(cuda_dev) for i, s in enumerate(slots)}
        lab = {k: (torch.rand(B, 1, generator=g) < 0.3).float().to(cuda_dev) for k in AUTOINT_LABELS}
        batches.append((inp, lab))

    def build():
        torch.manual_seed(11)
        ret = AUTOINT(slots, [], False, dnn_hidden_units=(32, 16), bucket_size=400, device=str(cuda_dev), seed=3,
                      id_map="hash")
        ret.model.predict(batches[0][0])
        return ret.model

    a, b = build(), build()
    eager = [float(a.train_step(*bt)[0]) for bt in batches]
    gs = GraphedTrainStep(b, *batches[0], warmup=3)
    graphed = [float(gs(*bt)[0]) for bt in batches]
    assert graphed == eager
    for x, y in zip(a.sub_model.parameters(), b.sub_model.parameters()):
        assert torch.equal(x, y)
    assert torch.equal(a.emb.idmap.counters, b.emb.idmap.counters)
    for i, s in enumerate(slots):
        t = pools[i].reshape(-1, 1).to(cuda_dev)
        ra = a.emb.idmap.resolve(t, a.emb.idmap.fields([i]), insert=False).reshape(-1)
        rb = b.emb.idmap.resolve(t, b.emb.idmap.fields([i]), insert=False).reshape(-1)
        assert torch.equal(ra >= 0, rb >= 0)
        assert torch.equal(a.emb.arena[ra[ra >= 0]], b.emb.arena[rb[rb >= 0]]), s


# ------------------------------------------------------------------------------------------ 10. sharded (CPU tests)
def test_sharded_classes_reject_hash():
    from recommendsystem_b200.api.embedding import Adam, category_column, embedding_column
    from recommendsystem_b200.api.sharded_embedding import ShardedEmbeddingFeatures
    from recommendsystem_b200.autoint import AutoIntConfig
    from recommendsystem_b200.sharded import ShardedAutoIntTrainer
    with pytest.raises(NotImplementedError):
        ShardedAutoIntTrainer(AutoIntConfig(id_map="hash"), "cuda:0")
    with pytest.raises(NotImplementedError):
        ShardedEmbeddingFeatures([embedding_column(category_column("a", 10), 8)], Adam(), id_map="hash")


def test_id_map_option_and_slot_sizing():
    from recommendsystem_b200.api.embedding import Adam, EmbeddingFeatures, category_column, embedding_column
    from recommendsystem_b200.idmap import slots_per_field
    assert slots_per_field([1, 2, 3, 64, 1000, 1_000_000]).tolist() == [2, 4, 8, 128, 2048, 2 ** 21]
    with pytest.raises(ValueError):
        EmbeddingFeatures([embedding_column(category_column("a", 10), 8)], Adam(), device="cpu", id_map="sign")
