"""Eviction from the collision-free id map: per-row show counts, show decay and `feature_drop_show`
(IdMap.count / IdMap.evict, rs_idmap_count / rs_idmap_evict in include/rs_b200.h).

Method of the parity tests (as tests/test_gpu_idmap.py): hash mode runs against mod mode on the same batches, the mod
side seeing ids remapped on the host to dense indices per field.  Here the host restatement also keeps its own show
counts, evicts the same keys, frees their dense index, and writes the init-rule record into a reused mod row before
the key's next step.  Outputs, losses, dense parameters, every live key's record and the evicted sets must agree bit
for bit.  Live keys stay within capacity: which new keys win a full field depends on the order of the atomics."""
import heapq

import numpy as np
import pytest
import torch

from test_gpu_idmap import _map, _opt, init_rule


# ---------------------------------------------------------------------------------------------- host restatement
class _Host:
    """Dense index and show count of every live key of every field; freed indices are reused, smallest first."""

    def __init__(self, n_fields, cap):
        self.idx = [dict() for _ in range(n_fields)]
        self.show = [dict() for _ in range(n_fields)]
        self.free = [list(range(cap)) for _ in range(n_fields)]

    def remap(self, f, ids):
        """Training lookup of `ids` (any shape, < 0 = padding) in field f: dense indices, and the keys that are new."""
        out = np.full(ids.shape, -1, np.int64)
        new = []
        for pos, k in np.ndenumerate(ids):
            k = int(k)
            if k < 0:
                continue
            if k not in self.idx[f]:
                self.idx[f][k] = heapq.heappop(self.free[f])
                self.show[f][k] = np.float32(0)
                new.append(k)
            self.show[f][k] = np.float32(self.show[f][k] + np.float32(1))
            out[pos] = self.idx[f][k]
        return out, new

    def evict(self, threshold, decay):
        dropped = []
        for f in range(len(self.idx)):
            gone = set()
            for k in list(self.idx[f]):
                s = np.float32(self.show[f][k]) * np.float32(decay)
                if s < np.float32(threshold):
                    heapq.heappush(self.free[f], self.idx[f].pop(k))
                    del self.show[f][k]
                    gone.add(k)
                else:
                    self.show[f][k] = s
            dropped.append(gone)
        return dropped

    def keys(self, f):
        return sorted(self.idx[f], key=self.idx[f].get)


def _rows_of(m, f, keys, dev):
    t = torch.tensor(list(keys), dtype=torch.int64, device=dev).reshape(-1, 1)
    return m.resolve(t, m.fields([f]), insert=False).reshape(-1)


def _check_show_and_drops(m, host, before, dropped, dev):
    """The map dropped exactly the host's keys, and every live key has the host's show."""
    for f in range(len(host.idx)):
        if before[f]:
            gone = {k for k, r in zip(before[f], _rows_of(m, f, before[f], dev).tolist()) if r < 0}
            assert gone == dropped[f], f
        ks = host.keys(f)
        if ks:
            r = _rows_of(m, f, ks, dev)
            assert (r >= 0).all()
            want = torch.tensor([host.show[f][k] for k in ks], dtype=torch.float32, device=dev)
            assert torch.equal(m.show[r], want), f
    assert m.stats()["rows_used"] == [len(x) for x in host.idx]


# -------------------------------------------------------------------------------------------- 1. kernels vs numpy
@pytest.mark.gpu
def test_count_and_evict_kernels(cuda_dev):
    dev = cuda_dev
    rows, d, seed, scale = [300, 200, 257], 4, 5, 0.1
    m, arena = _map(rows, dev, d=d, seed=seed, scale=scale)
    F = len(rows)
    fields = m.fields(range(F))
    g = np.random.default_rng(11)
    pools = [g.choice(2 ** 62, 180, replace=False).astype(np.int64) for _ in range(F)]
    zipf = 1.0 / np.arange(1, 181) ** 1.1
    zipf /= zipf.sum()
    occ = [dict() for _ in range(F)]
    for _ in range(6):                                            # duplicates, padding and Zipf-skewed repeats
        ids = np.stack([g.choice(pools[f], 512, p=zipf) for f in range(F)], 1)
        ids[g.random(ids.shape) < 0.1] = -1
        r = m.resolve(torch.from_numpy(ids).to(dev), fields, insert=True)
        m.count(r)
        for f in range(F):
            for k in ids[:, f][ids[:, f] >= 0].tolist():
                occ[f][k] = occ[f].get(k, 0) + 1
    show0 = m.show.clone()
    unseen = torch.from_numpy(g.integers(2 ** 62, 2 ** 63 - 1, (64, F))).to(dev)
    m.resolve(torch.from_numpy(np.stack([pools[f][:64] for f in range(F)], 1)).to(dev), fields, insert=False)
    m.resolve(unseen, fields, insert=False)
    assert torch.equal(m.show, show0), "inference lookups count nothing"
    used = m.stats()["rows_used"]
    kor0 = m.key_of_row.cpu().numpy()
    show_h = show0.cpu().numpy()
    rec0 = arena.clone()
    for f in range(F):
        b = int(m.base[f])
        assert {int(k): float(s) for k, s in zip(kor0[b:b + used[f]], show_h[b:b + used[f]])} == \
            {k: float(c) for k, c in occ[f].items()}, f
        assert (show_h[b + used[f]:b + rows[f]] == 0).all()

    decay, thr = 0.7, 2.5
    m.evict(thr, decay)
    kor, show = m.key_of_row.cpu().numpy(), m.show.cpu().numpy()
    st = m.stats()
    for f in range(F):
        b, u, R = int(m.base[f]), used[f], rows[f]
        dec = show_h[b:b + u] * np.float32(decay)                  # host fp32 decay
        keep = ~(dec < np.float32(thr))
        live = int(keep.sum())
        assert st["rows_used"][f] == live and st["evicted"][f] == u - live
        # the k-th dropped row below live receives the k-th kept row at or above it (ascending)
        order = np.arange(u)
        holes, movers = order[:live][~keep[:live]], order[live:][keep[live:]]
        src = order[:live].copy()
        src[holes] = movers
        assert np.array_equal(kor[b:b + live], kor0[b:b + u][src]), f
        assert len(set(kor[b:b + live].tolist())) == live and (kor[b + live:b + R] == -1).all()
        assert np.array_equal(show[b:b + live], dec[src]), "decayed fp32 show moved with its key"
        assert (show[b + live:b + R] == 0).all(), "vacated rows have show 0"
        assert torch.equal(arena[b:b + live], rec0[b + torch.from_numpy(src).to(dev)]), "records moved bit for bit"
        surv = kor0[b:b + u][keep]
        r = _rows_of(m, f, surv.tolist(), dev).cpu().numpy()
        assert (r >= 0).all() and (kor[r] == surv).all(), "each surviving key finds its own row"
        gone = kor0[b:b + u][~keep]
        assert len(gone) and (_rows_of(m, f, gone.tolist(), dev) == -1).all(), "evicted ids look up as -1"
        if f == 0:
            gone0 = gone[:20]
    # re-admission: a fresh record from the init rule, show 0
    arena[:, 1:, :] = 7.0                                        # stale moments everywhere
    f = 0
    t = torch.from_numpy(gone0).reshape(-1, 1).to(dev)
    r = m.resolve(t, m.fields([f]), insert=True).reshape(-1)
    assert (r >= 0).all() and (m.show[r] == 0).all()
    for k, x in zip(gone0.tolist(), r.tolist()):
        np.testing.assert_allclose(arena[x, 0].cpu().numpy(), init_rule(seed, f, k, d, scale), rtol=2e-6, atol=1e-10)
        assert (arena[x, 1:] == 0).all()
    m2, arena2 = _map(rows, dev, d=d, seed=seed, scale=scale)
    r2 = m2.resolve(t, m2.fields([f]), insert=True).reshape(-1)
    assert torch.equal(arena[r, 0], arena2[r2, 0]), "the same record as a first insert, bit for bit"


@pytest.mark.gpu
@pytest.mark.parametrize("opt", ["adagrad_row", "adagrad_elem"])
def test_evict_moves_adagrad_state(cuda_dev, opt):
    """AdaGrad arenas: w [R, d] and g2sum [R] or [R, d] move with their keys."""
    from recommendsystem_b200.idmap import IdMap
    dev, d, rows = cuda_dev, 8, [128, 96]
    w = torch.zeros(sum(rows), d, device=dev)
    g2 = torch.zeros((sum(rows), d) if opt == "adagrad_elem" else (sum(rows),), device=dev)
    m = IdMap(rows, dev, 3, 0.1, w, [(g2, 0.1)])
    g = np.random.default_rng(12)
    ids = torch.from_numpy(np.stack([g.choice(2 ** 40, 90, replace=False) for _ in rows], 1)).to(dev)
    r = m.resolve(ids, m.fields([0, 1]), insert=True)
    m.count(r)
    m.count(r[::2].contiguous())                                 # even positions: show 2
    w.copy_(torch.randn_like(w))
    g2.copy_(torch.rand_like(g2))
    before = {}
    for f in range(2):
        rf = r[:, f]
        before[f] = (w[rf].clone(), g2[rf].clone())
    m.evict(1.5)
    for f in range(2):
        rf = m.resolve(ids, m.fields([0, 1]), insert=False)[:, f]
        keep = torch.zeros(90, dtype=torch.bool, device=dev)
        keep[::2] = True
        assert torch.equal(rf >= 0, keep)
        assert torch.equal(w[rf[keep]], before[f][0][keep]) and torch.equal(g2[rf[keep]], before[f][1][keep])
    assert m.stats()["evicted"] == [45, 45] and m.stats()["rows_used"] == [45, 45]


# ------------------------------------------------------------------------------- 2. parity with mod mode (layers)
def _init_records(layer, f, keys):
    """The records the hash map's insert gives `keys` of column f: (w [n, d], [state [n] / [n, k], ...])."""
    from recommendsystem_b200.api.embedding import Adam
    from recommendsystem_b200.idmap import IdMap
    dev, d, total = layer.dev, layer.d, int(layer.rows.sum())
    if isinstance(layer.opt, Adam):
        rec = torch.zeros(total, 3, d, device=dev)
        w, states = rec[:, 0, :], [(rec[:, 1, :], 0.0), (rec[:, 2, :], 0.0)]
    else:
        w = torch.zeros(total, d, device=dev)
        states = [(torch.zeros_like(layer.g2sum), float(layer.opt.initial_g2sum))]
    scratch = IdMap(layer.rows, dev, layer.idmap.seed, layer.idmap.scale, w, states)
    r = _rows_of_insert(scratch, f, keys, dev)
    return w[r], [s[r] for s, _ in states]


def _rows_of_insert(m, f, keys, dev):
    t = torch.tensor(list(keys), dtype=torch.int64, device=dev).reshape(-1, 1)
    return m.resolve(t, m.fields([f]), insert=True).reshape(-1)


def _seed_new(h, md, f, host, new):
    if not new:
        return
    from recommendsystem_b200.api.embedding import Adam
    w, states = _init_records(h, f, new)
    dst = int(md.base[f]) + torch.tensor([host.idx[f][k] for k in new], device=h.dev)
    md.table[dst] = w
    if isinstance(h.opt, Adam):
        md.m[dst], md.v[dst] = states
    else:
        md.g2sum[dst] = states[0]


def _layer_records(layer, rows):
    from recommendsystem_b200.api.embedding import Adam
    if isinstance(layer.opt, Adam):
        return layer.arena[rows].reshape(len(rows), -1)
    return torch.cat([layer.table[rows], layer.g2sum[rows].reshape(len(rows), -1)], 1)


@pytest.mark.gpu
@pytest.mark.parametrize("opt", ["adam", "adagrad_row", "adagrad_elem"])
def test_embedding_features_evict_matches_mod(cuda_dev, opt):
    from recommendsystem_b200.api.embedding import EmbeddingFeatures, category_column, embedding_column
    dev = cuda_dev
    d, B, T, bag, cap = 8, 64, 4, 3, 200
    cols = ["a", "b", "s", "bag", "csr"]

    def layer(mode):
        ec = [embedding_column(category_column("a", cap), d), embedding_column(category_column("b", cap), d),
              embedding_column(category_column("s", cap), d, combiner=None, seq_max_len=T),
              embedding_column(category_column("bag", cap), d), embedding_column(category_column("csr", cap), d)]
        return EmbeddingFeatures(ec, _opt(opt), device=str(dev), seed=42, id_map=mode)

    g = np.random.default_rng(13)
    pools = {c: g.choice(2 ** 62, 180, replace=False).astype(np.int64) for c in cols}
    p = 1.0 / np.arange(1, 181) ** 1.2
    p /= p.sum()
    h, md = layer("hash"), layer("mod")
    host = _Host(len(cols), cap)
    steps, every, thr, decay = 8, 2, 1.5, 0.5
    n_dropped = 0
    for st in range(steps):
        bt = {"a": g.choice(pools["a"], B, p=p), "b": g.choice(pools["b"], B, p=p)}
        s = g.choice(pools["s"], (B, T), p=p)
        s[g.random((B, T)) < 0.3] = -1
        bt["s"] = s
        bg = g.choice(pools["bag"], (B, bag), p=p)
        bg[g.random((B, bag)) < 0.2] = -1
        bt["bag"] = bg
        offs = np.concatenate([[0], np.cumsum(g.integers(0, 4, B))]).astype(np.int64)
        bt["csr"] = (g.choice(pools["csr"], int(offs[-1]), p=p).astype(np.int64), offs)
        rem = {}
        for ci, c in enumerate(cols):
            vals = bt[c][0] if c == "csr" else bt[c]
            mapped, new = host.remap(ci, vals)
            _seed_new(h, md, ci, host, new)
            rem[c] = (mapped, offs) if c == "csr" else mapped
        todev = lambda b: {c: (tuple(torch.from_numpy(x).to(dev) for x in v) if isinstance(v, tuple)
                               else torch.from_numpy(v).to(dev)) for c, v in b.items()}
        oh, om = h(todev(bt)), md(todev(rem))
        for c in cols:
            if c == "s":
                assert torch.equal(oh[c][0], om[c][0]) and torch.equal(oh[c][1], om[c][1]), (st, c)
            else:
                assert torch.equal(oh[c], om[c]), (st, c)
        gr = {c: torch.from_numpy(g.standard_normal((B, d)).astype(np.float32)).to(dev) for c in ("a", "b", "bag", "csr")}
        gr["s"] = torch.from_numpy(g.standard_normal((B, T, d)).astype(np.float32)).to(dev)
        h.backward(gr)
        md.backward(gr)
        if st % every == every - 1:
            before = [host.keys(ci) for ci in range(len(cols))]
            dropped = host.evict(thr, decay)
            n_dropped += sum(len(x) for x in dropped)
            h.evict(thr, decay)
            _check_show_and_drops(h.idmap, host, before, dropped, dev)
    assert n_dropped > 0
    assert sum(h.idmap.stats()["evicted"]) == n_dropped
    for ci, c in enumerate(cols):
        ks = host.keys(ci)
        rh = _rows_of(h.idmap, ci, ks, dev)
        rm = int(md.base[ci]) + torch.tensor([host.idx[ci][k] for k in ks], device=dev)
        assert torch.equal(_layer_records(h, rh), _layer_records(md, rm)), c


# ------------------------------------------------------------------------------- 2b. parity with mod mode (AutoInt)
def _autoint_cfg(mode, dtype, fuse, F, B, cap, seed):
    from recommendsystem_b200.autoint import AutoIntConfig
    return AutoIntConfig(num_fields=F, rows_per_field=cap, batch=B, mlp_hidden=(128, 64), dtype=dtype, lr_dense=1e-3,
                         lr_sparse=1e-2, seed=seed, fuse_embedding=fuse, id_map=mode)


def _trainer_state(tr):
    m = tr.idmap
    return [m.counters.clone(), m.key_of_row.clone(), m.show.clone(), m.evicted.clone(), tr.arena.clone()]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,fuse,capture", [("bf16", True, True), ("f32", False, False)])
def test_autoint_evict_matches_mod(cuda_dev, dtype, fuse, capture):
    from recommendsystem_b200.autoint import AutoIntTrainer
    from recommendsystem_b200.idmap import IdMap
    dev = cuda_dev
    F, B, cap, seed = 39, 256, 300, 9
    h = AutoIntTrainer(_autoint_cfg("hash", dtype, fuse, F, B, cap, seed), dev)
    md = AutoIntTrainer(_autoint_cfg("mod", dtype, fuse, F, B, cap, seed), dev,
                        tables=torch.zeros(F * cap, 16, device=dev))
    assert h.fused == md.fused == (dtype == "bf16" and fuse)
    g = np.random.default_rng(14)
    pools = np.stack([g.choice(2 ** 62, 250, replace=False) for _ in range(F)]).astype(np.int64)
    p = 1.0 / np.arange(1, 251) ** 1.1
    p /= p.sum()
    host = _Host(F, cap)

    def prepare(ids):
        """host remap of a batch; the mod rows of its new keys get the init-rule records."""
        rem = np.full_like(ids, -1)
        for f in range(F):
            rem[:, f], new = host.remap(f, ids[:, f])
            if new:
                sw = torch.zeros(h.total_rows, 16, device=dev)
                r = _rows_of_insert(IdMap(h.rows_host, dev, h.cfg.seed, h.cfg.table_init_scale, sw), f, new, dev)
                dst = int(md.base_host[f]) + torch.tensor([host.idx[f][k] for k in new], device=dev)
                md.table[dst] = sw[r]
                md.table_m[dst] = 0.0
                md.table_v[dst] = 0.0
        return rem

    def evict(thr, decay):
        before = [host.keys(f) for f in range(F)]
        dropped = host.evict(thr, decay)
        h.evict(thr, decay)
        _check_show_and_drops(h.idmap, host, before, dropped, dev)
        return sum(len(x) for x in dropped)

    batches = []
    for _ in range(8):
        ids = np.stack([g.choice(pools[f], B, p=p) for f in range(F)], 1)
        ids[g.random((B, F)) < 0.05] = -1
        batches.append((ids, (g.random((B, 1)) < 0.3).astype(np.float32)))
    lh, lm, n_dropped = [], [], 0
    for st, (ids, y) in enumerate(batches):
        rem = prepare(ids)
        yt = torch.from_numpy(y).to(dev)
        if st == 2 and capture:
            # capture after an eviction, with this step's ids (new and re-admitted keys) in the static buffers:
            # the undone warm-up step leaves map, shows and records as they were
            h.ids.copy_(torch.from_numpy(ids).to(dev))
            md.ids.copy_(torch.from_numpy(rem).to(dev))
            torch.cuda.synchronize()
            before = _trainer_state(h)
            h.capture()
            md.capture()
            assert all(torch.equal(a, b) for a, b in zip(before, _trainer_state(h)))
        lh.append(float(h.step(torch.from_numpy(ids).to(dev), yt)))
        lm.append(float(md.step(torch.from_numpy(rem).to(dev), yt)))
        if st % 2 == 1:
            n_dropped += evict(25.0, 0.5)
    assert n_dropped > 0
    assert lh == lm
    assert torch.equal(h.flat, md.flat) and torch.equal(h.flat_m, md.flat_m) and torch.equal(h.flat_v, md.flat_v)
    for f in range(F):
        ks = host.keys(f)
        rh = _rows_of(h.idmap, f, ks, dev)
        rm = int(md.base_host[f]) + torch.tensor([host.idx[f][k] for k in ks], device=dev)
        assert torch.equal(h.arena[rh], md.arena[rm]), f


# ----------------------------------------------------------------------------------------------- 3. capacity reuse
@pytest.mark.gpu
def test_evicted_rows_are_reused(cuda_dev):
    dev = cuda_dev
    m, _ = _map([64, 32], dev)
    g = np.random.default_rng(15)
    keys = g.choice(2 ** 40, 300, replace=False).astype(np.int64)
    t = torch.from_numpy(keys[:100]).reshape(-1, 1).to(dev)
    m.count(m.resolve(t, m.fields([0]), insert=True))
    assert m.stats()["rows_used"] == [64, 0] and m.stats()["overflow"] == [36, 0]
    k = 10
    live = m.key_of_row[:64].clone()
    m.count(m.resolve(live[k:].reshape(-1, 1).contiguous(), m.fields([0]), insert=True))     # show 2, the rest 1
    m.evict(1.5)
    assert m.stats()["rows_used"] == [64 - k, 0] and m.stats()["evicted"] == [k, 0]
    fresh = torch.from_numpy(keys[200:200 + k]).reshape(-1, 1).to(dev)
    r = m.resolve(fresh, m.fields([0]), insert=True)
    assert (r >= 0).all() and len(set(r.reshape(-1).tolist())) == k
    assert m.stats()["rows_used"] == [64, 0] and m.stats()["overflow"] == [36, 0]
    assert (_rows_of(m, 0, live[:k].tolist(), dev) == -1).all()


# -------------------------------------------------------------------------------------------- 4. undo and resume
@pytest.mark.gpu
def test_graphed_train_step_after_evict(cuda_dev):
    from recommendsystem_b200.api.builders import AUTOINT, AUTOINT_LABELS
    from recommendsystem_b200.api.graph import GraphedTrainStep
    dev = cuda_dev
    B = 96
    slots = [str(3000 + i) for i in range(8)]
    g = torch.Generator().manual_seed(16)
    pools = torch.randint(0, 2 ** 62, (len(slots), 150), generator=g)
    batches = []
    for _ in range(6):
        inp = {s: pools[i][torch.randint(0, 150, (B,), generator=g)].to(dev) for i, s in enumerate(slots)}
        lab = {k: (torch.rand(B, 1, generator=g) < 0.3).float().to(dev) for k in AUTOINT_LABELS}
        batches.append((inp, lab))

    def build():
        torch.manual_seed(11)
        ret = AUTOINT(slots, [], False, dnn_hidden_units=(32, 16), bucket_size=400, device=str(dev), seed=3,
                      id_map="hash")
        ret.model.predict(batches[0][0])
        return ret.model

    a, b = build(), build()
    for net in (a, b):
        for bt in batches[:2]:
            net.train_step(*bt)
        with pytest.raises(ValueError):
            net.emb.evict()                                      # Adam: the threshold must be given
        net.emb.evict(1.5, 0.9)
    assert a.emb.idmap.stats()["evicted"] == b.emb.idmap.stats()["evicted"] and sum(a.emb.idmap.stats()["evicted"])
    m = b.emb.idmap
    before = [m.counters.clone(), m.key_of_row.clone(), m.show.clone(), b.emb.arena.clone()]
    gs = GraphedTrainStep(b, *batches[2], warmup=3)
    assert all(torch.equal(x, y) for x, y in zip(before, [m.counters, m.key_of_row, m.show, b.emb.arena]))
    eager, graphed = [], []
    for i, bt in enumerate(batches[2:]):
        eager.append(float(a.train_step(*bt)[0]))
        graphed.append(float(gs(*bt)[0]))
        if i == 1:
            a.emb.evict(2.5, 0.5)
            b.emb.evict(2.5, 0.5)
    assert graphed == eager
    for x, y in zip(a.sub_model.parameters(), b.sub_model.parameters()):
        assert torch.equal(x, y)
    assert torch.equal(a.emb.idmap.counters, b.emb.idmap.counters)
    assert torch.equal(a.emb.idmap.evicted, b.emb.idmap.evicted)
    for i in range(len(slots)):
        ra = _rows_of(a.emb.idmap, i, pools[i].tolist(), dev)
        rb = _rows_of(b.emb.idmap, i, pools[i].tolist(), dev)
        assert torch.equal(ra >= 0, rb >= 0)
        assert torch.equal(a.emb.arena[ra[ra >= 0]], b.emb.arena[rb[rb >= 0]])
        assert torch.equal(a.emb.idmap.show[ra[ra >= 0]], b.emb.idmap.show[rb[rb >= 0]])


@pytest.mark.gpu
@pytest.mark.parametrize("capture", [False, True])
def test_evict_checkpoint_resume_is_exact(cuda_dev, tmp_path, capture):
    from recommendsystem_b200 import checkpoint as ck
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    dev = cuda_dev
    B, F, cap = 128, 39, 300
    cfg = lambda: AutoIntConfig(num_fields=F, rows_per_field=cap, batch=B, mlp_hidden=(32, 16), lr_dense=1e-3,
                                lr_sparse=1e-2, id_map="hash", seed=5)
    g = np.random.default_rng(17)
    pool = g.integers(0, 2 ** 63 - 1, (F, 280))
    data = [(torch.from_numpy(np.stack([g.choice(pool[f], B) for f in range(F)], 1)).to(dev),
             torch.from_numpy((g.random((B, 1)) < 0.3).astype(np.float32)).to(dev)) for _ in range(6)]

    def run(tr, part):
        for i in part:
            tr.step(*data[i])
            if i in (1, 3):
                tr.evict(1.5, 0.75)

    a = AutoIntTrainer(cfg(), dev)
    run(a, range(6))
    b = AutoIntTrainer(cfg(), dev)
    run(b, range(3))
    ck.save_checkpoint(b, tmp_path, step=3)
    c = AutoIntTrainer(cfg(), dev)
    ck.load_checkpoint(c, tmp_path)
    for x, y in zip(_trainer_state(b), _trainer_state(c)):
        assert torch.equal(x, y)
    if capture:
        c.ids.copy_(data[3][0])
        c.capture()
    run(c, range(3, 6))
    assert sum(a.idmap.stats()["evicted"]) > 0
    assert torch.equal(a.idmap.counters, c.idmap.counters) and torch.equal(a.idmap.evicted, c.idmap.evicted)
    assert torch.equal(a.flat, c.flat)
    allk = torch.from_numpy(pool.T.copy()).to(dev)
    ra = a.idmap.resolve(allk, a.idmap.fields(range(F)), insert=False)
    rc = c.idmap.resolve(allk, c.idmap.fields(range(F)), insert=False)
    assert torch.equal(ra >= 0, rc >= 0)
    ok = ra >= 0
    assert torch.equal(a.arena[ra[ok]], c.arena[rc[ok]]), "per-key [w|m|v]"
    assert torch.equal(a.idmap.show[ra[ok]], c.idmap.show[rc[ok]]), "per-key show"
    # a map saved before eviction existed (no show / evicted) still loads: zero shows, nothing evicted
    with np.load(tmp_path / "idmap.npz") as z:
        old = {k: z[k] for k in z.files if k not in ("show", "evicted")}
    np.savez(tmp_path / "idmap.npz", **old)
    e = AutoIntTrainer(cfg(), dev)
    ck.load_checkpoint(e, tmp_path)
    assert torch.equal(e.idmap.key_of_row, b.idmap.key_of_row) and torch.equal(e.idmap.counters, b.idmap.counters)
    assert (e.idmap.show == 0).all() and (e.idmap.evicted == 0).all()
    assert torch.equal(e.arena, b.arena)


@pytest.mark.gpu
def test_evict_argument_and_state_errors(cuda_dev):
    from recommendsystem_b200.api.embedding import EmbeddingFeatures, category_column, embedding_column
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    dev = cuda_dev
    tr = AutoIntTrainer(AutoIntConfig(num_fields=4, rows_per_field=50, batch=16, mlp_hidden=(32, 16)), dev)
    with pytest.raises(ValueError):
        tr.evict(1.0)                                            # mod mode
    e = EmbeddingFeatures([embedding_column(category_column("a", 50), 8)], _opt("adagrad_row"), device=str(dev),
                          id_map="hash")
    ids = {"a": torch.arange(20, device=dev)}
    e(ids)
    with pytest.raises(RuntimeError):
        e.evict(1.0)                                             # a training forward waits for its backward
    e.backward({"a": torch.ones(20, 8, device=dev)})
    with pytest.raises(ValueError):
        e.evict(1.0, decay=0.0)
    e.evict()                                                    # feature_drop_show = -1: drops nothing
    assert e.idmap.stats()["rows_used"] == [20] and e.idmap.stats()["evicted"] == [0]
    with torch.no_grad():
        e(ids)
    e.evict(1.5)                                                 # an inference call leaves nothing pending
    assert e.idmap.stats()["rows_used"] == [0] and e.idmap.stats()["evicted"] == [20]
    with torch.no_grad():
        assert (e(ids)["a"] == 0).all(), "evicted ids read zeros"


# ------------------------------------------------------------------------------------------------- 5. CPU tests
def test_evict_arguments_are_checked():
    from recommendsystem_b200.idmap import check_evict_args
    assert check_evict_args(3, 0.5) == (3.0, 0.5)
    assert check_evict_args(-1, 1.0) == (-1.0, 1.0)
    for thr, decay in ((1.0, 0.0), (1.0, -0.5), (1.0, 1.5), (1.0, float("nan")), (float("inf"), 1.0),
                       (float("nan"), 0.5), (1e39, 0.5)):
        with pytest.raises(ValueError):
            check_evict_args(thr, decay)


def test_feature_drop_show_is_the_default_threshold():
    from recommendsystem_b200.api.embedding import AdaGrad, Adam, EmbeddingFeatures, category_column, embedding_column
    assert AdaGrad().feature_drop_show == -1 and AdaGrad(feature_drop_show=3).feature_drop_show == 3

    class Recorder:
        def __init__(self):
            self.calls = []

        def evict(self, threshold, decay):
            self.calls.append((threshold, decay))

    col = [embedding_column(category_column("a", 10), 8)]
    e = EmbeddingFeatures(col, AdaGrad(feature_drop_show=4, initial_g2sum=0.1), device="cpu")
    with pytest.raises(ValueError, match="id_map='hash'"):
        e.evict()                                                # mod mode
    e.idmap = Recorder()
    e.evict()
    e.evict(2.0, 0.5)
    assert e.idmap.calls == [(4.0, 1.0), (2.0, 0.5)]
    with pytest.raises(ValueError, match="decay"):
        e.evict(decay=2.0)
    a = EmbeddingFeatures(col, Adam(), device="cpu")
    a.idmap = Recorder()
    with pytest.raises(ValueError, match="threshold"):
        a.evict()
    a.evict(1.0)
    assert a.idmap.calls == [(1.0, 1.0)]
