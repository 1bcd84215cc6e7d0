"""Evaluation in the AutoInt trainer: rs_tower_fwd bit for bit against the p_out of rs_tower_step, the eval step's p
against the p_raw of a train step from the same state in every mode, evaluate() against BinaryMetrics, and the
guarantee that evaluation changes no trainer state (hash mode: inserts and counts no id)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32).cpu().numpy()


# ---------------------------------------------------------------------------------------------- 1. the kernel
@pytest.mark.parametrize("F", [39, 13])
@pytest.mark.parametrize("B", [1, 127, 128, 8192, 8193])
def test_tower_fwd_bit_exact_with_tower_step(cuda_dev, B, F):
    from recommendsystem_b200 import ops
    g = torch.Generator(device=cuda_dev).manual_seed(B * 100 + F)
    K0, N0, N1, Ki = F * 16, 256, 128, F * 16
    assert ops.tower_supported(K0, N0, N1, Ki)
    r = lambda *s, sc=1.0: (torch.randn(*s, device=cuda_dev, generator=g) * sc)
    bf = lambda t: t.to(torch.bfloat16).contiguous()
    X = bf(r(B, K0))
    W0, W1 = bf(r(K0, N0, sc=K0 ** -0.5)), bf(r(N0, N1, sc=N0 ** -0.5))
    W0T, W1T = W0.t().contiguous(), W1.t().contiguous()
    b0, b1 = r(N0, sc=0.1), r(N1, sc=0.1)
    w, ob = r(N1 + Ki, sc=0.2), r(1, sc=0.1)
    y = (torch.rand(B, device=cuda_dev, generator=g) < 0.3).float()
    Z = bf(r(B, N1 + Ki))
    Z0 = Z.clone()
    Z_fwd = Z.clone()                          # the step writes Z[:, :N1]; the forward reads Z[:, N1:] only
    e = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=cuda_dev)
    p_step, p_fwd = e(B, 1), e(B, 1)
    ops.tower_step(X, W0T, W1T, W0, W1, b0, b1, w, ob, y, Z, p_step, e(B, N1 + Ki), e(B, N0), e(B, N0), e(B, K0))
    ops.tower_fwd(X, W0T, W1T, W0, W1, b0, b1, w, ob, Z_fwd, p_fwd)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(_bits(p_fwd), _bits(p_step))
    np.testing.assert_array_equal(_bits(Z_fwd), _bits(Z0))          # the forward writes nothing but p_out
    assert 0.0 < float(p_fwd.float().mean()) < 1.0


# -------------------------------------------------------------------------------------------- trainers
MODES = {
    "bf16_tower": dict(dtype="bf16"),
    "bf16_no_tower": dict(dtype="bf16", fuse_tower=False),
    "bf16_unfused": dict(dtype="bf16", fuse_embedding=False),
    "f32": dict(dtype="f32"),
}


def _bags(bag, F=39):
    return [8 if (bag and f % 3 == 0) else 1 for f in range(F)]


def _trainer(mode="bf16_tower", id_map="mod", bag=False, B=512, F=39, **kw):
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    cfg = AutoIntConfig(num_fields=F, rows_per_field=4000, embed_dim=16, unit_num=16, head_num=2, layer_num=3, batch=B,
                        lr_dense=1e-3, lr_sparse=1e-2, id_map=id_map, bag_size=_bags(bag, F), **MODES[mode], **kw)
    tr = AutoIntTrainer(cfg, "cuda:0")
    want = {"bf16_tower": (True, True), "bf16_no_tower": (True, False), "bf16_unfused": (False, False),
            "f32": (False, False)}[mode]
    assert (tr.fused, tr.fuse_tower) == want
    return tr


def _batch(rng, tr, n=None, hi=3000):
    """(ids [n, S], labels [n, 1]) on the device; bags partly padded."""
    n = tr.cfg.batch if n is None else n
    ids = rng.integers(0, hi, size=(n, tr.S)).astype(np.int64)
    ids[rng.random(ids.shape) < 0.2] = -1
    y = (rng.random((n, 1)) < 0.3).astype(np.float32)
    return torch.from_numpy(ids).cuda(), torch.from_numpy(y).cuda()


# ------------------------------------------------------------------------- 2. eval p == the train step's p
@pytest.mark.parametrize("bag", [False, True])
@pytest.mark.parametrize("id_map", ["mod", "hash"])
@pytest.mark.parametrize("mode", list(MODES))
def test_eval_p_equals_train_p_raw(cuda_dev, mode, id_map, bag):
    tr = _trainer(mode, id_map, bag)
    rng = np.random.default_rng(7)
    for _ in range(2):                         # a state the steps have moved
        tr.step(*_batch(rng, tr))
    ids, y = _batch(rng, tr)
    if id_map == "hash":
        tr.step(ids, y)                        # every id of the batch has its row: the train step inserts none
    tr.evaluate([(ids, y)])
    p_eval = tr.p_raw.clone()
    tr.step(ids, y)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(_bits(p_eval), _bits(tr.p_raw))


# ------------------------------------------------------------------------------- 3. evaluate == BinaryMetrics
@pytest.mark.parametrize("where", ["host", "device"])
@pytest.mark.parametrize("mode", ["bf16_tower", "f32"])
def test_evaluate_matches_binary_metrics(cuda_dev, mode, where):
    from recommendsystem_b200.api.metrics import BinaryMetrics
    tr = _trainer(mode)
    rng = np.random.default_rng(11)
    tr.step(*_batch(rng, tr))
    B = tr.cfg.batch
    stream = [_batch(rng, tr), _batch(rng, tr), _batch(rng, tr, n=B // 2)]
    ref = BinaryMetrics(device=cuda_dev)
    ps, ys = [], []
    for ids, y in stream:                      # every batch's p, from evaluating it alone
        tr.evaluate([(ids, y)])
        n = ids.shape[0]
        ref.update_state(y, tr.p_raw[:n])
        ps.append(tr.p_raw[:n].float().cpu().numpy().reshape(-1))
        ys.append(y.cpu().numpy().reshape(-1))
    if where == "host":
        stream = [(i.cpu().pin_memory(), y.cpu().pin_memory()) for i, y in stream]
    for _ in range(2):                         # the second call replays the captured eval step
        got = tr.evaluate(stream)
        want = ref.result()
        for k in want:
            assert got[k] == want[k], (k, got[k], want[k])
        assert got["count"] == 2.5 * B
        p = np.clip(np.concatenate(ps).astype(np.float64), 1e-6, 1.0)
        yy = np.concatenate(ys).astype(np.float64)
        loss = np.mean(-yy * np.log(p + 1e-6) - (1 - yy) * np.log(1 - p + 1e-6))
        assert abs(got["loss"] - loss) <= 1e-6, (got["loss"], loss)


# ----------------------------------------------------------------------------------------- 4. no state changes
def _state(tr):
    s = {"records": tr.store.records, "flat": tr.flat, "flat_m": tr.flat_m, "flat_v": tr.flat_v,
         "flat_bf16": tr.flat_bf16, "adam_scalars": tr.adam_scalars}
    if tr.bf16:
        s.update({f"WT16 {k}": v for k, v in tr.WT16.items()})
    if tr.idmap is not None:
        s.update({f"idmap {k}": getattr(tr.idmap, k) for k in ("slots", "key_of_row", "counters", "show", "evicted")})
    return {k: v.clone() for k, v in s.items()}


@pytest.mark.parametrize("mode", ["bf16_tower", "bf16_unfused"])
def test_evaluate_changes_no_state(cuda_dev, mode):
    tr = _trainer(mode, "hash", bag=True)
    rng = np.random.default_rng(5)
    tr.step(*_batch(rng, tr))
    before = _state(tr)
    tr.evaluate([_batch(rng, tr, hi=2 ** 40), _batch(rng, tr, n=100, hi=2 ** 40)])
    after = _state(tr)
    for k in before:
        assert torch.equal(before[k], after[k]), k


@pytest.mark.parametrize("graph", [False, True])
def test_evaluate_between_steps_leaves_training_unchanged(cuda_dev, graph):
    rng = np.random.default_rng(9)
    a, b = _trainer(), _trainer()
    batches = [_batch(rng, a) for _ in range(4)]
    held_out = [_batch(rng, a), _batch(rng, a, n=300)]
    if graph:
        a.capture(); b.capture()
    la = [float(a.step(*x)) for x in batches]
    lb = [float(b.step(*x)) for x in batches[:2]]
    b.evaluate(held_out)
    lb += [float(b.step(*x)) for x in batches[2:]]
    torch.cuda.synchronize()
    assert la == lb
    for k, v in _state(a).items():
        assert torch.equal(v, _state(b)[k]), k


@pytest.mark.parametrize("where", ["host", "device"])
def test_evaluate_inside_fit_host_leaves_training_unchanged(cuda_dev, where):
    """evaluate() between two batches of a fit_host loop (batch n+1 already uploaded, loss n not yet handed out)
    trains on the same batches and yields the same losses and tables as fit_host alone."""
    rng = np.random.default_rng(21)
    a, b = _trainer(), _trainer()
    train = [_batch(rng, a) for _ in range(5)]
    held_out = [_batch(rng, a), _batch(rng, a, n=200)]
    if where == "host":
        train = [(i.cpu().pin_memory(), y.cpu().pin_memory()) for i, y in train]
        held_out = [(i.cpu().pin_memory(), y.cpu().pin_memory()) for i, y in held_out]
    a.capture(); b.capture()
    la = list(a.fit_host(train))
    lb, results = [], []
    for i, loss in enumerate(b.fit_host(train)):
        lb.append(loss)
        if i % 2 == 0:
            results.append(b.evaluate(held_out))
    torch.cuda.synchronize()
    assert la == lb
    for k, v in _state(a).items():
        assert torch.equal(v, _state(b)[k]), k
    assert len(results) == 3 and all(r["count"] == a.cfg.batch + 200 for r in results)


# ------------------------------------------------------------------------------------------ 5. hash mode
def test_hash_unseen_ids_read_as_padding(cuda_dev):
    tr = _trainer(id_map="hash")
    rng = np.random.default_rng(13)
    ids, y = _batch(rng, tr)
    tr.step(ids, y)
    used = tr.idmap.stats()["rows_used"]
    fresh = rng.random(ids.shape) < 0.3
    fresh = torch.from_numpy(fresh).cuda()
    unseen = torch.where(fresh, torch.from_numpy(rng.integers(2 ** 41, 2 ** 42, size=ids.shape)).cuda(), ids)
    padded = torch.where(fresh, torch.full_like(ids, -1), ids)
    got = tr.evaluate([(unseen, y)])
    p_unseen = tr.p_raw.clone()
    assert tr.idmap.stats()["rows_used"] == used
    want = tr.evaluate([(padded, y)])
    np.testing.assert_array_equal(_bits(p_unseen), _bits(tr.p_raw))
    assert got == want


# ------------------------------------------------------------------------------------------- 6. refusals
def test_evaluate_refusals(cuda_dev):
    tr = _trainer(B=128)
    rng = np.random.default_rng(1)
    ids, y = _batch(rng, tr)
    bad = [(ids[:, :-1], y), (ids[:0], y[:0]), (torch.cat([ids, ids[:1]]), torch.cat([y, y[:1]])), (ids, y[:-1]),
           (ids[0], y[:1]), (ids, y.reshape(-1)), (ids[:5], y[:5].reshape(-1))]
    for i, l in bad:
        with pytest.raises(ValueError):
            tr.evaluate([(i, l)])
