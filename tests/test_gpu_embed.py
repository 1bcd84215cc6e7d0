"""GPU parity: K1/K2 gather (bit-exact), K3 sorted-segment grad + fused optimizers,
K7 routing (bit-exact) — CUDA path through the C-ABI vs oracle/oracle_np.py."""
import numpy as np
import pytest

from util import REL_F32, assert_close

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _tables(rng, F, d, rmin=50, rmax=4000):
    rows = rng.integers(rmin, rmax, size=F).astype(np.int64)
    base = np.zeros(F, np.int64)
    base[1:] = np.cumsum(rows)[:-1]
    table = (rng.standard_normal((int(rows.sum()), d)) * 0.1).astype(np.float32)
    return rows, base, table


@pytest.mark.parametrize("B,F,d", [(1, 1, 4), (7, 39, 16), (1024, 39, 16), (333, 91, 32), (64, 5, 8),
                                   (257, 3, 64), (100, 2, 128), (50, 39, 12)])
def test_gather_bit_exact(cuda_dev, B, F, d):
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(B * 1000 + F + d)
    rows, base, table = _tables(rng, F, d)
    ids = rng.integers(0, 2 ** 40, size=(B, F)).astype(np.int64)
    ids[rng.random((B, F)) < 0.05] = -1          # padding ids
    ref, ref_rows = onp.embed_gather(table, ids, rows, base)
    out, keys, rws = ops.embed_gather(_t(table, cuda_dev), _t(ids, cuda_dev), _t(base, cuda_dev),
                                      _t(rows, cuda_dev), want_keys=True, want_rows=True)
    assert np.array_equal(out.cpu().numpy(), ref)
    assert np.array_equal(rws.cpu().numpy().astype(np.int64), ref_rows)
    k = keys.cpu().numpy().view(np.uint64).reshape(-1)
    assert np.array_equal((k & 0xFFFFFFFF).astype(np.int64), np.arange(B * F))
    assert np.array_equal((k >> 32).astype(np.uint32), ref_rows.reshape(-1).astype(np.int32).view(np.uint32))
    # bf16 output = round-to-nearest-even of the fp32 row
    outb, _, _ = ops.embed_gather(_t(table, cuda_dev), _t(ids, cuda_dev), _t(base, cuda_dev),
                                  _t(rows, cuda_dev), out_dtype=torch.bfloat16)
    assert torch.equal(outb.cpu(), torch.from_numpy(ref).to(torch.bfloat16))


def test_gather_empty(cuda_dev):
    from recommendsystem_b200 import ops
    table = torch.zeros(10, 16, device=cuda_dev)
    ids = torch.zeros(0, 39, dtype=torch.int64, device=cuda_dev)
    z = torch.zeros(39, dtype=torch.int64, device=cuda_dev)
    out, _, _ = ops.embed_gather(table, ids, z, z + 1)
    assert out.shape == (0, 39, 16)


def test_gather_rows_seq_mask(cuda_dev):
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(5)
    table = rng.standard_normal((500, 32)).astype(np.float32)
    rowidx = rng.integers(0, 500, size=(37, 50)).astype(np.int32)
    lens = rng.integers(0, 51, size=37)
    rowidx[np.arange(50)[None, :] >= lens[:, None]] = -1
    ref, refm = onp.embed_gather_rows(table, rowidx)
    out, mask, _ = ops.embed_gather_rows(_t(table, cuda_dev), _t(rowidx, cuda_dev), want_mask=True)
    assert np.array_equal(out.cpu().numpy(), ref)
    assert np.array_equal(mask.cpu().numpy(), refm)


def test_bag_mean(cuda_dev):
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(6)
    F, d, B = 5, 16, 40
    rows, base, table = _tables(rng, F, d)
    lens = rng.integers(0, 6, size=B * F)
    offsets = np.zeros(B * F + 1, np.int64)
    offsets[1:] = np.cumsum(lens)
    ids = rng.integers(0, 10 ** 9, size=int(offsets[-1])).astype(np.int64)
    ref = onp.embed_bag_mean(table, ids, offsets, rows, base, F)
    out = ops.embed_gather_bag_mean(_t(table, cuda_dev), _t(ids, cuda_dev), _t(offsets, cuda_dev),
                                    _t(base, cuda_dev), _t(rows, cuda_dev), F)
    assert np.array_equal(out.cpu().numpy(), ref)       # same fp32 order => bit-exact


def _sorted_keys(ops, rowidx_t, table_rows):
    n = rowidx_t.numel()
    keys = (rowidx_t.reshape(-1).to(torch.int64) & 0xFFFFFFFF) << 32 | torch.arange(n, device=rowidx_t.device)
    return ops.sort_keys(keys, ops.row_bits(table_rows))


@pytest.mark.parametrize("n,d,R", [(1, 16, 10), (1000, 16, 50), (5000, 16, 100000), (4097, 8, 300),
                                   (3000, 32, 7), (2000, 4, 64), (640, 64, 100)])
def test_segsum_deterministic_and_exact(cuda_dev, n, d, R):
    """Sorted-segment sum: same left-to-right fp32 order as the oracle => bit-exact;
    two runs give identical bits."""
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(n + d)
    rowidx = rng.integers(0, R, size=n).astype(np.int32)
    rowidx[rng.random(n) < 0.03] = -1
    grad = rng.standard_normal((n, d)).astype(np.float32)
    ks = _sorted_keys(ops, _t(rowidx, cuda_dev), R)
    seg_rows, seg_sum = ops.segsum(_t(grad, cuda_dev), ks)
    seg_rows2, seg_sum2 = ops.segsum(_t(grad, cuda_dev), ks)
    heads = seg_rows.cpu().numpy() >= 0
    uniq, sums = onp.segment_sum_sorted(rowidx, grad)
    assert np.array_equal(seg_rows.cpu().numpy()[heads].astype(np.int64), uniq)
    assert np.array_equal(seg_sum.cpu().numpy()[heads], sums)
    assert torch.equal(seg_sum[torch.from_numpy(heads).to(cuda_dev)], seg_sum2[torch.from_numpy(heads).to(cuda_dev)])
    assert torch.equal(seg_rows, seg_rows2)


@pytest.mark.parametrize("n,d,R,gdt", [(5000, 16, 2000, "f32"), (3000, 8, 40, "f32"), (4000, 32, 100000, "f32"),
                                        (5000, 16, 2000, "bf16")])
def test_sparse_adam(cuda_dev, n, d, R, gdt):
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(n + d + R)
    w = (rng.standard_normal((R, d)) * 0.1).astype(np.float32)
    m = (rng.standard_normal((R, d)) * 0.01).astype(np.float32)
    v = (rng.random((R, d)) * 0.01).astype(np.float32)
    lr, b1, b2, eps = 1e-2, 0.9, 0.999, 1e-8
    wt, mt, vt = _t(w, cuda_dev), _t(m, cuda_dev), _t(v, cuda_dev)
    scal = torch.zeros(4, device=cuda_dev)
    for step in range(1, 4):
        rowidx = rng.integers(0, R, size=n).astype(np.int32)
        grad = rng.standard_normal((n, d)).astype(np.float32)
        gt = _t(grad, cuda_dev)
        if gdt == "bf16":
            gt = gt.to(torch.bfloat16)
            grad = gt.float().cpu().numpy()
        ops.adam_advance(scal, b1, b2)
        _, _, corr = onp.adam_scalars(step, b1, b2)
        assert abs(float(scal[3]) - float(corr)) <= 1e-6 * float(corr)
        ks = _sorted_keys(ops, _t(rowidx, cuda_dev), R)
        ops.segsum_adam(wt, mt, vt, gt, ks, lr, b1, b2, eps, scal, grad_scale=0.5)
        w, m, v = onp.sparse_adam(w.astype(np.float64), m.astype(np.float64), v.astype(np.float64), rowidx,
                                  grad.astype(np.float64), lr, b1, b2, eps, float(corr), grad_scale=0.5)
        assert_close(wt.cpu().numpy(), w, REL_F32, "adam w")
        assert_close(mt.cpu().numpy(), m, REL_F32, "adam m")
        assert_close(vt.cpu().numpy(), v, REL_F32, "adam v")
        w, m, v = wt.cpu().numpy(), mt.cpu().numpy(), vt.cpu().numpy()


@pytest.mark.parametrize("per_element", [False, True])
def test_sparse_adagrad(cuda_dev, per_element):
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(11)
    n, d, R = 4000, 32, 900
    w = (rng.standard_normal((R, d)) * 0.1).astype(np.float32)
    g2 = np.full((R, d) if per_element else (R,), 0.1, np.float32)
    rowidx = rng.integers(0, R, size=n).astype(np.int32)
    grad = rng.standard_normal((n, d)).astype(np.float32)
    wt, g2t = _t(w, cuda_dev), _t(g2, cuda_dev)
    ks = _sorted_keys(ops, _t(rowidx, cuda_dev), R)
    ops.segsum_adagrad(wt, g2t, _t(grad, cuda_dev), ks, 0.005, 1e-7, per_element)
    w2, g22 = onp.sparse_adagrad(w.astype(np.float64), g2.astype(np.float64), rowidx, grad.astype(np.float64),
                                 0.005, 1e-7, per_element)
    assert_close(wt.cpu().numpy(), w2, REL_F32, "adagrad w")
    assert_close(g2t.cpu().numpy(), g22, REL_F32, "adagrad g2sum")


@pytest.mark.parametrize("n_b,F,world", [(1, 1, 1), (300, 39, 8), (1024, 39, 2), (77, 5, 4), (513, 91, 8),
                                         (4096, 39, 8), (10, 3, 64)])
def test_route_ids_bit_exact(cuda_dev, n_b, F, world):
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(n_b + F + world)
    rows = rng.integers(10, 100000, size=F).astype(np.int64)
    per = (rows + world - 1) // world
    lbase = np.zeros(F, np.int64)
    lbase[1:] = np.cumsum(per)[:-1]
    ids = rng.integers(0, 2 ** 45, size=(n_b, F)).astype(np.int64)
    ids[rng.random((n_b, F)) < 0.02] = -1
    sr, inv, cnt, off = onp.route_ids(ids, F, rows, lbase, world)
    g_sr, g_inv, g_cnt, g_off = ops.route_ids(_t(ids, cuda_dev), F, _t(rows, cuda_dev), _t(lbase, cuda_dev), world)
    assert np.array_equal(g_cnt.cpu().numpy(), cnt)
    assert np.array_equal(g_off.cpu().numpy(), off)
    assert np.array_equal(g_sr.cpu().numpy(), sr)
    assert np.array_equal(g_inv.cpu().numpy(), inv)
    # permute_rows gather/scatter are inverse permutations
    src = torch.randn(n_b * F, 16, device=cuda_dev)
    fwd = ops.permute_rows(src, g_inv, scatter=True)
    back = ops.permute_rows(fwd, g_inv, scatter=False)
    assert torch.equal(back, src)


def test_dense_adam(cuda_dev):
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(3)
    n = 100003
    w, m, v, g = [rng.standard_normal(n).astype(np.float32) * s for s in (1, 0.01, 0, 1)]
    v = np.abs(rng.standard_normal(n).astype(np.float32)) * 0.01
    wt, mt, vt = _t(w, cuda_dev), _t(m, cuda_dev), _t(v, cuda_dev)
    scal = torch.zeros(4, device=cuda_dev)
    ops.adam_advance(scal, 0.9, 0.999)
    shadow = torch.empty(n, dtype=torch.bfloat16, device=cuda_dev)
    ops.dense_adam(wt, mt, vt, _t(g, cuda_dev), 1e-3, 0.9, 0.999, 1e-8, scal, shadow)
    _, _, corr = onp.adam_scalars(1, 0.9, 0.999)
    w2, m2, v2 = onp.dense_adam(w.astype(np.float64), m.astype(np.float64), v.astype(np.float64),
                                g.astype(np.float64), 1e-3, 0.9, 0.999, 1e-8, float(corr))
    assert_close(wt.cpu().numpy(), w2, REL_F32, "dense adam w")
    assert torch.equal(shadow, wt.to(torch.bfloat16))


@pytest.mark.parametrize("n_b,T,world", [(64, 50, 8), (333, 7, 2), (100, 20, 4)])
def test_route_ids_padded_spread_bit_exact(cuda_dev, n_b, T, world):
    """rs_route_ids_padded_spread: a sequence column that is ~60 % padding.  Padding ids take a slot at owner
    hash(i) mod world: the buckets stay balanced (the default capacity holds, where owner-0 padding would overflow it) and
    the layout equals the oracle's bit for bit."""
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    from recommendsystem_b200.sharded import bucket_capacity
    rng = np.random.default_rng(n_b + T + world)
    rows = np.asarray([7919], np.int64)
    lbase = np.zeros(1, np.int64)
    ids = rng.integers(0, 2 ** 45, size=(n_b, T)).astype(np.int64)
    lens = rng.integers(0, T + 1, size=n_b)
    ids[np.arange(T)[None, :] >= (lens * 0.8).astype(np.int64)[:, None]] = -1
    flat = ids.reshape(-1, 1)
    cap = bucket_capacity(flat.size, world)
    sr, inv, cnt, ovf = onp.route_ids_padded(flat, 1, rows, lbase, world, cap, pad_spread=True)
    assert ovf == 0
    assert onp.route_ids_padded(flat, 1, rows, lbase, world, cap)[3] == 1 or world == 2      # owner-0 padding overflows
    g_sr, g_inv, g_cnt, g_ovf = ops.route_ids_padded(_t(flat, cuda_dev), 1, _t(rows, cuda_dev), _t(lbase, cuda_dev),
                                                     world, cap, pad_spread=True)
    assert int(g_ovf.item()) == 0
    assert np.array_equal(g_cnt.cpu().numpy(), cnt)
    assert np.array_equal(g_inv.cpu().numpy(), inv)
    assert np.array_equal(g_sr.cpu().numpy(), sr)


@pytest.mark.parametrize("n_b,F,world,cap", [(300, 39, 8, 1700), (1024, 39, 2, 20096), (77, 5, 4, 128),
                                             (64, 1, 2, 16)])
def test_route_ids_padded_bit_exact(cuda_dev, n_b, F, world, cap):
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(n_b + F + world)
    rows = rng.integers(10, 100000, size=F).astype(np.int64)
    per = (rows + world - 1) // world
    lbase = np.zeros(F, np.int64)
    lbase[1:] = np.cumsum(per)[:-1]
    ids = rng.integers(0, 2 ** 45, size=(n_b, F)).astype(np.int64)
    ids[rng.random((n_b, F)) < 0.02] = -1
    sr, inv, cnt, ovf = onp.route_ids_padded(ids, F, rows, lbase, world, cap)
    g_sr, g_inv, g_cnt, g_ovf = ops.route_ids_padded(_t(ids, cuda_dev), F, _t(rows, cuda_dev), _t(lbase, cuda_dev),
                                                     world, cap)
    assert int(g_ovf.item()) == ovf
    assert np.array_equal(g_cnt.cpu().numpy(), cnt)
    assert np.array_equal(g_inv.cpu().numpy(), inv)
    assert np.array_equal(g_sr.cpu().numpy(), sr)
    # un-permute with dropped lookups (-1) yields zero rows; scatter skips them
    src = torch.randn(world * cap, 16, device=cuda_dev)
    got = ops.permute_rows(src, g_inv, scatter=False).cpu().numpy()
    ref = np.where((inv >= 0)[:, None], src.cpu().numpy()[np.maximum(inv, 0)], 0)
    assert np.array_equal(got, ref)


@pytest.mark.parametrize("W", [1, 2, 3, 8])
@pytest.mark.parametrize("d,odt", [(16, "bf16"), (16, "f32"), (8, "f32"), (32, "bf16")])
def test_embed_gather_peer_sharded_layout(cuda_dev, W, d, odt):
    """rs_embed_gather_peer_fwd on W shards (all resident on this GPU here; CUDA-IPC peer mappings in the
    multi-process trainer): owner = row mod W, local row = local_base[f] + row div W must reproduce the
    unsharded gather BIT-EXACTLY, padding ids included."""
    from recommendsystem_b200 import ops
    from recommendsystem_b200.sharded import shard_layout
    rng = np.random.default_rng(W * 100 + d)
    F, B = 7, 333
    rows = rng.integers(1, 300, size=F).astype(np.int64)
    base = np.concatenate([[0], np.cumsum(rows)[:-1]]).astype(np.int64)
    table = rng.standard_normal((int(rows.sum()), d)).astype(np.float32)
    ids = rng.integers(0, 2 ** 45, size=(B, F)).astype(np.int64)
    ids[5, 2] = -1
    ids[0, 0] = -7
    local_rows, local_base = shard_layout(rows, W)
    shards = []
    for r in range(W):
        sh = np.zeros((int(local_rows.sum()), d), np.float32)
        for f in range(F):
            src = table[base[f] + r: base[f] + rows[f]: W]
            sh[local_base[f]: local_base[f] + len(src)] = src
        shards.append(torch.from_numpy(sh).to(cuda_dev))
    dt = torch.bfloat16 if odt == "bf16" else torch.float32
    tids = torch.from_numpy(ids).to(cuda_dev)
    got = ops.embed_gather_peer(shards, tids, torch.from_numpy(local_base).to(cuda_dev),
                                torch.from_numpy(rows).to(cuda_dev), dt)
    ref, _, _ = ops.embed_gather(torch.from_numpy(table).to(cuda_dev), tids, torch.from_numpy(base).to(cuda_dev),
                                 torch.from_numpy(rows).to(cuda_dev), dt)
    assert torch.equal(got, ref)
    assert float(got[5, 2].abs().sum()) == 0.0


@pytest.mark.parametrize("n", [1, 1000, 666, 32808, 300001])
def test_embed_keys_from_rows(cuda_dev, n):
    """The owners' sort keys of the sharded exchange: rs_embed_keys_from_rows = (row << 32 | slot), padding (row -1)
    included, = the keys rs_embed_gather_rows_ld writes as a by-product of a gather by the same rows."""
    from recommendsystem_b200 import cabi, ops
    rng = np.random.default_rng(n)
    R, d = 5000, 16
    rowidx = rng.integers(-1, R, size=n).astype(np.int32)
    rows = torch.from_numpy(rowidx).to(cuda_dev)
    keys = torch.empty(n, dtype=torch.int64, device=cuda_dev)
    cabi.call("rs_embed_keys_from_rows", rows.data_ptr(), n, keys.data_ptr(), ops._stream())
    want = ((rowidx.astype(np.int64) & 0xFFFFFFFF) << 32) | np.arange(n, dtype=np.int64)
    assert np.array_equal(keys.cpu().numpy().view(np.uint64), want.view(np.uint64))
    table = torch.zeros(R, 3, d, device=cuda_dev)[:, 0, :]
    keys_gather = torch.empty_like(keys)
    cabi.call("rs_embed_gather_rows_ld", table.data_ptr(), table.stride(0), rows.data_ptr(), n, d, None, cabi.RS_F32,
              None, keys_gather.data_ptr(), ops._stream())
    assert torch.equal(keys, keys_gather)


@pytest.mark.parametrize("d", [8, 16, 32])
@pytest.mark.parametrize("hot", [[(7, 1000)], [(3, 33), (9, 64), (11, 500)], [(0, 4097), (1, 31), (2, 32), (5, 95)]])
def test_segsum_long_runs_bit_exact(cuda_dev, d, hot):
    """Skewed ids: rows that occur hundreds / thousands of times in a batch (runs spanning many 32-key warp
    windows, at every alignment).  The warp-cooperative continuation must add the rows in the same
    left-to-right order as the oracle: bit-exact segment sums, and the fused Adam update on top of them."""
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(d + len(hot))
    R = 64
    rowidx = [rng.integers(12, R, size=700).astype(np.int32)]
    for r, cnt in hot:
        rowidx.append(np.full(cnt, r, np.int32))
    rowidx = np.concatenate(rowidx)
    rng.shuffle(rowidx)
    n = len(rowidx)
    grad = rng.standard_normal((n, d)).astype(np.float32)
    ks = _sorted_keys(ops, _t(rowidx, cuda_dev), R)
    seg_rows, seg_sum = ops.segsum(_t(grad, cuda_dev), ks)
    heads = seg_rows.cpu().numpy() >= 0
    uniq, sums = onp.segment_sum_sorted(rowidx, grad)
    assert np.array_equal(seg_rows.cpu().numpy()[heads].astype(np.int64), uniq)
    assert np.array_equal(seg_sum.cpu().numpy()[heads], sums)
    # fused sparse Adam over the same keys
    w = (rng.standard_normal((R, d)) * 0.1).astype(np.float32)
    wt, mt, vt = _t(w, cuda_dev), torch.zeros(R, d, device=cuda_dev), torch.zeros(R, d, device=cuda_dev)
    scal = torch.zeros(4, device=cuda_dev)
    ops.adam_advance(scal, 0.9, 0.999)
    ops.segsum_adam(wt, mt, vt, _t(grad, cuda_dev), ks, 1e-2, 0.9, 0.999, 1e-8, scal)
    _, _, corr = onp.adam_scalars(1, 0.9, 0.999)
    w2, m2, v2 = onp.sparse_adam(w.astype(np.float64), np.zeros((R, d)), np.zeros((R, d)), rowidx, grad, 1e-2, 0.9, 0.999,
                                 1e-8, float(corr))
    assert_close(wt.cpu().numpy(), w2, REL_F32, "sparse Adam after long runs")
