"""GPU parity of the sparse-embedding kernels at the sizes the benchmarks run: past one grid wave.

The gather, segment-sum / fused-optimizer and dense-Adam kernels cap their grid and loop (grid-stride), so every
case here is sized from the device's SM count to take at least two trips, and asserts that it does.  The host
references are vectorised restatements of oracle/oracle_np.py (pinned against it on small cases); optimizer state is
compared ROW BY ROW, and rows an update must not touch are checked bit-identical on the device.
"""
import numpy as np
import pytest

from util import REL_F32

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

# Launch caps in csrc/embed.cu:
#   launch_gather     min(cdiv(n, 4 warps * 32*LPL), sm*16) CTAs of 128 threads; LPL = 4 (d <= 8), 2 (d <= 16), else 1
#   dispatch_segsum   min(cdiv(n, 128), sm*16) CTAs of 128 threads, 32 sorted keys per warp per trip
#   rs_dense_adam     min(cdiv(n, 256), sm*8) CTAs of 256 threads, one element per thread per trip
HEADLINE_ROWS = [1_000_000] * 39                    # bench.py's AutoInt arena: 39 fields x 1 M rows (row_bits 26)
LR, B1, B2, EPS = 1e-2, 0.9, 0.999, 1e-8


def _sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def gather_wave(d):
    lpl = 4 if d <= 8 else (2 if d <= 16 else 1)
    return _sm() * 16 * 4 * 32 * lpl


def segsum_wave():
    return _sm() * 16 * 4 * 32


def dense_adam_wave():
    return _sm() * 8 * 256


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _batch(n0, F, wave, trips=2):
    """Rows of a batch of F fields: the benchmarked n0 lookups, or more when this part's wave needs it to take
    `trips` grid-stride trips."""
    B = max(-(-n0 // F), ((trips - 1) * wave) // F + 1)
    assert B * F > (trips - 1) * wave
    return B


def _ids(rng, shape, rows, dist, pad=0.03):
    """Ids of fields rows[f] (last axis): uniform, or Zipf(1.05) popularity over a random permutation of each field's
    rows (bench.py --ids zipf); a fraction `pad` is padding (-1)."""
    rows = np.asarray(rows, np.int64)
    if dist == "uniform":
        ids = rng.integers(0, 2 ** 40, size=shape).astype(np.int64)
    else:
        R = int(rows.max())
        p = 1.0 / np.arange(1, R + 1, dtype=np.float64) ** 1.05
        rank = rng.choice(R, size=shape, p=p / p.sum())
        ids = rng.permutation(R)[rank].astype(np.int64)
    ids[rng.random(shape) < pad] = -1
    return ids


def _layout(rows):
    rows = np.asarray(rows, np.int64)
    return rows, np.concatenate([[0], np.cumsum(rows)[:-1]]).astype(np.int64)


# ------------------------------------------------------------ vectorised references


def seg_sum_ref(rowidx, grad):
    """oracle_np.segment_sum_sorted, vectorised: (unique rows >= 0 ascending, their fp32 sums in lookup order).
    Stable sort, then the k-th element of every run longer than k is added for k = 1, 2, ... (left to right)."""
    rowidx = np.asarray(rowidx, np.int64).reshape(-1)
    grad = grad.reshape(len(rowidx), -1)
    order = np.argsort(rowidx, kind="stable")
    order = order[rowidx[order] >= 0]
    sr = rowidx[order]
    if sr.size == 0:
        return np.zeros(0, np.int64), np.zeros((0, grad.shape[1]), grad.dtype)
    new = np.r_[True, sr[1:] != sr[:-1]]
    start = np.flatnonzero(new)
    run = np.cumsum(new) - 1
    k = np.arange(sr.size) - start[run]
    sums = grad[order[start]].copy()
    by_k = np.argsort(k, kind="stable")
    counts = np.bincount(k)
    o = int(counts[0])
    for c in counts[1:]:
        sel = by_k[o:o + c]
        sums[run[sel]] += grad[order[sel]]          # one element per run: no index repeats
        o += int(c)
    return sr[start], sums


def scaled_sum_ref(rowidx, grad, grad_scale):
    """The per-row gradient the fused kernels apply: every occurrence scaled in fp32, summed left to right in fp32."""
    return seg_sum_ref(rowidx, (grad.astype(np.float32) * np.float32(grad_scale)).astype(np.float32))


def adam_ref(w, m, v, g, corr):
    """fp64 Adam on rows (oracle_np.sparse_adam restricted to the touched rows)."""
    b1, b2, lr, eps = (np.float64(np.float32(t)) for t in (B1, B2, LR, EPS))
    g = g.astype(np.float64)
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    return w - lr * np.float64(corr) * m / (np.sqrt(v) + eps), m, v


def adagrad_ref(w, g2, g, lr, eps, per_element):
    g = g.astype(np.float64)
    g2 = g2 + g * g if per_element else g2 + (g * g).sum(1) / g.shape[1]
    den = np.sqrt(g2) + eps if per_element else (np.sqrt(g2) + eps)[:, None]
    return w - lr * g / den, g2


def assert_rows_close(got, ref, rel, what, ulp_of=None):
    """Per row: |got - ref| <= rel * max|ref row| (+ 2 ulps of |ulp_of| element-wise, for a value rounded to fp32)."""
    got = np.asarray(got, np.float64).reshape(len(got), -1)
    ref = np.asarray(ref, np.float64).reshape(len(ref), -1)
    err = np.abs(got - ref)
    bound = rel * np.abs(ref).max(1, keepdims=True)
    if ulp_of is not None:
        bound = bound + 2 * np.spacing(np.abs(np.asarray(ulp_of, np.float32))).reshape(bound.shape[0], -1)
    bad = np.flatnonzero((err > bound).any(1))
    worst = float((err / np.maximum(np.abs(ref).max(1, keepdims=True), 1e-30)).max()) if err.size else 0.0
    assert bad.size == 0, f"{what}: {bad.size} of {len(got)} rows out of bound (first {bad[:5]}), worst row rel {worst:.2e}"


def assert_untouched(after, before, touched):
    """Rows outside `touched` (host int64) are bit-identical to `before` (compared on the device)."""
    changed = (after != before).reshape(after.shape[0], -1).any(1)
    keep = torch.ones(after.shape[0], dtype=torch.bool, device=after.device)
    keep[_t(touched, after.device)] = False
    n = int((changed & keep).sum())
    assert n == 0, f"{n} rows changed that the batch does not touch"


def _gather_keys(rows_flat):
    """What the gather kernels write: (uint32(row) << 32) | lookup index."""
    r = rows_flat.astype(np.int64).reshape(-1)
    return ((r & 0xFFFFFFFF) << 32 | np.arange(r.size, dtype=np.int64)).view(np.uint64)


def _sorted_keys_ref(keys_u64):
    """Stable sort on the row half (padding = all-ones row sorts last)."""
    return keys_u64[np.argsort(keys_u64 >> np.uint64(32), kind="stable")]


# ------------------------------------------------------------------- pins


def test_references_pinned_to_oracle():
    """The vectorised references equal oracle_np's loops on small cases (bit for bit)."""
    from oracle import oracle_np as onp
    rng = np.random.default_rng(1)
    R, d, n = 40, 12, 3000
    rowidx = rng.integers(-1, R, size=n)
    rowidx[100:400] = 7                              # a long run
    grad = rng.standard_normal((n, d)).astype(np.float32)
    u0, s0 = onp.segment_sum_sorted(rowidx, grad)
    u1, s1 = seg_sum_ref(rowidx, grad)
    assert np.array_equal(u0, u1) and np.array_equal(s0, s1)
    w = rng.standard_normal((R, d))
    m = rng.standard_normal((R, d)) * 0.01
    v = rng.random((R, d)) * 0.01
    corr = float(onp.adam_scalars(2, B1, B2)[2])
    w0, m0, v0 = onp.sparse_adam(w, m, v, rowidx, grad, LR, B1, B2, EPS, corr, grad_scale=0.5)
    u, g = scaled_sum_ref(rowidx, grad, 0.5)
    w1, m1, v1 = adam_ref(w[u], m[u], v[u], g, corr)
    assert np.array_equal(w0[u], w1) and np.array_equal(m0[u], m1) and np.array_equal(v0[u], v1)
    for per_element in (False, True):
        g2 = rng.random((R, d) if per_element else R) + 0.1
        w0, g20 = onp.sparse_adagrad(w, g2, rowidx, grad, 0.05, 1e-7, per_element, grad_scale=2.0)
        u, g = scaled_sum_ref(rowidx, grad, 2.0)
        w1, g21 = adagrad_ref(w[u], g2[u], g, 0.05, 1e-7, per_element)
        assert np.allclose(w0[u], w1, rtol=1e-14, atol=0) and np.allclose(g20[u], g21, rtol=1e-14, atol=0)
    # bag mean: fp32 left-to-right sum, as oracle_np.embed_bag_mean (which divides; the training kernel multiplies)
    F = 3
    rows, base = _layout([50, 7, 300])
    table = rng.standard_normal((int(rows.sum()), d)).astype(np.float32)
    lens = rng.integers(0, 7, size=60)
    offsets = np.r_[0, np.cumsum(lens)].astype(np.int64)
    ids = rng.integers(-1, 10 ** 6, size=int(offsets[-1])).astype(np.int64)
    ref = onp.embed_bag_mean(table, ids, offsets, rows, base, F)
    out, _, inv = bag_fwd_ref(table, ids, offsets, rows, base, F)
    cnt = np.bincount(np.repeat(np.arange(60), lens)[ids >= 0], minlength=60)
    assert np.allclose(out, ref, rtol=4e-7, atol=0) and np.array_equal(inv > 0, cnt > 0)


# ------------------------------------------------------------------ gather


@pytest.mark.parametrize("d", [4, 12, 16, 32, 96])
@pytest.mark.parametrize("ld_mult", [1, 3])
def test_gather_fwd_ld_three_waves(cuda_dev, d, ld_mult):
    """rs_embed_gather_fwd_ld over >= 3 waves: rows (padding zero), sort keys and arena rows bit-exact, f32 and bf16
    outputs, table row stride d (AdaGrad / plain tables) or 3d (Adam [w|m|v] records)."""
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(d * 10 + ld_mult)
    F = 39
    wave = gather_wave(d)
    B = _batch(0, F, wave, trips=4)
    n = B * F
    assert n > 3 * wave
    rows, base = _layout(rng.integers(50, 5000, size=F))
    full = (rng.standard_normal((int(rows.sum()), 3 * d)) * 0.1).astype(np.float32)
    tab = full[:, :d] if ld_mult == 3 else np.ascontiguousarray(full[:, :d])
    tab_t = _t(full, cuda_dev)[:, :d] if ld_mult == 3 else _t(tab, cuda_dev)
    assert tab_t.stride(0) == ld_mult * d
    ids = _ids(rng, (B, F), rows, "uniform", pad=0.05)
    ref, ref_rows = onp.embed_gather(tab, ids, rows, base)
    args = (tab_t, _t(ids, cuda_dev), _t(base, cuda_dev), _t(rows, cuda_dev))
    out, keys, rws = ops.embed_gather(*args, want_keys=True, want_rows=True)
    assert np.array_equal(out.cpu().numpy(), ref)
    assert np.array_equal(rws.cpu().numpy().astype(np.int64), ref_rows)
    assert np.array_equal(keys.cpu().numpy().view(np.uint64), _gather_keys(ref_rows))
    outb, _, _ = ops.embed_gather(*args, out_dtype=torch.bfloat16)
    assert torch.equal(outb, out.to(torch.bfloat16))


def test_gather_rows_ld_seq_shape(cuda_dev):
    """rs_embed_gather_rows_ld at the cfg5 sequence shape (16384 x 50, about half padding) from [w|m|v] records:
    rows, mask and keys bit-exact."""
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(50)
    d, T = 32, 50
    B = _batch(16384 * T, T, gather_wave(d))
    R = 300_000
    full = rng.standard_normal((R, 3 * d)).astype(np.float32)
    rowidx = rng.integers(0, R, size=(B, T)).astype(np.int32)
    lens = rng.integers(0, T + 1, size=B)
    rowidx[np.arange(T)[None, :] >= lens[:, None]] = -1
    assert 0.4 < (rowidx < 0).mean() < 0.6
    ref, refm = onp.embed_gather_rows(full[:, :d], rowidx)
    tab = _t(full, cuda_dev)[:, :d]
    out, mask, keys = ops.embed_gather_rows(tab, _t(rowidx, cuda_dev), want_mask=True, want_keys=True)
    assert np.array_equal(out.cpu().numpy(), ref)
    assert np.array_equal(mask.cpu().numpy(), refm)
    assert np.array_equal(keys.cpu().numpy().view(np.uint64), _gather_keys(rowidx))
    outb, _, _ = ops.embed_gather_rows(tab, _t(rowidx, cuda_dev), out_dtype=torch.bfloat16)
    assert torch.equal(outb, out.to(torch.bfloat16))


# ------------------------------------------------------- sort + segment sum


def _check_sort_segsum(dev, rowidx, grad, rbits, wave=None):
    """Sort the gather-style keys of `rowidx` (padding < 0), segment-sum `grad` over them twice: sorted keys, heads
    and sums bit-exact against numpy, identical bits on the second run."""
    from recommendsystem_b200 import ops
    keys = _gather_keys(rowidx)
    ks = ops.sort_keys(_t(keys.view(np.int64), dev), rbits)
    assert np.array_equal(ks.cpu().numpy().view(np.uint64), _sorted_keys_ref(keys))
    gt = _t(grad, dev)
    seg_rows, seg_sum = ops.segsum(gt, ks)
    seg_rows2, seg_sum2 = ops.segsum(gt, ks)
    sr = seg_rows.cpu().numpy()
    heads = sr >= 0
    uniq, sums = seg_sum_ref(rowidx, grad.astype(np.float32))
    assert np.array_equal(sr[heads].astype(np.int64), uniq)
    assert np.array_equal(seg_sum.cpu().numpy()[heads], sums)
    assert torch.equal(seg_rows, seg_rows2)
    h = torch.from_numpy(heads).to(dev)
    assert torch.equal(seg_sum[h], seg_sum2[h])
    return ks


@pytest.mark.parametrize("n0,d", [(8192 * 39, 16), (16384 * 91, 32)])
@pytest.mark.parametrize("dist", ["uniform", "zipf"])
def test_sort_segsum_headline_arena(cuda_dev, n0, d, dist):
    """ops.sort_keys (26 row bits: the 39 x 1 M headline arena) + ops.segsum at the headline (319,488 keys) and cfg5
    (1.49 M keys) sizes, uniform and Zipf(1.05) ids, with padding: bit-exact and run-to-run identical."""
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rows, base = _layout(HEADLINE_ROWS)
    rbits = ops.row_bits(int(rows.sum()))
    assert rbits == 26
    F = len(rows)
    wave = segsum_wave()
    B = _batch(n0, F, wave)
    assert B * F > wave
    rng = np.random.default_rng(n0 + d + len(dist))
    ids = _ids(rng, (B, F), rows, dist)
    rowidx = onp.embed_rows(ids, rows, base).reshape(-1)
    grad = rng.standard_normal((rowidx.size, d)).astype(np.float32)
    _check_sort_segsum(cuda_dev, rowidx, grad, rbits)


def _runs_layout(n, specials, rng):
    """Run lengths covering [0, n) in sorted order: `specials` (start, length) runs, random 1-3 long runs between."""
    lens, pos = [], 0
    for s, ln in sorted(specials):
        assert s >= pos and s + ln <= n
        while pos < s:
            k = int(min(rng.integers(1, 4), s - pos))
            lens.append(k)
            pos += k
        lens.append(ln)
        pos += ln
    while pos < n:
        k = int(min(rng.integers(1, 4), n - pos))
        lens.append(k)
        pos += k
    return np.asarray(lens)


def test_segsum_constructed_runs(cuda_dev):
    """Runs placed where the warp windows and the grid wave split them: starting on the last key of a 32-key window
    (lengths 1, 2, 33, 700, 1000), spanning exactly one and exactly two aligned windows, starting on the last key of
    the first wave and straddling the wave boundary, and ending at key n - 1."""
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(77)
    W = segsum_wave()
    n = W + 4000
    specials = [(32 * 10 + 31, 1), (32 * 20 + 31, 2), (32 * 30 + 31, 33), (32 * 50 + 31, 1000), (32 * 100, 32),
                (32 * 200, 64), (W // 2 - 1, 700), (W - 1 - 32 * 40, 2), (W - 1, 150), (n - 777, 777)]
    lens = _runs_layout(n, specials, rng)
    row_of_run = np.cumsum(rng.integers(1, 200, size=lens.size))
    rbits = ops.row_bits(sum(HEADLINE_ROWS))
    assert row_of_run[-1] < 2 ** rbits - 1
    sorted_rows = np.repeat(row_of_run, lens)
    starts = np.r_[0, np.cumsum(lens)[:-1]]
    for s, ln in specials:                         # the layout really has these runs
        i = np.searchsorted(starts, s)
        assert starts[i] == s and lens[i] == ln
    rowidx = np.empty(n, np.int64)
    rowidx[rng.permutation(n)] = sorted_rows       # stable sort restores the layout
    grad = rng.standard_normal((n, 8)).astype(np.float32)
    ks = _check_sort_segsum(cuda_dev, rowidx, grad, rbits)
    assert np.array_equal((ks.cpu().numpy().view(np.uint64) >> np.uint64(32)).astype(np.int64), sorted_rows)


@pytest.mark.parametrize("k", [17, 26])
@pytest.mark.parametrize("delta", [-1, 0, 1])
def test_sort_row_bits_edges(cuda_dev, k, delta):
    """Arenas of 2^k - 1, 2^k and 2^k + 1 rows: row_bits is just wide enough, the top rows sort before padding keys
    (gather-style and all-ones) that sit next to them, and padding is never summed."""
    from recommendsystem_b200 import ops
    total = 2 ** k + delta
    rbits = ops.row_bits(total)
    assert rbits == (k if delta < 0 else k + 1)
    assert total - 1 < 2 ** rbits - 1              # the largest row stays below the padding key's row bits
    rng = np.random.default_rng(k * 3 + delta)
    n = 60_000
    rowidx = rng.integers(0, total, size=n)
    top = rng.random(n)
    rowidx[top < 0.2] = total - 1
    rowidx[(top >= 0.2) & (top < 0.25)] = total - 2
    rowidx[(top >= 0.25) & (top < 0.27)] = 0
    rowidx[(top >= 0.27) & (top < 0.4)] = -1
    grad = rng.standard_normal((n, 4)).astype(np.float32)
    _check_sort_segsum(cuda_dev, rowidx, grad, rbits)
    # padding written by the bag kernel is all ones (low half too): still last, in input order
    keys = _gather_keys(rowidx)
    keys[rowidx < 0] = np.uint64(0xFFFFFFFFFFFFFFFF)
    ks = ops.sort_keys(_t(keys.view(np.int64), cuda_dev), rbits)
    assert np.array_equal(ks.cpu().numpy().view(np.uint64), _sorted_keys_ref(keys))
    seg_rows, _ = ops.segsum(_t(grad, cuda_dev), ks)
    assert np.array_equal(seg_rows.cpu().numpy()[seg_rows.cpu().numpy() >= 0].astype(np.int64),
                          np.unique(rowidx[rowidx >= 0]))


# ------------------------------------------------------------ fused optimizers


def _grads(rng, n, d, gdt, dev):
    g = rng.standard_normal((n, d)).astype(np.float32)
    gt = _t(g, dev)
    if gdt == "bf16":
        gt = gt.to(torch.bfloat16)
        g = gt.float().cpu().numpy()
    return g, gt


@pytest.mark.parametrize("d,n0,F,R,gdt,scale,dist", [
    (16, 8192 * 39, 39, 20_000, "f32", 1.0, "uniform"),       # headline AutoInt
    (16, 8192 * 39, 39, 20_000, "bf16", 0.5, "zipf"),
    (96, 4096 * 176, 176, 2_000, "f32", 1.0, "uniform"),      # rank/ctr: 24 of 32 lanes busy
    (12, 8192 * 39, 39, 5_000, "f32", 0.25, "zipf"),          # 3 of 4 lanes busy
    (20, 8192 * 39, 39, 5_000, "bf16", 2.0, "uniform"),       # 5 of 8 lanes busy
])
def test_segsum_adam_arena_records(cuda_dev, d, n0, F, R, gdt, scale, dist):
    """gather keys -> sort -> segsum_adam on the Arena's interleaved [w|m|v] records (state_ld = 3d), two steps from
    random non-zero moments: m, v and dw of every touched row against fp64 Adam on the fp32 left-to-right sums;
    every other row bit-identical."""
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    from recommendsystem_b200.arena import Arena
    rng = np.random.default_rng(d * 1000 + F)
    ar = Arena([R] * F, d, cuda_dev)
    assert ar.w.stride(0) == 3 * d
    gen = torch.Generator(device=cuda_dev).manual_seed(d)
    ar.w.normal_(0.0, 0.1, generator=gen)
    ar.m.normal_(0.0, 0.01, generator=gen)
    ar.v.uniform_(1e-4, 1e-2, generator=gen)
    wave = segsum_wave()
    B = _batch(n0, F, wave)
    scal = torch.zeros(4, device=cuda_dev)
    for step in (1, 2):
        ids = _ids(rng, (B, F), ar.rows, dist)
        rowidx = onp.embed_rows(ids, ar.rows, ar.base).reshape(-1)
        g, gt = _grads(rng, rowidx.size, d, gdt, cuda_dev)
        tids, rb, rr = ar.lookup(_t(ids, cuda_dev), range(F), insert=False)
        _, keys, _ = ops.embed_gather(ar.w, tids, rb, rr, want_keys=True)
        ks = ops.sort_keys(keys, ar.row_bits)
        before = ar.records.clone()
        ops.adam_advance(scal, B1, B2)
        ops.segsum_adam(ar.w, ar.m, ar.v, gt, ks, LR, B1, B2, EPS, scal, grad_scale=scale)
        uniq, gsum = scaled_sum_ref(rowidx, g, scale)
        u = _t(uniq, cuda_dev)
        old = before[u].cpu().numpy().astype(np.float64)
        new = ar.records[u].cpu().numpy()
        w, m, v = adam_ref(old[:, 0], old[:, 1], old[:, 2], gsum, onp.adam_scalars(step, B1, B2)[2])
        assert_rows_close(new[:, 1], m, REL_F32, f"step {step} m")
        assert_rows_close(new[:, 2], v, REL_F32, f"step {step} v")
        assert_rows_close(new[:, 0] - old[:, 0], w - old[:, 0], REL_F32, f"step {step} dw", ulp_of=new[:, 0])
        assert_untouched(ar.records, before, uniq)


@pytest.mark.parametrize("d,n0,F,R,per_element,gdt,scale,dist", [
    (32, 16384 * 91, 91, 20_000, False, "f32", 1.0, "uniform"),    # cfg5 VideoDnn: AdaGrad per row
    (32, 16384 * 91, 91, 20_000, True, "bf16", 0.5, "zipf"),
    (12, 8192 * 39, 39, 5_000, False, "f32", 0.25, "zipf"),        # idle lanes in the g2sum butterfly
    (20, 8192 * 39, 39, 5_000, False, "bf16", 2.0, "uniform"),
    (12, 8192 * 39, 39, 5_000, True, "f32", 1.0, "uniform"),
])
def test_segsum_adagrad_arena(cuda_dev, d, n0, F, R, per_element, gdt, scale, dist):
    """gather keys -> sort -> segsum_adagrad on an AdaGrad Arena, two steps from random g2sum: g2sum and dw of every
    touched row against fp64 AdaGrad on the fp32 left-to-right sums; every other row bit-identical."""
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    from recommendsystem_b200.arena import Arena
    rng = np.random.default_rng(d * 100 + F + per_element)
    lr, eps = 0.05, 1e-7
    ar = Arena([R] * F, d, cuda_dev, adagrad=(0.1, per_element))
    gen = torch.Generator(device=cuda_dev).manual_seed(d + 1)
    ar.w.normal_(0.0, 0.1, generator=gen)
    ar.g2sum.uniform_(0.05, 0.5, generator=gen)
    B = _batch(n0, F, segsum_wave())
    for step in (1, 2):
        ids = _ids(rng, (B, F), ar.rows, dist)
        rowidx = onp.embed_rows(ids, ar.rows, ar.base).reshape(-1)
        g, gt = _grads(rng, rowidx.size, d, gdt, cuda_dev)
        tids, rb, rr = ar.lookup(_t(ids, cuda_dev), range(F), insert=False)
        _, keys, _ = ops.embed_gather(ar.w, tids, rb, rr, want_keys=True)
        ks = ops.sort_keys(keys, ar.row_bits)
        w0, s0 = ar.w.clone(), ar.g2sum.clone()
        ops.segsum_adagrad(ar.w, ar.g2sum, gt, ks, lr, eps, per_element, grad_scale=scale)
        uniq, gsum = scaled_sum_ref(rowidx, g, scale)
        u = _t(uniq, cuda_dev)
        wo = w0[u].cpu().numpy().astype(np.float64)
        wn, sn = ar.w[u].cpu().numpy(), ar.g2sum[u].cpu().numpy()
        w, s = adagrad_ref(wo, s0[u].cpu().numpy().astype(np.float64), gsum, lr, eps, per_element)
        assert_rows_close(sn, s, REL_F32, f"step {step} g2sum")
        assert_rows_close(wn - wo, w - wo, REL_F32, f"step {step} dw", ulp_of=wn)
        assert_untouched(ar.w, w0, uniq)
        assert_untouched(ar.g2sum, s0, uniq)


# ------------------------------------------------------------------ CSR bags


def bag_fwd_ref(table, ids, offsets, rows, base, F):
    """rs_embed_bag_fwd_ld restated: (fp32 sum in id order) * fp32(1 / count) per bag (0 for an empty or all-padding
    bag), sort keys (row << 32 | position; all ones for padding), inv_cnt."""
    n_bags = len(offsets) - 1
    bag = np.repeat(np.arange(n_bags), np.diff(offsets))
    valid = ids >= 0
    f = bag % F
    r = np.where(valid, base[f] + np.mod(ids, rows[f]), -1)
    cnt = np.bincount(bag[valid], minlength=n_bags)
    inv = np.where(cnt > 0, np.float32(1) / np.maximum(cnt, 1).astype(np.float32), np.float32(0)).astype(np.float32)
    ub, sums = seg_sum_ref(np.where(valid, bag, -1), table[np.maximum(r, 0)])
    out = np.zeros((n_bags, table.shape[1]), np.float32)
    out[ub] = sums * inv[ub, None]
    keys = np.where(valid, (r & 0xFFFFFFFF) << 32 | np.arange(ids.size), -1).astype(np.int64).view(np.uint64)
    return out, keys, inv


@pytest.mark.parametrize("opt,ddt", [("adam", "f32"), ("adagrad", "bf16")])
def test_csr_bags_fwd_grad_update(cuda_dev, opt, ddt):
    """rs_embed_bag_fwd_ld (from the arena's rows, stride 3d with Adam records) and rs_embed_bag_grad over 200 k bags
    with empty, all-padding, single-id and several-hundred-id bags: outputs, keys and inv_cnt bit-exact; then sort +
    the fused optimizer against a dense fp64 restatement of mean-combiner backward + optimizer."""
    from oracle import oracle_np as onp
    from recommendsystem_b200 import cabi, ops
    from recommendsystem_b200.arena import Arena
    rng = np.random.default_rng(len(opt))
    d = 32
    rows_f = [50_000, 3_000, 200_000, 777, 40_000]
    F = len(rows_f)
    ar = Arena(rows_f, d, cuda_dev, adagrad=None if opt == "adam" else (0.1, False))
    gen = torch.Generator(device=cuda_dev).manual_seed(5)
    ar.w.normal_(0.0, 0.1, generator=gen)
    if opt == "adam":
        ar.m.normal_(0.0, 0.01, generator=gen)
        ar.v.uniform_(1e-4, 1e-2, generator=gen)
    else:
        ar.g2sum.uniform_(0.05, 0.5, generator=gen)
    n_bags = 200_000
    lens = rng.integers(0, 6, size=n_bags)
    kind = rng.random(n_bags)
    lens[kind < 0.005] = rng.integers(200, 600, size=int((kind < 0.005).sum()))       # long bags
    lens[(kind >= 0.005) & (kind < 0.03)] = 1
    offsets = np.r_[0, np.cumsum(lens)].astype(np.int64)
    ids = rng.integers(0, 2 ** 40, size=int(offsets[-1])).astype(np.int64)
    ids[rng.random(ids.size) < 0.05] = -1
    allpad = np.flatnonzero((kind >= 0.03) & (kind < 0.04) & (lens > 0))
    for b in allpad[:500]:
        ids[offsets[b]:offsets[b + 1]] = -1
    assert (lens == 0).sum() > 1000 and (lens == 1).sum() > 1000 and lens.max() >= 500
    w_host = ar.w.cpu().numpy()
    ref_out, ref_keys, ref_inv = bag_fwd_ref(w_host, ids, offsets, ar.rows, ar.base, F)
    assert (ref_inv[allpad[:500]] == 0).all()
    ids_t, off_t = _t(ids, cuda_dev), _t(offsets, cuda_dev)
    rb, rr = ar.geom(range(F))
    out = torch.empty(n_bags, d, device=cuda_dev)
    outb = torch.empty(n_bags, d, dtype=torch.bfloat16, device=cuda_dev)
    keys = torch.empty(ids.size, dtype=torch.int64, device=cuda_dev)
    inv = torch.empty(n_bags, device=cuda_dev)
    st = ops._stream()
    cabi.call("rs_embed_bag_fwd_ld", ar.w.data_ptr(), ar.w.stride(0), ids_t.data_ptr(), off_t.data_ptr(),
              rb.data_ptr(), rr.data_ptr(), n_bags, F, d, out.data_ptr(), cabi.RS_F32, keys.data_ptr(),
              inv.data_ptr(), st)
    cabi.call("rs_embed_bag_fwd_ld", ar.w.data_ptr(), ar.w.stride(0), ids_t.data_ptr(), off_t.data_ptr(),
              rb.data_ptr(), rr.data_ptr(), n_bags, F, d, outb.data_ptr(), cabi.RS_BF16, None, None, st)
    assert np.array_equal(out.cpu().numpy(), ref_out)
    assert torch.equal(outb, out.to(torch.bfloat16))
    assert np.array_equal(keys.cpu().numpy().view(np.uint64), ref_keys)
    assert np.array_equal(inv.cpu().numpy(), ref_inv)
    # backward of the mean: occurrence p of bag b gets dout[b] * inv_cnt[b] (padding positions too; the sort drops them)
    dout, dout_t = _grads(rng, n_bags, d, ddt, cuda_dev)
    g_occ = torch.empty(ids.size, d, device=cuda_dev)
    cabi.call("rs_embed_bag_grad", dout_t.data_ptr(), ops._dt(dout_t), off_t.data_ptr(), inv.data_ptr(), n_bags, d,
              g_occ.data_ptr(), st)
    bag = np.repeat(np.arange(n_bags), lens)
    assert np.array_equal(g_occ.cpu().numpy(), dout[bag] * ref_inv[bag, None])
    # chained update against the dense fp64 gradient of the mean combiner
    ks = ops.sort_keys(keys, ar.row_bits)
    state = ar.records if opt == "adam" else ar.w
    before, g2_before = state.clone(), (None if opt == "adam" else ar.g2sum.clone())
    valid = ids >= 0
    r = (ar.base[bag % F] + np.mod(ids, ar.rows[bag % F]))[valid]
    cnt = np.bincount(bag[valid], minlength=n_bags).astype(np.float64)
    uniq, pos = np.unique(r, return_inverse=True)
    G = np.zeros((uniq.size, d))
    np.add.at(G, pos, dout.astype(np.float64)[bag[valid]] / cnt[bag[valid], None])
    u = _t(uniq, cuda_dev)
    if opt == "adam":
        scal = torch.zeros(4, device=cuda_dev)
        ops.adam_advance(scal, B1, B2)
        ops.segsum_adam(ar.w, ar.m, ar.v, g_occ, ks, LR, B1, B2, EPS, scal)
        old = before[u].cpu().numpy().astype(np.float64)
        new = ar.records[u].cpu().numpy()
        w, m, v = adam_ref(old[:, 0], old[:, 1], old[:, 2], G, onp.adam_scalars(1, B1, B2)[2])
        assert_rows_close(new[:, 1], m, 1e-4, "bag adam m")
        assert_rows_close(new[:, 2], v, 1e-4, "bag adam v")
        assert_rows_close(new[:, 0] - old[:, 0], w - old[:, 0], 1e-4, "bag adam dw", ulp_of=new[:, 0])
    else:
        ops.segsum_adagrad(ar.w, ar.g2sum, g_occ, ks, 0.05, 1e-7, False)
        wo = before[u].cpu().numpy().astype(np.float64)
        w, s = adagrad_ref(wo, g2_before[u].cpu().numpy().astype(np.float64), G, 0.05, 1e-7, False)
        assert_rows_close(ar.g2sum[u].cpu().numpy(), s, 1e-4, "bag adagrad g2sum")
        wn = ar.w[u].cpu().numpy()
        assert_rows_close(wn - wo, w - wo, 1e-4, "bag adagrad dw", ulp_of=wn)
        assert_untouched(ar.g2sum, g2_before, uniq)
    assert_untouched(state, before, uniq)


# ------------------------------------------------------------------ dense Adam


def test_dense_adam_three_waves(cuda_dev):
    """rs_dense_adam over 3 waves plus an odd tail, two steps from non-zero moments, with the bf16 shadow: every
    element's m, v and dw against fp64 Adam, bounded by the size of the terms it sums; the shadow is w rounded."""
    from oracle import oracle_np as onp
    from recommendsystem_b200 import ops
    rng = np.random.default_rng(8)
    n = 3 * dense_adam_wave() + 4321
    w = rng.standard_normal(n).astype(np.float32)
    m = (rng.standard_normal(n) * 0.01).astype(np.float32)
    v = (rng.random(n) * 0.01 + 1e-4).astype(np.float32)
    wt, mt, vt = _t(w, cuda_dev), _t(m, cuda_dev), _t(v, cuda_dev)
    shadow = torch.empty(n, dtype=torch.bfloat16, device=cuda_dev)
    scal = torch.zeros(4, device=cuda_dev)
    lr = 1e-3
    f32 = np.finfo(np.float32).eps
    for step in (1, 2):
        g = rng.standard_normal(n).astype(np.float32)
        ops.adam_advance(scal, B1, B2)
        ops.dense_adam(wt, mt, vt, _t(g, cuda_dev), lr, B1, B2, EPS, scal, shadow)
        corr = float(onp.adam_scalars(step, B1, B2)[2])
        w64, m64, v64, g64 = (a.astype(np.float64) for a in (w, m, v, g))
        w2, m2, v2 = onp.dense_adam(w64, m64, v64, g64, lr, B1, B2, EPS, corr)
        wn, mn, vn = wt.cpu().numpy(), mt.cpu().numpy(), vt.cpu().numpy()
        mag_m = np.abs(B1 * m64) + np.abs((1 - B1) * g64)
        mag_v = B2 * v64 + (1 - B2) * g64 * g64
        assert (np.abs(mn - m2) <= 4 * f32 * mag_m).all(), "dense adam m"
        assert (np.abs(vn - v2) <= 4 * f32 * mag_v).all(), "dense adam v"
        bound = 16 * f32 * lr * corr * mag_m / (np.sqrt(v2) + EPS) + 2 * np.spacing(np.abs(wn))
        assert (np.abs((wn - w64) - (w2 - w64)) <= bound).all(), "dense adam dw"
        assert torch.equal(shadow, wt.to(torch.bfloat16))
        w, m, v = wn, mn, vn
