"""GPU parity of the fused DIN unit at the benchmarked size and at its limits.

din_fwd_kernel / din_bwd_kernel are persistent: at most DIN_MAX_CTAS_PER_SM = 4 CTAs per SM of DIN_WARPS = 4 warps, one
sample per warp per trip (csrc/din.cu, din_grid).  The cfg3 cases are sized so that every warp takes at least three
samples at any occupancy, which is where the backward's per-warp parameter-gradient accumulators carry over from one
sample to the next.  Also: strided keys / values with a strided gradient layout, the longest sequence the backward's
shared memory holds, and the layouts the autograd wrapper has to copy.
"""

import numpy as np
import pytest

from util import REL_BF16, REL_F32, assert_close, glorot_uniform

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

DIN_WARPS, DIN_MAX_CTAS_PER_SM = 4, 4            # csrc/din.cu
# dW1 / db1 / dW2 / db2 are fp32 sums over B*T positions in both modes.  Measured on one NVIDIA B200 (1000 W power limit)
# at B = 8192, T = 100: the worst norm-wise error against fp64 was 1.6e-6 (db2, mode A, bf16 inputs), all others at most
# 6e-7; the bound leaves a 6x margin.
REL_DPARAMS = 1e-5
NAMES_A = ["dq", "dkeys", "dvalues", "dW1", "db1", "dW2", "db2"]
NAMES_B = ["dq", "dfacts", "dW1", "db1", "dW2", "db2"]
f64 = lambda a: np.asarray(a, np.float64)


def _sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _params(rng, nin, Hd=16):
    W1 = glorot_uniform(rng, nin, Hd)
    b1 = (0.1 * rng.standard_normal(Hd)).astype(np.float32)
    W2 = glorot_uniform(rng, Hd, 1)
    b2 = (0.1 * rng.standard_normal(1) + 0.2).astype(np.float32)
    return W1, b1, W2, b2


def _dev(a, dev, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return t.to(dtype) if dtype is not None else t


def _rounded(t):
    """fp64 host copy of a device tensor (bf16 inputs: the bf16 values the kernel reads)."""
    return t.float().cpu().numpy().astype(np.float64)


def _round(a, dtype):
    """The values a device tensor of `dtype` holds for the fp32 host array `a`."""
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(dtype).float().numpy()


def clear_relu_kinks(rng, q, keys, sl, W, dtype, tau=1e-4):
    """Mode A is piecewise linear: where a live hidden or score pre-activation is within fp32 rounding of 0, the fp32
    kernel and the fp64 reference may take different sides of the ReLU and a gradient jumps by O(1).  Redraw the key
    rows (host, fp32, in place) whose pre-activations lie within `tau` of a kink, evaluated on the values the kernel
    reads."""
    W1, b1, W2, b2 = (f64(w) for w in W)
    T = keys.shape[1]
    live = np.arange(T)[None, :] < sl[:, None]
    qr = f64(_round(q, dtype))[:, None, :]
    for _ in range(20):
        kr = f64(_round(keys, dtype))
        qt = np.broadcast_to(qr, kr.shape)
        h1 = np.concatenate([qt, kr, qt * kr], -1) @ W1 + b1
        s1 = (np.maximum(h1, 0) @ W2 + b2)[..., 0]
        bad = live & ((np.abs(h1) < tau).any(-1) | (np.abs(s1) < tau))
        if not bad.any():
            return
        keys[bad] = rng.standard_normal((int(bad.sum()), keys.shape[2])).astype(np.float32)
    raise AssertionError("could not clear the ReLU kinks")


def _inputs(rng, mode, B, T, H, dtype, dev):
    """Device inputs of one DIN call; W* stay fp32."""
    q = rng.standard_normal((B, H)).astype(np.float32)
    keys = rng.standard_normal((B, T, H)).astype(np.float32)
    dout = _dev(rng.standard_normal((B, H)).astype(np.float32), dev, dtype)
    Wh = _params(rng, (3 if mode == "A" else 4) * H)
    W = [_dev(a, dev) for a in Wh]
    if mode == "A":
        values = _dev(rng.standard_normal((B, T, H)).astype(np.float32), dev, dtype)
        sl = rng.integers(0, T + 1, size=B).astype(np.int32)
        sl[0] = T
        clear_relu_kinks(rng, q, keys, sl, Wh, dtype)
        return _dev(q, dev, dtype), _dev(keys, dev, dtype), values, _dev(sl, dev), None, W, dout
    lens = rng.integers(0, T + 1, size=B)
    lens[0] = 0                                       # all-masked sample
    mask = (np.arange(T)[None, :] < lens[:, None]).astype(np.uint8)
    return _dev(q, dev, dtype), _dev(keys, dev, dtype), None, None, _dev(mask, dev), W, dout


def _reference(mode, q, keys, values, sl, mask, W, dout):
    from oracle import oracle_np as onp
    Wh = [_rounded(w) for w in W]
    if mode == "A":
        a = (_rounded(q), _rounded(keys), _rounded(values), sl.cpu().numpy(), *Wh)
        return onp.din_a_fwd(*a), onp.din_a_bwd(*a, _rounded(dout))
    a = (_rounded(q), _rounded(keys), mask.cpu().numpy(), *Wh)
    return onp.din_b_fwd(*a), onp.din_b_bwd(*a, _rounded(dout))


def _check(mode, dtype, out, got, ref_out, refs, what, errs=None):
    """Activation outputs / gradients to REL_BF16 (bf16) or test_gpu_din.py's fp32 bounds; parameter gradients are fp32
    in both modes: REL_DPARAMS.  `errs` collects the measured norm-wise errors."""
    act_rel = REL_BF16 if dtype == torch.bfloat16 else (REL_F32 if mode == "A" else 2 * REL_F32)
    assert_close(out.float().cpu().numpy(), ref_out, REL_BF16 if dtype == torch.bfloat16 else REL_F32, what + " fwd")
    names = NAMES_A if mode == "A" else NAMES_B
    got = [g for g in got if g is not None]
    for g, r, name in zip(got, refs, names):
        g = g.float().cpu().numpy().reshape(r.shape)
        param = name in ("dW1", "db1", "dW2", "db2")
        if errs is not None:
            errs[name] = float(np.max(np.abs(g - r)) / np.max(np.abs(r)))
        # db2 of mode B is analytically 0 (softmax is shift invariant): absolute bound, as in test_gpu_din.py
        assert_close(g, r, REL_DPARAMS if param else act_rel, f"{what} {name}",
                     atol=1e-4 if (mode == "B" and name == "db2") else 0.0)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("mode", ["A", "B"])
def test_din_cfg3_shape(cuda_dev, mode, dtype):
    """B = 8192 (every warp takes >= 3 samples at any occupancy), T = 100, H = 16, forward and backward against fp64 on
    the inputs the kernel reads; the backward twice with identical bits."""
    from recommendsystem_b200 import cabi, ops
    B, T, H = 8192, 100, 16
    assert B >= 3 * _sm() * DIN_MAX_CTAS_PER_SM * DIN_WARPS
    rng = np.random.default_rng(3 + (mode == "B") + 2 * (dtype == torch.bfloat16))
    q, keys, values, sl, mask, W, dout = _inputs(rng, mode, B, T, H, dtype, cuda_dev)
    m = cabi.DIN_A if mode == "A" else cabi.DIN_B
    out = ops.din_fwd(m, q, keys, values, sl, mask, *W)
    got = ops.din_bwd(m, q, keys, values, sl, mask, *W, dout)
    ref_out, refs = _reference(mode, q, keys, values, sl, mask, W, dout)
    errs = {}
    _check(mode, dtype, out, got, ref_out, refs, f"din {mode} {dtype}", errs)
    print(f"din {mode} {dtype} B={B} T={T}: norm-wise errors " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert torch.equal(out, ops.din_fwd(m, q, keys, values, sl, mask, *W))
    got2 = ops.din_bwd(m, q, keys, values, sl, mask, *W, dout)
    assert all(torch.equal(a, b) for a, b in zip(got, got2) if a is not None)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("H", [16, 8])
def test_din_a_strided_kv_and_grads(cuda_dev, H, dtype):
    """Mode A with separate values: keys and values are the first H columns of [B, T, 2H] buffers (kv_ld = 2H), and
    rs_din_bwd writes dkeys / dvalues into [B, T, 2H] buffers (dkv_ld = 2H): the H columns match fp64, the other
    columns keep their bits."""
    from recommendsystem_b200 import cabi, ops
    B, T, ld = 4096, 100, 2 * H
    rng = np.random.default_rng(H + (dtype == torch.bfloat16))
    kh = rng.standard_normal((B, T, ld)).astype(np.float32)
    qh = rng.standard_normal((B, H)).astype(np.float32)
    sl = rng.integers(0, T + 1, size=B).astype(np.int32)
    sl[0] = T
    Wh = _params(rng, 3 * H)
    kcols = np.ascontiguousarray(kh[:, :, :H])
    clear_relu_kinks(rng, qh, kcols, sl, Wh, dtype)
    kh[:, :, :H] = kcols
    kbuf = _dev(kh, cuda_dev, dtype)
    vbuf = _dev(rng.standard_normal((B, T, ld)).astype(np.float32), cuda_dev, dtype)
    keys, values = kbuf[:, :, :H], vbuf[:, :, :H]
    q = _dev(qh, cuda_dev, dtype)
    dout = _dev(rng.standard_normal((B, H)).astype(np.float32), cuda_dev, dtype)
    sl = _dev(sl, cuda_dev)
    W = [_dev(a, cuda_dev) for a in Wh]
    out = ops.din_fwd(cabi.DIN_A, q, keys, values, sl, None, *W)
    dq = torch.empty_like(q)
    sentinel = torch.full((B, T, ld), -7.25, dtype=dtype, device=cuda_dev)
    dkeys, dvalues = sentinel.clone(), sentinel.clone()
    nparams = sum(w.numel() for w in W)
    dparams = torch.empty(nparams, device=cuda_dev)
    ws = torch.empty(cabi.load().rs_din_workspace_bytes(cabi.DIN_A, B, T, H, 16), dtype=torch.uint8, device=cuda_dev)
    cabi.call("rs_din_bwd", cabi.DIN_A, q.data_ptr(), keys.data_ptr(), values.data_ptr(), ld, ops._dt(q),
              sl.data_ptr(), None, *[w.data_ptr() for w in W], dout.data_ptr(), dq.data_ptr(), dkeys.data_ptr(),
              dvalues.data_ptr(), ld, dparams.data_ptr(), B, T, H, 16, ws.data_ptr(), ws.numel(), ops._stream())
    parts, o = [], 0
    for w in W:
        parts.append(dparams[o:o + w.numel()].view(w.shape))
        o += w.numel()
    assert torch.equal(dkeys[:, :, H:], sentinel[:, :, H:]) and torch.equal(dvalues[:, :, H:], sentinel[:, :, H:])
    ref_out, refs = _reference("A", q, keys, values, sl, None, W, dout)
    _check("A", dtype, out, [dq, dkeys[:, :, :H], dvalues[:, :, :H], *parts], ref_out, refs, f"din A strided H={H}")
    # the ops wrapper on the same strided views gives the same bits
    got = ops.din_bwd(cabi.DIN_A, q, keys, values, sl, None, *W, dout)
    assert torch.equal(got[0], dq) and torch.equal(got[1], dkeys[:, :, :H]) and torch.equal(got[2], dvalues[:, :, :H])
    assert all(torch.equal(a, b) for a, b in zip(got[3:], parts))


@pytest.mark.parametrize("mode", ["A", "B"])
@pytest.mark.parametrize("H,T_max", [(16, 448), (8, 512)])
def test_din_longest_sequence(cuda_dev, H, T_max, mode):
    """The longest T whose backward fits the shared-memory limit of din_bwd (200 KB per CTA: T <= 448 at H = 16,
    T <= 512 at H = 8; one CTA per SM, so each warp takes many samples) against fp64; one step past it the call is
    refused naming shared memory, before any kernel runs."""
    from recommendsystem_b200 import cabi, ops
    B = 1024
    rng = np.random.default_rng(T_max + (mode == "B"))
    q, keys, values, sl, mask, W, dout = _inputs(rng, mode, B, T_max, H, torch.float32, cuda_dev)
    m = cabi.DIN_A if mode == "A" else cabi.DIN_B
    out = ops.din_fwd(m, q, keys, values, sl, mask, *W)
    got = ops.din_bwd(m, q, keys, values, sl, mask, *W, dout)
    ref_out, refs = _reference(mode, q, keys, values, sl, mask, W, dout)
    _check(mode, torch.float32, out, got, ref_out, refs, f"din {mode} H={H} T={T_max}")
    q, keys, values, sl, mask, W, dout = _inputs(rng, mode, 4, T_max + 1, H, torch.float32, cuda_dev)
    with pytest.raises(cabi.RsError, match="shared memory"):
        ops.din_bwd(m, q, keys, values, sl, mask, *W, dout)


def _din_grads(mod, q, keys, values, sl):
    leaves = [q, keys, values]
    out = mod(q, keys, values, sl)
    out.backward(torch.ones_like(out) * 0.5 + torch.arange(out.numel(), device=out.device).view(out.shape) * 1e-3)
    grads = [t.grad.clone() for t in leaves] + [p.grad.clone() for p in mod.parameters()]
    for t in leaves + list(mod.parameters()):
        t.grad = None
    return out.detach(), grads


def test_din_module_values_layouts(cuda_dev):
    """api.din.DIN with values as a T-slice of a longer sequence, and as an expanded tensor, equals the same call on
    contiguous copies, forward and backward; the ops layer refuses those layouts instead of misreading them."""
    from recommendsystem_b200 import cabi, ops
    from recommendsystem_b200.api.din import DIN
    B, T, H, T_long = 64, 30, 16, 50
    g = torch.Generator(device=cuda_dev).manual_seed(0)
    mod = DIN()
    mod.build(H, cuda_dev)
    sl = torch.randint(1, T + 1, (B,), device=cuda_dev, generator=g, dtype=torch.int32)
    q = torch.randn(B, H, device=cuda_dev, generator=g).requires_grad_()
    keys = torch.randn(B, T, H, device=cuda_dev, generator=g).requires_grad_()
    seq = torch.randn(B, T_long, H, device=cuda_dev, generator=g)
    one = torch.randn(1, T, H, device=cuda_dev, generator=g)
    for name, view in (("T-slice", seq[:, :T]), ("expanded", one.expand(B, T, H))):
        assert not ops.din_rows_at(view, H)
        src = view.detach().clone().requires_grad_()            # same values, contiguous
        lay = view.detach().requires_grad_() if name == "T-slice" else one.clone().requires_grad_()
        vals = lay if name == "T-slice" else lay.expand(B, T, H)
        ref_out, ref_g = _din_grads(mod, q, keys, src, sl)
        out = mod(q, keys, vals, sl)
        assert torch.equal(out, ref_out), name
        out.backward(torch.ones_like(out) * 0.5 + torch.arange(out.numel(), device=out.device).view(out.shape) * 1e-3)
        dvals = lay.grad if name == "T-slice" else lay.grad[0]
        want = ref_g[2] if name == "T-slice" else ref_g[2].sum(0)
        assert torch.equal(q.grad, ref_g[0]) and torch.equal(keys.grad, ref_g[1]), name
        assert torch.allclose(dvals, want, rtol=1e-6, atol=1e-7), name
        for p, r in zip(mod.parameters(), ref_g[3:]):
            assert torch.equal(p.grad, r), name
        for t in [q, keys] + list(mod.parameters()):
            t.grad = None
        W = [mod.din_nn_0_kernel, mod.din_nn_0_bias, mod.din_nn_1_kernel, mod.din_nn_1_bias]
        with pytest.raises(ValueError, match="values"):
            ops.din_fwd(cabi.DIN_A, q.detach(), keys.detach(), view, sl, None, *W)
    # the T-slice as keys too (mode B: no values)
    from recommendsystem_b200.api.staytime_layer import DIN as DinB
    mb = DinB()
    mb.build(H, cuda_dev)
    fb = mb(q.detach(), seq[:, :T], None)
    assert torch.equal(fb, mb(q.detach(), seq[:, :T].contiguous(), None))
    # mixed dtypes and unaddressable masks / lengths are refused
    with pytest.raises(ValueError, match="dtype"):
        mod(q.detach().bfloat16(), keys.detach(), keys.detach(), sl)
    with pytest.raises(ValueError, match="dtype"):
        mod(q.detach(), keys.detach(), keys.detach().bfloat16(), sl)
    W = [mod.din_nn_0_kernel.detach(), mod.din_nn_0_bias.detach(), mod.din_nn_1_kernel.detach(),
         mod.din_nn_1_bias.detach()]
    with pytest.raises(ValueError, match="seq_len"):
        ops.din_fwd(cabi.DIN_A, q.detach(), keys.detach(), keys.detach(), sl.long(), None, *W)
    mask = torch.ones(B, T_long, dtype=torch.uint8, device=cuda_dev)[:, :T]
    Wb = [mb.layer_1_kernel.detach(), mb.layer_1_bias.detach(), mb.layer_2_kernel.detach(), mb.layer_2_bias.detach()]
    with pytest.raises(ValueError, match="mask"):
        ops.din_fwd(cabi.DIN_B, q.detach(), keys.detach(), None, None, mask, *Wb)
