"""Thin host-side wrappers: torch CUDA tensors in, C-ABI calls (include/rs_b200.h) on
torch's current stream out.  torch is used for device memory and streams only; every
kernel that runs here is a hand-written sm_100a kernel from librs_b200.so.  No CPU
or eager-PyTorch fallback exists: a non-CUDA tensor raises.
"""
from __future__ import annotations

import math

import torch

from . import cabi
from .cabi import RS_BF16, RS_F32, call

_DT = {torch.float32: RS_F32, torch.bfloat16: RS_BF16}


def _dt(t: torch.Tensor) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise TypeError(f"unsupported dtype {t.dtype} (float32 / bfloat16 only)") from None


def _ptr(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("recommendsystem_b200 kernels need CUDA tensors (no CPU fallback)")
    return t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _need(cond, msg):
    if not cond:
        raise ValueError(msg)


class _Workspace:
    """Scratch buffers keyed by (purpose, device, STREAM).  Two rules make them safe under captured multi-stream
    steps: (1) a buffer is never freed — when a larger request replaces it the old tensor is retired, not
    released, because an already captured CUDA graph may still hold its address; (2) every stream has its own
    buffer per purpose, so kernels that the step runs concurrently on the main and the side stream (split-K
    partials of a weight-gradient GEMM beside a dgrad GEMM) never share scratch."""

    def __init__(self):
        self.bufs = {}
        self.retired = []

    def get(self, key, nbytes, device):
        dev = torch.device(device)
        k = (key, dev, torch.cuda.current_stream(dev).cuda_stream)
        b = self.bufs.get(k)
        if b is None or b.numel() < nbytes:
            if b is not None:
                self.retired.append(b)
            b = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=dev)
            self.bufs[k] = b
        return b


WS = _Workspace()

# ----------------------------------------------------------------- embedding


def embed_gather(table, ids, row_base, rows, out_dtype=torch.float32, want_keys=False, want_rows=False):
    """ids int64 [..., F] -> out [..., F, d]; optional sort keys / arena rows."""
    _need(ids.dtype == torch.int64 and ids.is_contiguous(), "ids must be contiguous int64")
    _need(table.dtype == torch.float32 and table.dim() == 2 and table.stride(1) == 1,
          "table must be fp32 [R,d] with contiguous rows (a row stride > d is allowed)")
    F = ids.shape[-1]
    n, d = ids.numel(), table.shape[1]
    out = torch.empty(*ids.shape, d, dtype=out_dtype, device=table.device)
    keys = torch.empty(n, dtype=torch.int64, device=table.device) if want_keys else None
    rws = torch.empty(ids.shape, dtype=torch.int32, device=table.device) if want_rows else None
    call("rs_embed_gather_fwd_ld", _ptr(table), table.stride(0), _ptr(ids), _ptr(row_base), _ptr(rows), n, F, d,
         _ptr(out), _DT[out_dtype], _ptr(keys), _ptr(rws), _stream())
    return out, keys, rws


def embed_gather_peer(shards, ids, local_base, rows, out_dtype=torch.float32):
    """Row-sharded gather over (peer) shard pointers: shards[r] is rank r's [local_rows, d] fp32 table (a
    CUDA-IPC mapping in the multi-process trainer; plain local tensors in single-process tests)."""
    import ctypes
    W = len(shards)
    F = ids.shape[-1]
    n, d = ids.numel(), shards[0].shape[1]
    ptrs = (ctypes.c_void_p * W)(*[t.data_ptr() for t in shards])
    out = torch.empty(*ids.shape, d, dtype=out_dtype, device=ids.device)
    _need(all(t.stride(1) == 1 and t.stride(0) == shards[0].stride(0) for t in shards), "shards: one common row stride")
    call("rs_embed_gather_peer_fwd", ctypes.addressof(ptrs), shards[0].stride(0), W, _ptr(ids), _ptr(local_base),
         _ptr(rows), n, F, d, _ptr(out), _DT[out_dtype], _stream())
    return out


def embed_gather_rows(table, rowidx, out_dtype=torch.float32, want_mask=False, want_keys=False):
    _need(rowidx.dtype == torch.int32 and rowidx.is_contiguous(), "rowidx must be contiguous int32")
    n, d = rowidx.numel(), table.shape[1]
    out = torch.empty(*rowidx.shape, d, dtype=out_dtype, device=table.device)
    mask = torch.empty(rowidx.shape, dtype=torch.uint8, device=table.device) if want_mask else None
    keys = torch.empty(n, dtype=torch.int64, device=table.device) if want_keys else None
    call("rs_embed_gather_rows_ld", _ptr(table), table.stride(0), _ptr(rowidx), n, d, _ptr(out), _DT[out_dtype],
         _ptr(mask), _ptr(keys), _stream())
    return out, mask, keys


def embed_gather_bag_mean(table, ids, offsets, row_base, rows, F, out_dtype=torch.float32):
    n_bags, d = offsets.numel() - 1, table.shape[1]
    out = torch.empty(n_bags, d, dtype=out_dtype, device=table.device)
    call("rs_embed_gather_bag_mean", _ptr(table), _ptr(ids), _ptr(offsets), _ptr(row_base), _ptr(rows),
         n_bags, F, d, _ptr(out), _DT[out_dtype], _stream())
    return out


def row_bits(total_rows: int) -> int:
    return max(1, min(32, int(math.ceil(math.log2(total_rows + 1)))))


def sort_keys(keys, rbits=32, out=None):
    n = keys.numel()
    out = torch.empty_like(keys) if out is None else out
    nbytes = cabi.load().rs_embed_sort_workspace_bytes(n)
    ws = WS.get("sort", nbytes, keys.device)
    call("rs_embed_sort_keys", _ptr(keys), _ptr(out), n, rbits, _ptr(ws), ws.numel(), _stream())
    return out


def segsum(grad, keys_sorted):
    n, d = keys_sorted.numel(), grad.shape[-1]
    seg_rows = torch.empty(n, dtype=torch.int32, device=grad.device)
    seg_sum = torch.empty(n, d, dtype=torch.float32, device=grad.device)
    call("rs_embed_segsum", _ptr(grad), _dt(grad), _ptr(keys_sorted), n, d, _ptr(seg_rows), _ptr(seg_sum),
         _stream())
    return seg_rows, seg_sum


def segsum_adam(w, m, v, grad, keys_sorted, lr, beta1, beta2, eps, scalars, grad_scale=1.0):
    _need(w.stride(1) == 1 and w.stride() == m.stride() == v.stride(), "w, m, v: one common row stride")
    call("rs_embed_segsum_adam_ld", _ptr(w), _ptr(m), _ptr(v), w.stride(0), _ptr(grad), _dt(grad), _ptr(keys_sorted),
         keys_sorted.numel(), w.shape[1], lr, beta1, beta2, eps, _ptr(scalars), grad_scale, _stream())


def segsum_adagrad(w, g2sum, grad, keys_sorted, lr, eps, per_element=False, grad_scale=1.0):
    call("rs_embed_segsum_adagrad", _ptr(w), _ptr(g2sum), _ptr(grad), _dt(grad), _ptr(keys_sorted),
         keys_sorted.numel(), w.shape[1], lr, eps, int(per_element), grad_scale, _stream())


def adam_advance(scalars, beta1, beta2):
    call("rs_adam_advance", _ptr(scalars), beta1, beta2, _stream())


def dense_adam(w, m, v, g, lr, beta1, beta2, eps, scalars, shadow=None):
    call("rs_dense_adam", _ptr(w), _ptr(m), _ptr(v), _ptr(g), w.numel(), lr, beta1, beta2, eps,
         _ptr(scalars), _ptr(shadow), _stream())


def route_ids(ids, F, rows, local_base, world):
    n = ids.numel()
    dev = ids.device
    send_rows = torch.empty(n, dtype=torch.int32, device=dev)
    inverse = torch.empty(n, dtype=torch.int32, device=dev)
    counts = torch.empty(world, dtype=torch.int32, device=dev)
    offsets = torch.empty(world + 1, dtype=torch.int32, device=dev)
    nbytes = cabi.load().rs_route_workspace_bytes(n, world)
    ws = WS.get("route", nbytes, dev)
    call("rs_route_ids", _ptr(ids), n, F, _ptr(rows), _ptr(local_base), world, _ptr(send_rows),
         _ptr(inverse), _ptr(counts), _ptr(offsets), _ptr(ws), ws.numel(), _stream())
    return send_rows, inverse, counts, offsets


def route_ids_padded(ids, F, rows, local_base, world, capacity, send_rows=None, inverse=None, counts=None,
                     overflow=None, pad_spread=False):
    n = ids.numel()
    dev = ids.device
    send_rows = torch.empty(world * capacity, dtype=torch.int32, device=dev) if send_rows is None else send_rows
    inverse = torch.empty(n, dtype=torch.int32, device=dev) if inverse is None else inverse
    counts = torch.empty(world, dtype=torch.int32, device=dev) if counts is None else counts
    overflow = torch.zeros(1, dtype=torch.int32, device=dev) if overflow is None else overflow
    nbytes = cabi.load().rs_route_workspace_bytes(n, world) + (world + 1) * 4
    ws = WS.get("route", nbytes, dev)
    call("rs_route_ids_padded_spread" if pad_spread else "rs_route_ids_padded", _ptr(ids), n, F, _ptr(rows),
         _ptr(local_base), world, capacity, _ptr(send_rows),
         _ptr(inverse), _ptr(counts), _ptr(overflow), _ptr(ws), ws.numel(), _stream())
    return send_rows, inverse, counts, overflow


def idmap_insert(slots, key_of_row, counters, geom, ids, field_of_col, seed, scale, w, states=()):
    """rs_idmap_insert: new (field, id) keys of `ids` [..., F] get rows; their records are initialised.  `w` is an
    fp32 [R, d] view with contiguous rows; `states` up to two (fp32 view [R] or [R, k], initial value) pairs."""
    _need(ids.dtype == torch.int64 and ids.is_contiguous(), "ids must be contiguous int64")
    _need(w.dtype == torch.float32 and w.dim() == 2 and w.stride(1) == 1, "w must be fp32 [R, d] with contiguous rows")
    st = []
    for t, v in states:
        _need(t.dtype == torch.float32 and (t.dim() == 1 or t.stride(1) == 1), "optimizer state: fp32, contiguous rows")
        st += [_ptr(t), t.stride(0), 1 if t.dim() == 1 else t.shape[1], float(v)]
    st += [None, 0, 0, 0.0] * (2 - len(states))
    call("rs_idmap_insert", _ptr(slots), _ptr(key_of_row), _ptr(counters), _ptr(geom), geom.shape[0], _ptr(ids),
         ids.numel(), field_of_col.numel(), _ptr(field_of_col), int(seed) & 0xFFFFFFFFFFFFFFFF, float(scale), _ptr(w),
         w.stride(0), w.shape[1], *st, _stream())


def idmap_lookup(slots, counters, geom, ids, field_of_col, out=None, after_insert=False):
    """rs_idmap_lookup: int64 arena rows of `ids` [..., F] (-1: padding, unseen or overflowed)."""
    _need(ids.dtype == torch.int64 and ids.is_contiguous(), "ids must be contiguous int64")
    out = torch.empty(ids.shape, dtype=torch.int64, device=ids.device) if out is None else out
    call("rs_idmap_lookup", _ptr(slots), _ptr(counters), _ptr(geom), geom.shape[0], _ptr(ids), ids.numel(),
         field_of_col.numel(), _ptr(field_of_col), _ptr(out), int(after_insert), _stream())
    return out


def idmap_rebuild(slots, key_of_row, counters, geom, max_rows):
    call("rs_idmap_rebuild", _ptr(slots), slots.numel() // 2, _ptr(key_of_row), _ptr(counters), _ptr(geom),
         geom.shape[0], int(max_rows), _stream())


def idmap_count(show, rows):
    """rs_idmap_count: show[r] += 1 for every row r >= 0 of `rows` (int64, any shape)."""
    _need(rows.dtype == torch.int64 and rows.is_contiguous(), "rows must be contiguous int64")
    _need(show.dtype == torch.float32 and show.is_contiguous(), "show must be contiguous fp32")
    call("rs_idmap_count", _ptr(show), _ptr(rows), rows.numel(), _stream())


def idmap_evict(slots, key_of_row, counters, geom, show, evicted, threshold, decay, w, states=()):
    """rs_idmap_evict: decay the live rows' show, drop the keys below `threshold`, compact every field's live rows
    (w and the `states` views move with them, the arguments of idmap_insert), rebuild the slots."""
    _need(w.dtype == torch.float32 and w.dim() == 2 and w.stride(1) == 1, "w must be fp32 [R, d] with contiguous rows")
    st = []
    for t in states:
        _need(t.dtype == torch.float32 and (t.dim() == 1 or t.stride(1) == 1), "optimizer state: fp32, contiguous rows")
        st += [_ptr(t), t.stride(0), 1 if t.dim() == 1 else t.shape[1]]
    st += [None, 0, 0] * (2 - len(states))
    total = key_of_row.numel()
    nbytes = cabi.load().rs_idmap_evict_workspace_bytes(total)
    ws = torch.empty(int(nbytes), dtype=torch.uint8, device=show.device)
    call("rs_idmap_evict", _ptr(slots), slots.numel() // 2, _ptr(key_of_row), _ptr(counters), _ptr(geom),
         geom.shape[0], total, _ptr(show), float(threshold), float(decay), _ptr(w), w.stride(0), w.shape[1], *st,
         _ptr(evicted), _ptr(ws), ws.numel(), _stream())


def permute_rows(src, index, scatter=False, out=None):
    n, d = index.numel(), src.shape[-1]
    out = torch.empty(n, d, dtype=src.dtype, device=src.device) if out is None else out
    call("rs_permute_rows", _ptr(src), _ptr(out), _ptr(index), n, d, _dt(src), int(scatter), _stream())
    return out


# ------------------------------------------------------------- interacting


def interacting_path(F, D, U, H, dtype, compute_bf16, dropout_rate=0.0):
    """Which kernels rs_interacting_fwd/_bwd run for these arguments: cabi.PATH_TCGEN05 / PATH_FFMA / PATH_NONE."""
    dt = cabi.RS_BF16 if dtype == torch.bfloat16 else cabi.RS_F32
    return int(cabi.load().rs_interacting_path(F, D, U, H, dt, int(compute_bf16), float(dropout_rate)))


def interacting_saved(B, F, U, L, device):
    """rs_interacting_saved_bytes(B, F, U, L) bytes; returned as the [L, B*F, U] view of the activations (the
    per-head softmax statistics of the tensor-core kernels follow them in the same storage)."""
    n = L * B * F
    buf = torch.empty(n * (U + 4), dtype=torch.float32, device=device)
    assert buf.numel() * 4 == cabi.load().rs_interacting_saved_bytes(B, F, U, L)
    return buf[:n * U].view(L, B * F, U)


def interacting_fwd(x, Wqkvr, bqkvr, gamma, beta, ln_eps, H, L, use_res=True, save=True, compute_bf16=False,
                    dropout_rate=0.0, dropout_seed=0, dropout_step=None):
    B, F, D = x.shape
    U = Wqkvr.shape[1] // 4
    _need(x.is_contiguous(), "x must be contiguous")
    y = torch.empty(B, F, U, dtype=x.dtype, device=x.device)
    saved = interacting_saved(B, F, U, L, x.device) if save else None
    call("rs_interacting_fwd_dropout", _ptr(x), D, 0, _dt(x), _ptr(Wqkvr), _ptr(bqkvr), _ptr(gamma), _ptr(beta),
         ln_eps, _ptr(y), U, 0, _ptr(saved), B, F, D, U, H, L, int(use_res), int(compute_bf16),
         float(dropout_rate), int(dropout_seed) & 0xFFFFFFFFFFFFFFFF, _ptr(dropout_step), _stream())
    return y, saved


def interacting_bwd(x, saved, Wqkvr, bqkvr, gamma, beta, ln_eps, H, L, dy, use_res=True, compute_bf16=False,
                    dropout_rate=0.0, dropout_seed=0, dropout_step=None):
    B, F, D = x.shape
    U = Wqkvr.shape[1] // 4
    dx = torch.empty_like(x)
    dparams = torch.empty(D * 4 * U + 4 * U + 2 * U, dtype=torch.float32, device=x.device)
    nbytes = cabi.load().rs_interacting_workspace_bytes(B, F, D, U)
    ws = WS.get("interacting", nbytes, x.device)
    dy = dy.contiguous()
    call("rs_interacting_bwd_dropout", _ptr(x), D, 0, _ptr(saved), _dt(x), _ptr(Wqkvr), _ptr(bqkvr), _ptr(gamma),
         _ptr(beta), ln_eps, _ptr(dy), U, 0, _ptr(dx), D, 0, _ptr(dparams), B, F, D, U, H, L, int(use_res),
         int(compute_bf16), float(dropout_rate), int(dropout_seed) & 0xFFFFFFFFFFFFFFFF, _ptr(dropout_step), _ptr(ws),
         ws.numel(), _stream())
    nW = D * 4 * U
    return dx, dparams[:nW].view(D, 4 * U), dparams[nW:nW + 4 * U], dparams[nW + 4 * U:nW + 5 * U], dparams[nW + 5 * U:]


# --------------------------------------------------------------------- DIN


def din_rows_at(t, ld):
    """True when row (b, t) of the [B, T, H] view `t` lies at element (b*T + t) * ld of its storage: the only layout
    the DIN kernels address (keys, values and their gradients share one row stride `ld`)."""
    B, T = t.shape[0], t.shape[1]
    return t.stride(2) == 1 and (T == 1 or t.stride(1) == ld) and (B == 1 or t.stride(0) == T * ld)


def din_kv_ld(keys):
    """The row stride of a [B, T, H] keys view as the DIN kernels read it (kv_ld)."""
    B, T, H = keys.shape
    return keys.stride(1) if T > 1 else (keys.stride(0) if B > 1 else H)


def _din_check(mode, q, keys, values, seq_len, mask, W1, b1, W2, b2, kv_ld):
    _need(q.dim() == 2 and q.is_contiguous(), "din: q must be a contiguous [B, H] tensor")
    B, H = q.shape
    _need(keys.dim() == 3 and keys.shape[0] == B and keys.shape[2] == H, "din: keys must be [B, T, H]")
    _need(keys.dtype == q.dtype, f"din: keys dtype {keys.dtype} differs from q dtype {q.dtype}")
    _need(din_rows_at(keys, kv_ld), f"din: keys rows must lie at (b*T + t) * {kv_ld} (strides {keys.stride()})")
    if values is not None:
        _need(values.shape == keys.shape, "din: values must have the shape of keys")
        _need(values.dtype == q.dtype, f"din: values dtype {values.dtype} differs from q dtype {q.dtype}")
        _need(din_rows_at(values, kv_ld),
              f"din: values rows must lie at (b*T + t) * {kv_ld}, as keys' (strides {values.stride()})")
    if seq_len is not None:
        _need(seq_len.dtype == torch.int32 and seq_len.is_contiguous() and seq_len.numel() == B,
              "din: seq_len must be contiguous int32 [B]")
    if mask is not None:
        _need(mask.dtype in (torch.uint8, torch.bool) and mask.is_contiguous() and mask.numel() == B * keys.shape[1],
              "din: mask must be contiguous uint8 [B, T]")
    for w in (W1, b1, W2, b2):
        _need(w.dtype == torch.float32 and w.is_contiguous(), "din: W1, b1, W2, b2 must be contiguous fp32")


def din_fwd(mode, q, keys, values, seq_len, mask, W1, b1, W2, b2, kv_ld=None):
    B, T = keys.shape[0], keys.shape[1]
    H = q.shape[1]
    Hd = W1.shape[1]
    kv_ld = kv_ld or din_kv_ld(keys)
    _din_check(mode, q, keys, values, seq_len, mask, W1, b1, W2, b2, kv_ld)
    out = torch.empty(B, H, dtype=q.dtype, device=q.device)
    call("rs_din_fwd", mode, _ptr(q), _ptr(keys), _ptr(values), kv_ld, _dt(q), _ptr(seq_len), _ptr(mask),
         _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), _ptr(out), B, T, H, Hd, _stream())
    return out


def din_bwd(mode, q, keys, values, seq_len, mask, W1, b1, W2, b2, dout, kv_ld=None):
    B, T = keys.shape[0], keys.shape[1]
    H = q.shape[1]
    Hd = W1.shape[1]
    kv_ld = kv_ld or din_kv_ld(keys)
    _din_check(mode, q, keys, values, seq_len, mask, W1, b1, W2, b2, kv_ld)
    _need(dout.shape == q.shape and dout.dtype == q.dtype, "din: dout must be [B, H] of q's dtype")
    dq = torch.empty_like(q)
    dkeys = torch.empty(B, T, H, dtype=q.dtype, device=q.device)
    dvalues = torch.empty(B, T, H, dtype=q.dtype, device=q.device) if mode == cabi.DIN_A else None
    nparams = W1.numel() + b1.numel() + W2.numel() + b2.numel()
    dparams = torch.empty(nparams, dtype=torch.float32, device=q.device)
    nbytes = cabi.load().rs_din_workspace_bytes(mode, B, T, H, Hd)
    ws = WS.get("din", nbytes, q.device)
    call("rs_din_bwd", mode, _ptr(q), _ptr(keys), _ptr(values), kv_ld, _dt(q), _ptr(seq_len), _ptr(mask),
         _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), _ptr(dout.contiguous()), _ptr(dq), _ptr(dkeys),
         _ptr(dvalues), H, _ptr(dparams), B, T, H, Hd, _ptr(ws), ws.numel(), _stream())
    o = 0
    parts = []
    for t in (W1, b1, W2, b2):
        parts.append(dparams[o:o + t.numel()].view(t.shape))
        o += t.numel()
    return (dq, dkeys, dvalues, *parts)


# -------------------------------------------------------------------- GEMM


def gemm(A, B, C=None, bias=None, aux=None, epilogue=cabi.EPI_NONE, transA=False, transB=False,
         out_dtype=None):
    """C[M,N] = epi(op(A) @ op(B)).  A, B are 2-D views whose last dim is contiguous."""
    _need(A.dim() == 2 and B.dim() == 2 and A.stride(1) == 1 and B.stride(1) == 1, "gemm: 2-D row-major views")
    M, K = (A.shape[1], A.shape[0]) if transA else A.shape
    K2, N = (B.shape[1], B.shape[0]) if transB else B.shape
    _need(K == K2, f"gemm: inner dims {K} vs {K2}")
    _need(A.dtype == B.dtype, "gemm: A/B dtype mismatch")
    if C is None:
        C = torch.empty(M, N, dtype=out_dtype or A.dtype, device=A.device)
    _need(C.stride(1) == 1, "gemm: C last dim must be contiguous")
    ws = WS.get("gemm", cabi.load().rs_gemm_workspace_bytes(), A.device)
    call("rs_gemm", _ptr(A), A.stride(0), int(transA), _ptr(B), B.stride(0), int(transB), _ptr(C), C.stride(0),
         _ptr(bias), _ptr(aux), aux.stride(0) if aux is not None else 0, epilogue, M, N, K, _dt(A), _dt(C),
         _ptr(ws), ws.numel(), _stream())
    return C


def transpose2d(src, out=None):
    _need(src.dim() == 2 and src.stride(1) == 1, "transpose2d: 2-D row-major view")
    M, N = src.shape
    out = torch.empty(N, M, dtype=src.dtype, device=src.device) if out is None else out
    call("rs_transpose2d", _ptr(src), src.stride(0), _ptr(out), out.stride(0), M, N, _dt(src), _stream())
    return out


def logit_head_workspace(B, zw, device):
    """A caller-owned partial-sum buffer for logit_head(..., ws=, defer_reduce=True) + logit_head_reduce."""
    return torch.empty(cabi.load().rs_logit_head_workspace_bytes(B, zw), dtype=torch.uint8, device=device)


def logit_head(Z, w, bias, y, dZ, dw, db, p_out=None, loss=None, a=1.0, relu_cols=0, ws=None, defer_reduce=False):
    """Fused Dense(1, sigmoid) + clip + BCE + head backward (rs_logit_head_fwd_bwd[_relu]); dZ[:, :relu_cols] comes
    out multiplied by relu'(Z).  defer_reduce: dw / db / loss are NOT written; the partial sums stay in `ws` (caller
    owned) for logit_head_reduce, which may run on another stream."""
    B, zw = Z.shape
    p_out = torch.empty(B, 1, dtype=Z.dtype, device=Z.device) if p_out is None else p_out
    loss = torch.empty(1, dtype=torch.float32, device=Z.device) if loss is None else loss
    _need(not defer_reduce or ws is not None, "logit_head: defer_reduce needs a caller-owned workspace")
    if ws is None:
        ws = WS.get("head", cabi.load().rs_logit_head_workspace_bytes(B, zw), Z.device)
    call("rs_logit_head_fwd_bwd_relu", _ptr(Z), Z.stride(0), _dt(Z), _ptr(w), _ptr(bias), _ptr(y), a, _ptr(p_out),
         _ptr(loss), _ptr(dZ), dZ.stride(0), None if defer_reduce else _ptr(dw), _ptr(db), B, zw, int(relu_cols),
         _ptr(ws), ws.numel(), _stream())
    return p_out, loss


def logit_head_reduce(ws, dw, db, loss, B, zw):
    """Sums the head's per-CTA partials (logit_head(..., defer_reduce=True)) into dw / db / loss on the current stream."""
    call("rs_logit_head_reduce", _ptr(ws), ws.numel(), _ptr(dw), _ptr(db), _ptr(loss), B, zw, _stream())


def logit_head_grad(Z, p, y, ws, a=1.0):
    """The head's dw / db / loss partials (left in `ws` for logit_head_reduce) from a p computed by tower_step."""
    B, zw = Z.shape
    call("rs_logit_head_grad", _ptr(Z), Z.stride(0), _dt(Z), _ptr(p), _ptr(y), a, B, zw, _ptr(ws), ws.numel(), _stream())


def tower_supported(K0, N0, N1, Ki) -> bool:
    return bool(cabi.load().rs_tower_supported(K0, N0, N1, Ki))


def tower_step(X, W0T, W1T, W0, W1, b0, b1, w, ob, y, Z, p_out, dZ, H0, dH0, dX, a=1.0):
    """The tower's part of the bf16 train step in one launch (rs_tower_step): H0, Z[:, :N1], p_out, dZ, dH0 and dX
    (stored, not accumulated) from X [B, K0] and Z[:, N1:]."""
    B, K0 = X.shape
    N0, N1 = W0T.shape[0], W1T.shape[0]
    Ki = Z.shape[1] - N1
    for t in (X, W0T, W1T, W0, W1, Z, dZ, H0, dH0, dX):
        _need(t.dtype == torch.bfloat16 and t.is_contiguous(), "tower_step: contiguous bf16 operands")
    call("rs_tower_step", _ptr(X), _ptr(W0T), _ptr(W1T), _ptr(W0), _ptr(W1), _ptr(b0), _ptr(b1), _ptr(w), _ptr(ob),
         _ptr(y), a, _ptr(Z), _ptr(p_out), _ptr(dZ), _ptr(H0), _ptr(dH0), _ptr(dX), B, K0, N0, N1, Ki, _stream())


def tower_fwd(X, W0T, W1T, W0, W1, b0, b1, w, ob, Z, p_out):
    """The forward half of tower_step (rs_tower_fwd): p_out from X [B, K0] and Z[:, N1:], bit-identical to the p_out
    tower_step writes; nothing else is written."""
    B, K0 = X.shape
    N0, N1 = W0T.shape[0], W1T.shape[0]
    Ki = Z.shape[1] - N1
    for t in (X, W0T, W1T, W0, W1, Z):
        _need(t.dtype == torch.bfloat16 and t.is_contiguous(), "tower_fwd: contiguous bf16 operands")
    _need(p_out.dtype == torch.bfloat16 and p_out.numel() == B, "tower_fwd: p_out must be bf16 [B]")
    call("rs_tower_fwd", _ptr(X), _ptr(W0T), _ptr(W1T), _ptr(W0), _ptr(W1), _ptr(b0), _ptr(b1), _ptr(w), _ptr(ob),
         _ptr(Z), _ptr(p_out), B, K0, N0, N1, Ki, _stream())


def colsum(x, out=None):
    _need(x.dim() == 2 and x.stride(1) == 1, "colsum: 2-D row-major view")
    M, N = x.shape
    out = torch.empty(N, dtype=torch.float32, device=x.device) if out is None else out
    nbytes = cabi.load().rs_colsum_workspace_bytes(M, N)
    ws = WS.get("colsum", nbytes, x.device)
    call("rs_colsum", _ptr(x), x.stride(0), _dt(x), _ptr(out), M, N, _ptr(ws), ws.numel(), _stream())
    return out


def act_bwd(g, ref, kind, out=None):
    M, N = g.shape
    out = torch.empty(M, N, dtype=g.dtype, device=g.device) if out is None else out
    call("rs_act_bwd", _ptr(g), g.stride(0), _ptr(ref), ref.stride(0), _ptr(out), out.stride(0), M, N, _dt(g),
         kind, _stream())
    return out


def copy2d(src, dst):
    M, N = src.shape
    call("rs_copy2d", _ptr(src), src.stride(0), _dt(src), _ptr(dst), dst.stride(0), _dt(dst), M, N, _stream())
    return dst


def add2d(a, b, out):
    M, N = a.shape
    call("rs_add2d", _ptr(a), a.stride(0), _ptr(b), b.stride(0), _ptr(out), out.stride(0), M, N, _dt(a), _stream())
    return out


def bce_sigmoid_fwd_bwd(p_raw, y, a=1.0, want_grad=True, loss=None):
    B, k = p_raw.shape
    loss = torch.empty(1, dtype=torch.float32, device=p_raw.device) if loss is None else loss
    dz = torch.empty_like(p_raw) if want_grad else None
    call("rs_bce_sigmoid_fwd_bwd", _ptr(p_raw), _dt(p_raw), _ptr(y), a, _ptr(loss), _ptr(dz), B, k, _stream())
    return loss, dz


# ------------------------------------------------------- labels and metrics
def staytime_labels(watch_ms, bins, landing=None, short_ms=7000, long_ms=18000, cap_s=160.0, sigma=4.0,
                    left=-19.0, right=180.5, landing_weight=5.0, want_weight=True):
    """rs_staytime_labels (staytime/parse.py:30-68): int64 watch durations [B] (ms) ->
    (staytime_label [B, nbins+1] fp32, short_label [B] int64, long_label [B] int64, sample_weight [B,1] | None)."""
    _need(watch_ms.dtype == torch.int64 and watch_ms.dim() == 1, "staytime_labels: watch_ms must be int64 [B]")
    _need(bins.dtype == torch.float32 and bins.dim() == 1 and bins.is_contiguous(), "staytime_labels: bins fp32 [nbins]")
    if landing is not None:
        _need(landing.dtype in (torch.uint8, torch.bool) and landing.shape == watch_ms.shape,
              "staytime_labels: landing must be uint8/bool [B]")
        landing = landing.view(torch.uint8) if landing.dtype == torch.bool else landing
    B, nb = watch_ms.numel(), bins.numel()
    dev = watch_ms.device
    label = torch.empty(B, nb + 1, dtype=torch.float32, device=dev)
    short = torch.empty(B, dtype=torch.int64, device=dev)
    long_ = torch.empty(B, dtype=torch.int64, device=dev)
    weight = torch.empty(B, 1, dtype=torch.float32, device=dev) if want_weight else None
    call("rs_staytime_labels", _ptr(watch_ms.contiguous()), _ptr(landing), _ptr(bins), nb, B, _ptr(label), _ptr(short),
         _ptr(long_), _ptr(weight), int(short_ms), int(long_ms), float(cap_s), float(sigma), float(left), float(right),
         float(landing_weight), _stream())
    return label, short, long_, weight


def binary_metrics_state(num_thresholds, device):
    n = cabi.load().rs_binary_metrics_state_bytes(int(num_thresholds))
    return torch.zeros(n // 8, dtype=torch.int64, device=device)


def binary_metrics_update(state, pred, label, thresholds, acc_threshold=0.5):
    """Accumulate one batch into `state` (rs_binary_metrics_update).  pred fp32 / bf16, label fp32, same numel."""
    _need(pred.numel() == label.numel(), "binary_metrics: pred and label sizes differ")
    _need(label.dtype == torch.float32, "binary_metrics: label must be float32")
    pred, label = pred.contiguous(), label.contiguous()
    n, T = pred.numel(), thresholds.numel()
    nbytes = cabi.load().rs_binary_metrics_workspace_bytes(n)
    ws = WS.get("binary_metrics", nbytes, pred.device)
    call("rs_binary_metrics_update", _ptr(pred), _dt(pred), _ptr(label), n, _ptr(thresholds), T, float(acc_threshold),
         _ptr(state), _ptr(ws), ws.numel(), _stream())


def binary_metrics_result(state, num_thresholds, out=None):
    """-> float64[6] on the device: AUC, accuracy, CTR, COPC, n, mean prediction (rs_binary_metrics_result)."""
    out = torch.empty(6, dtype=torch.float64, device=state.device) if out is None else out
    call("rs_binary_metrics_result", _ptr(state), int(num_thresholds), _ptr(out), _stream())
    return out


# ------------------------------------------------------------ cross network


def cross_fwd(x, W, b):
    """DCN-v1 cross layers x_{l+1} = x0 (x_l . w_l) + b_l + x_l (rough_rank/layer.py:256-264, staytime/layer.py:66-72).
    x [B, dim] (fp32 / bf16, row stride allowed), W, b fp32 [L, dim]."""
    _need(x.dim() == 2 and x.stride(1) == 1, "cross: x must be [B, dim] with contiguous rows")
    B, dim = x.shape
    L = W.shape[0]
    out = torch.empty(B, dim, dtype=x.dtype, device=x.device)
    ws = WS.get("cross", cabi.load().rs_cross_workspace_bytes(B, dim, L), x.device)
    call("rs_cross_fwd", _ptr(x), x.stride(0), _dt(x), _ptr(W), _ptr(b), _ptr(out), dim, B, dim, L, _ptr(ws), ws.numel(),
         _stream())
    return out


def cross_bwd(x, dout, W, b):
    _need(x.stride(1) == 1 and dout.stride(1) == 1, "cross: contiguous rows")
    B, dim = x.shape
    L = W.shape[0]
    dx = torch.empty(B, dim, dtype=x.dtype, device=x.device)
    dW = torch.empty(L, dim, dtype=torch.float32, device=x.device)
    db = torch.empty(L, dim, dtype=torch.float32, device=x.device)
    ws = WS.get("cross", cabi.load().rs_cross_workspace_bytes(B, dim, L), x.device)
    call("rs_cross_bwd", _ptr(x), x.stride(0), _ptr(dout), dout.stride(0), _dt(x), _ptr(W), _ptr(b), _ptr(dx), dim,
         _ptr(dW), _ptr(db), B, dim, L, _ptr(ws), ws.numel(), _stream())
    return dx, dW, db
