"""torch.autograd.Function wrappers around the C-ABI kernels (forward AND backward are CUDA
kernels from librs_b200.so; nothing here falls back to eager PyTorch math for the hot ops)."""
from __future__ import annotations

import torch

from .. import cabi, ops


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("recommendsystem_b200 layers need CUDA tensors (no CPU fallback)")


class InteractingFn(torch.autograd.Function):
    """InteractingLayer.call (InteractingLayer.py:37-61) fused forward / backward."""

    @staticmethod
    def forward(ctx, x, Wqkvr, bqkvr, gamma, beta, ln_eps, H, L, use_res, dropout_rate=0.0, dropout_seed=0,
                dropout_step=None):
        _require_cuda(x, Wqkvr)
        x = x.contiguous()
        # bf16 activations take the tcgen05 kernels where they are built (falls back to FFMA arithmetic otherwise)
        ctx.tc = x.dtype == torch.bfloat16
        y, saved = ops.interacting_fwd(x, Wqkvr, bqkvr, gamma, beta, ln_eps, H, L, use_res, compute_bf16=ctx.tc,
                                       dropout_rate=dropout_rate, dropout_seed=dropout_seed, dropout_step=dropout_step)
        ctx.save_for_backward(x, saved if saved is not None else x.new_empty(0), Wqkvr, bqkvr, gamma, beta)
        ctx.cfg = (ln_eps, H, L, use_res, dropout_rate, dropout_seed)
        ctx.dropout_step = dropout_step          # device counter: the backward of THIS step reads the same value
        return y

    @staticmethod
    def backward(ctx, dy):
        x, saved, Wqkvr, bqkvr, gamma, beta = ctx.saved_tensors
        ln_eps, H, L, use_res, rate, seed = ctx.cfg
        dx, dW, db, dg, dbt = ops.interacting_bwd(x, saved if saved.numel() else None, Wqkvr, bqkvr, gamma, beta,
                                                  ln_eps, H, L, dy.contiguous().to(x.dtype), use_res,
                                                  compute_bf16=ctx.tc, dropout_rate=rate, dropout_seed=seed,
                                                  dropout_step=ctx.dropout_step)
        return dx, dW, db, dg, dbt, None, None, None, None, None, None, None


class CrossFn(torch.autograd.Function):
    """DCN-v1 cross network (CrossNet.call rough_rank/layer.py:256-264; DeepCrossLayer.call staytime/layer.py:66-72):
    W, b are the L per-layer kernels / biases stacked as fp32 [L, dim]."""

    @staticmethod
    def forward(ctx, x, W, b):
        _require_cuda(x, W, b)
        if x.stride(-1) != 1:
            x = x.contiguous()
        W, b = W.contiguous(), b.contiguous()
        ctx.save_for_backward(x, W, b)
        return ops.cross_fwd(x, W, b)

    @staticmethod
    def backward(ctx, dout):
        x, W, b = ctx.saved_tensors
        if dout.stride(-1) != 1 or dout.dtype != x.dtype:
            dout = dout.contiguous().to(x.dtype)
        dx, dW, db = ops.cross_bwd(x, dout, W, b)
        return dx, dW, db


class DinFn(torch.autograd.Function):
    """DIN attention unit, mode A (din.py) or B (staytime/layer.py)."""

    @staticmethod
    def forward(ctx, mode, q, keys, values, seq_len, mask, W1, b1, W2, b2):
        _require_cuda(q, keys)
        if keys.dtype != q.dtype or (values is not None and values.dtype != q.dtype):
            raise ValueError(f"DIN: q, keys and values must share one dtype (got {q.dtype}, {keys.dtype}, "
                             f"{None if values is None else values.dtype})")
        q = q.contiguous()
        # the kernels address row (b, t) of keys and values at (b*T + t) * kv_ld: a view laid out otherwise (a T-slice
        # of a longer sequence, an expanded tensor) is copied, and both are copied when their row strides differ
        if not ops.din_rows_at(keys, ops.din_kv_ld(keys)):
            keys = keys.contiguous()
        if values is not None and not ops.din_rows_at(values, ops.din_kv_ld(keys)):
            values = values.contiguous()
            keys = keys.contiguous()
        out = ops.din_fwd(mode, q, keys, values, seq_len, mask, W1, b1.contiguous(), W2.contiguous(), b2.contiguous())
        ctx.mode = mode
        ctx.has_values = values is not None
        ctx.save_for_backward(q, keys, values if values is not None else q.new_empty(0),
                              seq_len if seq_len is not None else q.new_empty(0, dtype=torch.int32),
                              mask if mask is not None else q.new_empty(0, dtype=torch.uint8), W1, b1, W2, b2)
        return out

    @staticmethod
    def backward(ctx, dout):
        q, keys, values, seq_len, mask, W1, b1, W2, b2 = ctx.saved_tensors
        values = values if ctx.has_values else None
        seq_len = seq_len if seq_len.numel() else None
        mask = mask if mask.numel() else None
        dq, dkeys, dvalues, dW1, db1, dW2, db2 = ops.din_bwd(ctx.mode, q, keys, values, seq_len, mask, W1,
                                                             b1.contiguous(), W2.contiguous(), b2.contiguous(),
                                                             dout.contiguous().to(q.dtype))
        return None, dq, dkeys, (dvalues if ctx.has_values else None), None, None, dW1, db1, dW2, db2


_ACT_EPI = {None: cabi.EPI_BIAS, "linear": cabi.EPI_BIAS, "relu": cabi.EPI_BIAS_RELU, "sigmoid": cabi.EPI_BIAS_SIGMOID}


class DenseFn(torch.autograd.Function):
    """y = act(x @ kernel[in,out] + bias) (tf.keras.layers.Dense / DNN.call, rough_rank/layer.py:100-109).
    fp32 tensors -> FFMA parity kernel; bf16 activations -> tcgen05 kernel (weights cast to bf16 shadows,
    fp32 master weights and fp32 weight gradients)."""

    @staticmethod
    def forward(ctx, x, kernel, bias, act):
        _require_cuda(x, kernel)
        lead = x.shape[:-1]
        x2 = x.reshape(-1, x.shape[-1])
        if x2.stride(-1) != 1:
            x2 = x2.contiguous()
        epi = _ACT_EPI[act]
        K, N = kernel.shape
        # the tensor-core kernel needs 16-byte TMA strides; narrow layers (heads, gates) use the fp32 kernel
        ctx.tc = x2.dtype == torch.bfloat16 and K % 8 == 0 and N % 8 == 0
        ctx.in_dtype = x2.dtype
        if x2.dtype == torch.bfloat16 and not ctx.tc:
            x2 = x2.float()
        ctx.pad = None
        if ctx.tc:
            wt = ops.transpose2d(kernel.to(torch.bfloat16).contiguous())          # [out,in] K-major
            y = ops.gemm(x2, wt, bias=bias, epilogue=epi, transB=True)
        else:
            # fp32: the 3xTF32 tensor-core GEMM needs 16-byte TMA rows (in / out multiples of 4, >= 8).  Narrow or odd
            # layers (SENet 1456 -> 22 -> 91, gates -> 3, heads -> 1) are zero-padded to the next such shape instead of
            # dropping to the FFMA kernel: the padded columns / rows are exact zeros and are sliced away again.
            M = x2.shape[0]
            Kp, Np = max(8, (K + 3) // 4 * 4), max(8, (N + 3) // 4 * 4)
            if (Kp != K or Np != N) and M * Kp * Np >= (1 << 20):
                ctx.pad = (K, N, Kp, Np)
                wp = torch.zeros(Kp, Np, dtype=kernel.dtype, device=kernel.device)
                wp[:K, :N] = kernel
                bp = torch.zeros(Np, dtype=bias.dtype, device=bias.device)
                bp[:N] = bias
                if Kp != K:
                    xp = torch.zeros(M, Kp, dtype=x2.dtype, device=x2.device)
                    xp[:, :K] = x2
                    x2 = xp
                y = ops.gemm(x2, wp, bias=bp, epilogue=epi)
                ctx.act = act
                ctx.save_for_backward(x2, wp, y)
                ctx.lead = lead
                return y[:, :N].reshape(*lead, N).to(ctx.in_dtype)
            y = ops.gemm(x2, kernel.contiguous(), bias=bias, epilogue=epi)
        ctx.act = act
        ctx.save_for_backward(x2, kernel, y)
        ctx.lead = lead
        return y.reshape(*lead, kernel.shape[1]).to(ctx.in_dtype)

    @staticmethod
    def backward(ctx, dy):
        x2, kernel, y = ctx.saved_tensors
        dy2 = dy.reshape(-1, dy.shape[-1]).to(y.dtype)
        if ctx.pad is not None:
            K, N, Kp, Np = ctx.pad                                               # padded fp32 layer (see forward)
            dyp = torch.zeros(dy2.shape[0], Np, dtype=y.dtype, device=y.device)
            dyp[:, :N] = dy2
            if ctx.act == "relu":
                dyp = ops.act_bwd(dyp, y, 0)
            elif ctx.act == "sigmoid":
                dyp = ops.act_bwd(dyp, y, 1)
            db = ops.colsum(dyp)[:N]
            dx = ops.gemm(dyp, kernel, transB=True)[:, :K] if ctx.needs_input_grad[0] else None
            dW = ops.gemm(x2, dyp, transA=True)[:K, :N]
            dx = dx.reshape(*ctx.lead, K).to(ctx.in_dtype) if dx is not None else None
            return dx, dW.contiguous(), db.contiguous(), None
        if dy2.stride(-1) != 1:
            dy2 = dy2.contiguous()
        if ctx.act == "relu":
            dy2 = ops.act_bwd(dy2, y, 0)
        elif ctx.act == "sigmoid":
            dy2 = ops.act_bwd(dy2, y, 1)
        db = ops.colsum(dy2)
        if ctx.tc:
            w16 = kernel.to(torch.bfloat16).contiguous()                         # [in,out]: K-major B for dgrad
            dx = ops.gemm(dy2, w16, transB=True) if ctx.needs_input_grad[0] else None
            if dy2.shape[1] > 32:
                # MN-major TMA/UMMA operands: x [B,in] and dy [B,out] are read as they lie
                dW = ops.gemm(x2, dy2, transA=True, out_dtype=torch.float32)
            else:
                M = x2.shape[0]
                Mp = (M + 7) // 8 * 8                                            # 16-byte rows for TMA
                xT = torch.zeros(x2.shape[1], Mp, dtype=x2.dtype, device=x2.device)
                dyT = torch.zeros(dy2.shape[1], Mp, dtype=x2.dtype, device=x2.device)
                ops.transpose2d(x2, xT[:, :M])
                ops.transpose2d(dy2, dyT[:, :M])
                dW = ops.gemm(xT[:, :M], dyT[:, :M], transB=True, out_dtype=torch.float32)
        else:
            dx = ops.gemm(dy2, kernel.contiguous(), transB=True) if ctx.needs_input_grad[0] else None
            dW = ops.gemm(x2, dy2, transA=True)
        dx = dx.reshape(*ctx.lead, kernel.shape[0]).to(ctx.in_dtype) if dx is not None else None
        return dx, dW.to(kernel.dtype), db.to(kernel.dtype), None


def dense(x, kernel, bias, activation=None):
    if activation == "softmax":
        return torch.softmax(DenseFn.apply(x, kernel, bias, None), dim=-1)
    if activation not in _ACT_EPI:
        raise ValueError(f"unsupported activation {activation!r}")
    return DenseFn.apply(x, kernel, bias, activation)
