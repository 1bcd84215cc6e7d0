"""The AutoInt tower's part of the bf16 step at the headline size (B = 8192, 39 x 16 -> 256 -> 128, head over 752
columns): the fused launch (rs_tower_step) against the chain it replaces (4 GEMMs + the logit head pass) on the same
trainer buffers.  Each is captured as ten back-to-back launches in one CUDA graph and timed with CUDA events; the
working set (~55 MB) fits in L2, so the figures are for L2-warm operands.
usage: python tools/tower_bench.py [--batch 8192] [--reps 20]"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from recommendsystem_b200 import cabi, ops  # noqa: E402
from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer  # noqa: E402

PEAK_BF16 = 2.25e15      # dense BF16 FLOP/s, one B200 (data sheet, 1000 W)
PEAK_HBM = 7.7e12        # bytes/s


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def time_graph(fn, n=10, reps=20):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(n):
            fn()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / (reps * n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    B = args.batch
    cfg = AutoIntConfig(num_fields=39, rows_per_field=100_000, embed_dim=16, unit_num=16, head_num=2, layer_num=3,
                        mlp_hidden=(256, 128), batch=B, dtype="bf16")
    tr = AutoIntTrainer(cfg, "cuda:0")
    assert tr.fuse_tower
    g = torch.Generator(device="cpu").manual_seed(0)
    tr.ids.copy_(torch.randint(0, 2 ** 40, (B, 39), generator=g))
    tr.labels.copy_((torch.rand(B, 1, generator=g) < 0.25).float())
    tr.step(tr.ids, tr.labels)           # realistic X / Z[:, n_deep:] in the buffers
    torch.cuda.synchronize()
    P, G = tr.P, tr.G
    K0, N0, N1, Ki = 39 * 16, 256, 128, 39 * 16
    X = tr.X.view(B, K0)
    acts = [X, tr.H[0], tr.Z[:, :N1]]

    def fused():
        ops.tower_step(X, tr.WT16["mlp_W0"], tr.WT16["mlp_W1"], tr.P16["mlp_W0"], tr.P16["mlp_W1"], P["mlp_b0"],
                       P["mlp_b1"], P["out_W"], P["out_b"], tr.labels, tr.Z, tr.p_raw, tr.dZ, tr.H[0], tr.dH[0],
                       tr.dX.view(B, K0))
        # the head's dw / db / loss partials: the chain's logit_head writes them, the fused path reads Z once more
        ops.logit_head_grad(tr.Z, tr.p_raw, tr.labels, tr.head_ws)

    def chain():
        for i in range(2):
            ops.gemm(acts[i], tr.WT16[f"mlp_W{i}"], acts[i + 1], bias=P[f"mlp_b{i}"], epilogue=cabi.EPI_BIAS_RELU,
                     transB=True)
        ops.logit_head(tr.Z, P["out_W"], P["out_b"], tr.labels, tr.dZ, G["out_W"], G["out_b"], p_out=tr.p_raw,
                       loss=tr.loss, relu_cols=N1, ws=tr.head_ws, defer_reduce=True)
        ops.gemm(tr.dH[1], tr.P16["mlp_W1"], tr.dH[0], aux=tr.H[0], epilogue=cabi.EPI_MUL_RELU_MASK, transB=True)
        ops.gemm(tr.dH[0], tr.P16["mlp_W0"], tr.dX.view(B, K0), transB=True)

    flops = 2 * 2 * B * (K0 * N0 + N0 * N1) + 2 * B * Ki * 2
    zw = N1 + Ki
    # algorithmic bytes: X, Z[:, N1:] read; H0, Z[:, :N1], p, dZ, dH0, dX written (weights L2-resident); the operands are
    # L2-warm here, so the rate below is not an HBM rate, only set against the HBM peak for scale
    nbytes = 2 * (B * K0 + B * Ki + B * N0 + B * N1 + B + B * zw + B * N0 + B * K0)
    print(f"card: {card()}")
    print(f"tower at B={B}: {flops / 1e9:.2f} GFLOP, {nbytes / 1e6:.1f} MB algorithmic HBM traffic")
    def kernel_only():
        ops.tower_step(X, tr.WT16["mlp_W0"], tr.WT16["mlp_W1"], tr.P16["mlp_W0"], tr.P16["mlp_W1"], P["mlp_b0"],
                       P["mlp_b1"], P["out_W"], P["out_b"], tr.labels, tr.Z, tr.p_raw, tr.dZ, tr.H[0], tr.dH[0],
                       tr.dX.view(B, K0))

    for name, fn in (("tower_step alone", kernel_only), ("tower_step + head_grad", fused),
                     ("4 GEMMs + logit head", chain)):
        us = time_graph(fn, reps=args.reps)
        t = us * 1e-6
        print(f"  {name:22s} {us:7.1f} us   {flops / t / 1e12:6.1f} TFLOP/s ({flops / PEAK_BF16 / t * 100:4.1f} % of "
              f"bf16 peak)   {nbytes / t / 1e9:6.0f} GB/s L2-warm ({nbytes / PEAK_HBM / t * 100:4.1f} % of HBM peak)")


if __name__ == "__main__":
    main()
