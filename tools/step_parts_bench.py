"""Developer tool (1 GPU): the non-InteractingLayer kernels of the AutoInt bench step, each timed alone inside a CUDA
graph (10 launches per replay), beside torch.matmul (cuBLAS) for the GEMM shapes."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch
from recommendsystem_b200 import cabi, ops
from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
from embed_sweep_util import timeit

dev = torch.device("cuda:0")
cfg = AutoIntConfig(batch=8192, dtype="bf16", rows_per_field=100_000)
tr = AutoIntTrainer(cfg, dev)
g = torch.Generator(device=dev).manual_seed(0)
ids = torch.randint(0, 100_000, (8192, 39), device=dev, generator=g)
y = (torch.rand(8192, 1, device=dev, generator=g) < 0.25).float()
tr.step(ids, y); torch.cuda.synchronize()
B, F, d = 8192, 39, 16
E = cabi
acts = [tr.X.view(B, F * d)] + tr.H + [tr.Z[:, :tr.n_deep]]
parts = {
    "mlp_fwd0 8192x624->256": lambda: tr._dense_fwd(acts[0], "mlp_W0", "mlp_b0", acts[1]),
    "mlp_fwd1 8192x256->128": lambda: tr._dense_fwd(acts[1], "mlp_W1", "mlp_b1", acts[2]),
    "logit_head": lambda: ops.logit_head(tr.Z, tr.P["out_W"], tr.P["out_b"], tr.labels, tr.dZ, tr.G["out_W"], tr.G["out_b"],
                                          p_out=tr.p_raw, loss=tr.loss, relu_cols=tr.n_deep),
    "mlp_dgrad1 8192x128->256 (+relu mask)": lambda: ops.gemm(tr.dH[1], tr._w("mlp_W1"), tr.dH[0], aux=acts[1],
                                                               epilogue=E.EPI_MUL_RELU_MASK, transB=True),
    "mlp_dgrad_x 8192x256->624": lambda: ops.gemm(tr.dH[0], tr._w("mlp_W0"), tr.dX.view(B, F * d), transB=True),
    "mlp_wgrad0 (side stream)": lambda: (ops.gemm(acts[0], tr.dH[0], tr.G["mlp_W0"], transA=True),
                                         ops.colsum(tr.dH[0], out=tr.G["mlp_b0"])),
    "mlp_wgrad1 (side stream)": lambda: (ops.gemm(acts[1], tr.dH[1], tr.G["mlp_W1"], transA=True),
                                         ops.colsum(tr.dH[1], out=tr.G["mlp_b1"])),
    "sort_keys (side stream)": lambda: ops.sort_keys(tr.keys, tr.row_bits, out=tr.keys_sorted),
    "dense_adam + shadows (side stream)": lambda: (ops.dense_adam(tr.flat, tr.flat_m, tr.flat_v, tr.flat_g, 1e-3, 0.9, 0.999, 1e-8,
                                                                  tr.adam_scalars, tr.flat_bf16), tr._refresh_wt()),
    "adam_advance": lambda: ops.adam_advance(tr.adam_scalars, 0.9, 0.999),
}
for name, fn in parts.items():
    print(json.dumps({"part": name, "us": round(timeit(fn), 2)}))
for (M, K, N) in ((8192, 624, 256), (8192, 256, 128), (8192, 128, 256), (8192, 256, 624)):
    a = torch.randn(M, K, device=dev, dtype=torch.bfloat16); b = torch.randn(K, N, device=dev, dtype=torch.bfloat16)
    print(json.dumps({"cublas bf16": [M, K, N], "us": round(timeit(lambda: torch.matmul(a, b)), 2)}))
