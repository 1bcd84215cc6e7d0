"""AutoInt train step on one B200: the reference's CTR hot path as one captured stream of
hand-written sm_100a kernels (include/rs_b200.h).

    ids [B,S] -> embedding gather / bag mean -> X [B,F,d] --+-> InteractingLayer (L x, shared weights) -> A
                                                            +-> Flatten -> MultiLayerDense(relu)       -> deep
    Z = concat[deep, Flatten(A)] -> Dense(1, sigmoid) -> clip(1e-6, 1) -> cross_entropy
    backward -> dense Adam (flat buffer) + sorted-segment sparse Adam on the touched rows

Reference: AutoInt.model_layer (autoint:18-56), BaseModel.output_layer / cross_entropy
(rank/ctr/base_model.py:7-12,160-201), InteractingLayer.call (InteractingLayer.py:37-61).
`model_config['model_param']` is not shipped by the reference; the defaults below are the
BASELINE.json configuration (SURVEY.md §8c lists them as explicit choices).

torch supplies device memory, streams and CUDA-graph capture; every kernel in the step
comes from librs_b200.so.  There is no CPU path.
"""
from __future__ import annotations

from contextlib import contextmanager
from dataclasses import dataclass, field
from typing import List, Sequence

import numpy as np
import torch

from . import cabi, ops
from .arena import Arena
from .idmap import check_evict_args


class PhaseTimer:
    """CUDA-event timing of the phases of an eagerly launched step (bench.py's per-kernel
    breakdown).  Events are recorded on the stream the kernels are launched on."""

    def __init__(self):
        self.records = {}      # phase -> list of (start, stop) events
        self.launches = {}     # phase -> library launches per occurrence

    def phase(self, name):
        return _Phase(self, name)

    def summary(self):
        """phase -> (mean ms, launches per step)"""
        torch.cuda.synchronize()
        return {k: (float(np.mean([a.elapsed_time(b) for a, b in v])), self.launches.get(k, 0))
                for k, v in self.records.items()}


class _Phase:
    def __init__(self, timer, name):
        self.t, self.name = timer, name

    def __enter__(self):
        if self.t is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.n0 = cabi.launch_count()
            self.a.record()
        return self

    def __exit__(self, *exc):
        if self.t is not None:
            self.b.record()
            self.t.records.setdefault(self.name, []).append((self.a, self.b))
            self.t.launches[self.name] = cabi.launch_count() - self.n0
        return False


@dataclass
class AutoIntConfig:
    num_fields: int = 39
    rows_per_field: int | Sequence[int] = 1_000_000
    embed_dim: int = 16
    # model_param.interact
    layer_num: int = 3
    unit_num: int = 16
    head_num: int = 2
    use_res: bool = True
    ln_eps: float = 1e-3
    # model_param.mlp / logits
    mlp_hidden: Sequence[int] = (256, 128)
    batch: int = 8192
    dtype: str = "f32"              # activation dtype: "f32" | "bf16" (tables and master weights stay fp32)
    lr_dense: float = 5e-5          # rank/ctr/base_model.py:192
    lr_sparse: float = 5e-5         # rank/ctr/base_model.py:163
    beta1: float = 0.9
    beta2: float = 0.999
    eps: float = 1e-8
    table_init_scale: float = 0.1
    seed: int = 20261018
    # bf16 / tcgen05 mode: the embedding lookup runs inside the InteractingLayer forward's tile loader and the
    # embedding-gradient push (multi-GPU) inside its backward's epilogue; False = separate gather / scatter kernels
    fuse_embedding: bool = True
    # "mod": row = row_base[f] + id mod rows_per_field[f].  "hash": every distinct (field, id) gets its own row of the
    # field's rows_per_field (a capacity) the first time a train step sees it (recommendsystem_b200.idmap)
    id_map: str = "mod"
    # bf16 mode with the fused lookup: the whole tower (both Dense(relu) layers, the logit head and their backward
    # down to dX) as one launch (rs_tower_step) where the kernel exists for the widths; False = 4 GEMMs + the head pass
    fuse_tower: bool = True
    # multi-valued fields (VarLenFeature ids, combiner='mean'): the most ids field f takes per sample (int: every field).
    # Field f owns the columns [off_f, off_f + K_f) of the [B, S] id input (S = sum K, off = exclusive cumsum of K); an
    # id < 0 is padding and X[b, f] is the mean of the rows of the bag's valid ids (zeros for an empty bag)
    bag_size: int | Sequence[int] = 1

    def rows(self) -> List[int]:
        if isinstance(self.rows_per_field, int):
            return [self.rows_per_field] * self.num_fields
        assert len(self.rows_per_field) == self.num_fields
        return list(self.rows_per_field)

    def bags(self) -> List[int]:
        """K_f per field; ValueError for a length other than num_fields or a K_f < 1."""
        if isinstance(self.bag_size, (int, np.integer)):
            K = [int(self.bag_size)] * self.num_fields
        else:
            K = [int(k) for k in self.bag_size]
            if len(K) != self.num_fields:
                raise ValueError(f"bag_size has {len(K)} entries for {self.num_fields} fields")
        if any(k < 1 for k in K):
            raise ValueError(f"bag_size: every field takes at least one id, got {K}")
        return K


class AutoIntTrainer:
    """Owns tables, optimizer state and dense parameters; `step()` launches one train step."""

    def __init__(self, cfg: AutoIntConfig, device="cuda:0", tables: torch.Tensor | None = None,
                 dense_init: dict | None = None):
        self.K = cfg.bags()
        self.S = sum(self.K)                 # id columns per sample
        if cfg.batch * self.S >= 2 ** 31:
            raise ValueError(f"batch * sum(bag_size) = {cfg.batch * self.S} slots: sort-key positions are 32-bit")
        # bags: the step's lookups take the mean over each field's slots; with every K_f = 1 they are plain gathers
        self.bag = self.S > cfg.num_fields
        cabi.load()
        self.cfg = cfg
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise RuntimeError("AutoIntTrainer runs on a CUDA device only (no CPU fallback)")
        self.act_dtype = {"f32": torch.float32, "bf16": torch.bfloat16}[cfg.dtype]
        F, d, U, B = cfg.num_fields, cfg.embed_dim, cfg.unit_num, cfg.batch
        if cfg.layer_num > 1 and d != U:
            raise ValueError("layer_num > 1 needs embed_dim == unit_num (InteractingLayer.py:41-46)")
        self.store = ar = Arena(cfg.rows(), d, self.dev, shard=self._arena_shard(), id_map=cfg.id_map, seed=cfg.seed,
                                scale=cfg.table_init_scale)
        self.arena, self.table, self.table_m, self.table_v, self.table_ld = ar.records, ar.w, ar.m, ar.v, ar.ld
        self.rows_host, self.base_host, self.rows_t, self.base_t = ar.rows, ar.base, ar.rows_t, ar.base_t
        self.total_rows, self.idmap, self.row_bits = ar.total_rows, ar.idmap, ar.row_bits
        self._init_tables(tables)

        # ---- dense parameters: one flat fp32 buffer (+ grads, m, v, bf16 shadow) with views
        self.spec = []
        widths = [F * d] + list(cfg.mlp_hidden)
        self.n_deep = widths[-1]
        self.zw = self.n_deep + F * U
        self._add("Wqkvr", (d, 4 * U)); self._add("bqkvr", (4 * U,))
        self._add("gamma", (U,)); self._add("beta", (U,))
        for i in range(len(cfg.mlp_hidden)):
            self._add(f"mlp_W{i}", (widths[i], widths[i + 1])); self._add(f"mlp_b{i}", (widths[i + 1],))
        self._add("out_W", (self.zw, 1)); self._add("out_b", (1,))
        n = (self.spec[-1][2] + int(np.prod(self.spec[-1][1])) + 3) // 4 * 4
        self.n_dense = n
        self.flat = torch.zeros(n, device=self.dev)
        self.flat_g = torch.zeros(n, device=self.dev)
        self.flat_m = torch.zeros(n, device=self.dev)
        self.flat_v = torch.zeros(n, device=self.dev)
        self.flat_bf16 = torch.zeros(n, device=self.dev, dtype=torch.bfloat16)
        self.P = {k: self.flat[o:o + int(np.prod(s))].view(s) for k, s, o in self.spec}
        self.G = {k: self.flat_g[o:o + int(np.prod(s))].view(s) for k, s, o in self.spec}
        self.P16 = {k: self.flat_bf16[o:o + int(np.prod(s))].view(s) for k, s, o in self.spec}
        self._init_dense(dense_init)
        self.adam_scalars = torch.zeros(4, device=self.dev)

        # ---- static activation buffers (fixed addresses => CUDA-graph capturable)
        T = self.act_dtype
        e = lambda *shape, dtype=T: torch.empty(*shape, device=self.dev, dtype=dtype)
        S = self.S
        self.ids = torch.zeros(B, S, dtype=torch.int64, device=self.dev)
        # hash mode: the step's first two launches map ids -> arena rows (static buffer) that every lookup reads
        self.ids_rows = None if self.idmap is None else torch.full((B, S), -1, dtype=torch.int64, device=self.dev)
        self.fields = tuple(range(F))
        self.slot_fields = tuple(f for f in range(F) for _ in range(self.K[f]))     # field of each id column
        # (ids, row_base, rows) the step's embedding lookups read (per-field geometry: bags index it by field)
        self.lookup = (self.ids if self.idmap is None else self.ids_rows, *ar.geom(self.fields))
        self.labels = torch.zeros(B, 1, device=self.dev)
        self.X = e(B, F, d)
        self.keys = torch.empty(B * S, dtype=torch.int64, device=self.dev)
        if self.bag:
            # bag (b, f) = slots [b S + off_f, b S + off_f + K_f): CSR offsets of the B F bags, 1 / count per bag, and the
            # per-slot gradient rows the sorted-segment update reads
            off = np.concatenate([[0], np.cumsum(self.K)]).astype(np.int64)
            self.slot_off = torch.from_numpy(off).to(self.dev)
            self.bag_offsets = torch.from_numpy(np.append((np.arange(B, dtype=np.int64)[:, None] * S + off[None, :F])
                                                          .reshape(-1), B * S)).to(self.dev)
            self.inv_cnt = torch.zeros(B * F, device=self.dev)
            self.g_occ = torch.empty(B * S, d, device=self.dev)
        self.keys_sorted = torch.empty_like(self.keys)
        self.saved = ops.interacting_saved(B, F, U, cfg.layer_num, self.dev)
        self.H = [e(B, w) for w in cfg.mlp_hidden[:-1]]
        self.Z = e(B, self.zw)
        self.p_raw = e(B, 1)
        self.loss = torch.zeros(1, device=self.dev)
        self.dZ = e(B, self.zw)
        # gradient of the last hidden layer = the first n_deep columns of dZ (the head writes them relu-masked)
        self.dH = [e(B, w) for w in cfg.mlp_hidden[:-1]] + [self.dZ[:, :cfg.mlp_hidden[-1]]]
        self.dX = e(B, F, d)
        self.bf16 = self.act_dtype == torch.bfloat16
        if self.bf16:
            # forward GEMMs take K-major operands: [out,in] bf16 weight shadows (weight gradients read
            # activations / gradients MN-major as they lie: no transposed copies)
            self.WT16 = {f"mlp_W{i}": torch.zeros(widths[i + 1], widths[i], dtype=torch.bfloat16, device=self.dev)
                         for i in range(len(cfg.mlp_hidden))}
            self._refresh_wt()
        self.side = torch.cuda.Stream(device=self.dev)
        # Further branches of the step (see _launch_step): the InteractingLayer kernels are persistent and fill every SM,
        # so whatever side work is not finished when the backward starts runs AFTER it; as one serial chain that tail was
        # ~75 us, as parallel branches (weight gradients | bias gradients | reductions) it hides behind the sparse update.
        self.branch = [torch.cuda.Stream(device=self.dev) for _ in range(3)]
        self.sort_done = torch.cuda.Event()
        self.adam_done = torch.cuda.Event()
        self.fused = bool(cfg.fuse_embedding and self.bf16 and ops.interacting_path(
            F, d, U, cfg.head_num, torch.bfloat16, True) == cabi.PATH_TCGEN05 and self.table_ld % 16 == 0)
        # the widths and buffers the tower kernel takes (whether it runs also depends on `fused`: fuse_tower)
        self._tower_ok = bool(cfg.fuse_tower and self.bf16 and len(cfg.mlp_hidden) == 2 and ops.tower_supported(
            F * d, cfg.mlp_hidden[0], cfg.mlp_hidden[1], F * U) and all(
            self.P16[k].data_ptr() % 16 == 0 for k in ("mlp_W0", "mlp_W1")))
        self.graph = None
        self.timer = None               # set to a PhaseTimer for an instrumented (eager) step
        self.stamps, self.stamp_names = None, {}     # set `stamps` to an int64 buffer for tools/step_timeline.py
        n_ws = max(cabi.load().rs_interacting_workspace_bytes(B, F, d, U),
                   cabi.load().rs_embed_sort_workspace_bytes(B * S),
                   cabi.load().rs_colsum_workspace_bytes(B, max(widths + [self.zw])))
        self.ws = torch.empty(int(n_ws) + 256, dtype=torch.uint8, device=self.dev)
        self.head_ws = ops.logit_head_workspace(B, self.zw, self.dev)     # head partials, reduced on the side stream

    @property
    def fuse_tower(self) -> bool:
        """The tower runs as one launch (rs_tower_step).  Only beside the fused InteractingLayer backward, which adds
        its own part to the dX the tower kernel stores."""
        return self._tower_ok and self.fused

    # ------------------------------------------------------------------ setup
    def _arena_shard(self):
        """(W, rank) of a row-sharded arena; None on one GPU."""
        return None

    def _init_tables(self, tables):
        """The global tables [total rows, d] given, or N(0, table_init_scale) from cfg.seed (hash mode: a row is
        initialised when its id is first inserted)."""
        if tables is not None:
            if self.idmap is not None:
                raise ValueError("tables= initialises rows by position; with id_map='hash' rows are initialised per id")
            self.store.load_global(tables)
        elif self.idmap is None:
            self.store.init_normal(self.cfg.seed, self.cfg.table_init_scale)

    def _add(self, name, shape):
        off = 0
        if self.spec:
            _, s, o = self.spec[-1]
            off = (o + int(np.prod(s)) + 3) // 4 * 4      # 16-byte aligned views
        self.spec.append((name, tuple(shape), off))

    def _init_dense(self, init):
        """Keras defaults: Dense kernels glorot_uniform, biases zero; LayerNorm gamma 1 / beta 0."""
        rng = np.random.default_rng(self.cfg.seed)
        U = self.cfg.unit_num
        for name, shape, _ in self.spec:
            if init is not None and name in init:
                v = np.asarray(init[name], np.float32).reshape(shape)
            elif name == "Wqkvr":
                lim = np.sqrt(6.0 / (shape[0] + U))      # four separate Dense(U) kernels side by side
                v = rng.uniform(-lim, lim, size=shape).astype(np.float32)
            elif name == "gamma":
                v = np.ones(shape, np.float32)
            elif len(shape) == 2:
                lim = np.sqrt(6.0 / (shape[0] + shape[1]))
                v = rng.uniform(-lim, lim, size=shape).astype(np.float32)
            else:
                v = np.zeros(shape, np.float32)
            self.P[name].copy_(torch.from_numpy(v))
        self.flat_bf16.copy_(self.flat)

    def _refresh_wt(self):
        for k, wt in self.WT16.items():
            ops.transpose2d(self.P16[k], wt)

    def dense_state(self):
        return {k: v.detach().cpu().numpy().copy() for k, v in self.P.items()}

    # ------------------------------------------------------------------- step
    def _w(self, name):
        """Weights as the GEMM consumes them (fp32 master or bf16 shadow)."""
        return self.P[name] if self.act_dtype == torch.float32 else self.P16[name]

    def _launch_step(self):
        """One train step on torch's current stream using the static buffers."""
        c = self.cfg
        F, d, U, B = c.num_fields, c.embed_dim, c.unit_num, c.batch
        E = cabi
        st = ops._stream()
        T = ops._DT[self.act_dtype]
        P = self.P
        ph = lambda name: _Phase(self.timer, name)
        main = torch.cuda.current_stream(self.dev)
        self._stamp("step_begin")
        if self.idmap is not None:
            with ph("idmap"):
                self.store.lookup(self.ids, self.slot_fields, insert=True, out=self.ids_rows)
        # Adam's step counter / bias corrections are read by the two optimizer kernels at the end of the step only:
        # advance them on the side stream now instead of between the backward and the sparse update
        self.side.wait_stream(main)
        with torch.cuda.stream(self.side):
            ops.adam_advance(self.adam_scalars, c.beta1, c.beta2)
            self.adam_done.record(self.side)
            if self.idmap is not None:
                # hash mode: the show counts of the mapped rows, a branch off the map lookup (nothing in the step
                # reads them; the forward only reads ids_rows) that joins the main stream at the end of the step
                with ph("idmap_count"):
                    self.idmap.count(self.ids_rows)
        if self.fused:
            # K1 inside K4: the forward's tile loader reads the embedding rows itself (local table, or the owners' HBM
            # over NVLink) and writes X and (one GPU) the sort keys as by-products
            tabs, world, lbase_t, keys = self._lookup_args()
            lk_ids, _, lk_rows = self.lookup
            with self._backward_keys(ph), ph("interacting_fwd"):
                if self.bag:      # the bag means, their 1 / count and the per-slot keys come out of the tile loader
                    cabi.call("rs_interacting_fwd_gather_bag", self.table.data_ptr(), self.table_ld, lk_ids.data_ptr(),
                              self.slot_off.data_ptr(), lbase_t.data_ptr(), lk_rows.data_ptr(), self.X.data_ptr(), d, 0,
                              keys, self.inv_cnt.data_ptr(), T, P["Wqkvr"].data_ptr(), P["bqkvr"].data_ptr(),
                              P["gamma"].data_ptr(), P["beta"].data_ptr(), c.ln_eps, self.Z[:, self.n_deep:].data_ptr(),
                              U, self.zw, self.saved.data_ptr(), B, F, self.S, d, U, c.head_num, c.layer_num,
                              int(c.use_res), st)
                else:
                    cabi.call("rs_interacting_fwd_gather", tabs, self.table_ld, world, lk_ids.data_ptr(),
                              lbase_t.data_ptr(), lk_rows.data_ptr(), self.X.data_ptr(), d, 0, keys, T,
                              P["Wqkvr"].data_ptr(), P["bqkvr"].data_ptr(), P["gamma"].data_ptr(), P["beta"].data_ptr(),
                              c.ln_eps, self.Z[:, self.n_deep:].data_ptr(), U, self.zw, self.saved.data_ptr(), B, F, d,
                              U, c.head_num, c.layer_num, int(c.use_res), st)
        else:
            # K1: gather (+ sort keys emitted for the backward)
            with self._backward_keys(ph):
                self._embed_forward(ph, st, T)
            # K4: InteractingLayer forward
            with ph("interacting_fwd"):
                # writes Flatten(A) straight into its columns of the concat buffer Z (autoint:36,45)
                cabi.call("rs_interacting_fwd", self.X.data_ptr(), d, 0, T, P["Wqkvr"].data_ptr(),
                          P["bqkvr"].data_ptr(), P["gamma"].data_ptr(), P["beta"].data_ptr(), c.ln_eps,
                          self.Z[:, self.n_deep:].data_ptr(), U, self.zw,
                          self.saved.data_ptr(), B, F, d, U,
                          c.head_num, c.layer_num, int(c.use_res), int(self.act_dtype == torch.bfloat16), st)
        self._stamp("interacting_fwd_end")
        # K5: MLP tower; last hidden layer lands in Z[:, :n_deep], Flatten(A) in Z[:, n_deep:]
        Xf = self.X.view(B, F * d)
        acts = [Xf] + self.H + [self.Z[:, :self.n_deep]]
        bw, bb, br = self.branch          # weight gradients | bias gradients | small reductions
        if self.fuse_tower:
            self._tower_fused(ph, acts, main)
        else:
            self._tower(ph, acts, main, B)
        # InteractingLayer backward -> dX, then dX += dH0 @ W0^T
        nW = d * 4 * U
        dparams = self.flat_g[self.spec[0][2]:]       # Wqkvr | bqkvr | gamma | beta are contiguous
        assert self.spec[1][2] == nW and self.spec[2][2] == nW + 4 * U and self.spec[3][2] == nW + 5 * U
        if self.fused:
            # the tower's input gradient first (plain store into dX); the InteractingLayer backward adds it to its own
            # dX row by row and, multi-GPU, stores the sum straight into the owners' receive buffers
            if not self.fuse_tower:
                with ph("mlp_dgrad_x"):
                    ops.gemm(self.dH[0], self._w("mlp_W0"), self.dX.view(B, F * d), transB=True)
                self._stamp("mlp_dgrad_x_end")
            with ph("interacting_bwd"):
                self._interacting_bwd_fused(None, st, T, main)      # parameter-gradient partials stay in self.ws
        else:
            with ph("interacting_bwd"):
                self._interacting_bwd(dparams, st, T)
        self._stamp("interacting_bwd_end")
        # all dense gradients exist now: their all-reduce (multi-GPU) and then the dense Adam run on the side
        # stream beside the embedding backward
        if not self.fused:
            with ph("mlp_dgrad_x"):
                ops.gemm(self.dH[0], self._w("mlp_W0"), self.dX.view(B, F * d), epilogue=E.EPI_ACCUM, transB=True)
        bw.wait_stream(main)                 # the last reader of the weights (and their bf16 shadows) is done
        with torch.cuda.stream(bw):
            if self.fused:
                with ph("interacting_bwd_reduce"):
                    cabi.call("rs_interacting_bwd_reduce", self.ws.data_ptr(), self.ws.numel(), dparams.data_ptr(), B, F, d,
                              U, c.head_num, ops._stream())
            bw.wait_stream(bb)
            bw.wait_stream(br)
            bw.wait_event(self.adam_done)
            self._dense_sync(ph)
            with ph("dense_adam"):
                ops.dense_adam(self.flat, self.flat_m, self.flat_v, self.flat_g, c.lr_dense, c.beta1, c.beta2, c.eps,
                               self.adam_scalars, self.flat_bf16)
            if self.bf16:                    # transposed bf16 shadows of the tower weights: one branch each
                for j, (k, wt) in enumerate(self.WT16.items()):
                    sj = (bw, bb, br)[j % 3]
                    if sj is not bw:
                        sj.wait_stream(bw)
                    with torch.cuda.stream(sj):
                        with ph("weight_shadows"):
                            ops.transpose2d(self.P16[k], wt)
            self._stamp("side_end")
        # K3: sparse Adam on touched rows
        main.wait_event(self.adam_done)
        self._embed_backward(ph, st, T, main)
        self._stamp("embed_backward_end")
        main.wait_stream(self.side)
        for sj in self.branch:
            main.wait_stream(sj)
        self._stamp("step_end")

    def _tower(self, ph, acts, main, B):
        """The tower as 4 GEMMs + the head pass (fp32 parity mode, unsupported widths, fuse_tower=False)."""
        c, E, G, P = self.cfg, cabi, self.G, self.P
        nmlp = len(c.mlp_hidden)
        br = self.branch[2]
        with ph("mlp_fwd"):
            for i in range(nmlp):
                self._dense_fwd(acts[i], f"mlp_W{i}", f"mlp_b{i}", acts[i + 1])
        self._stamp("mlp_fwd_end")
        with ph("logits_loss"):
            # final Dense(1, sigmoid) + clip + BCE + the head's backward, one pass over Z
            # dZ[:, :n_deep] leaves the head already multiplied by relu'(last hidden layer): it IS dH[nmlp-1]
            # (its own parameter gradients and the loss are summed on the side stream: only the dense Adam and the
            # host read them, the tower's backward needs dZ alone)
            ops.logit_head(self.Z, P["out_W"], P["out_b"], self.labels, self.dZ, G["out_W"], G["out_b"],
                           p_out=self.p_raw, loss=self.loss, relu_cols=self.n_deep, ws=self.head_ws, defer_reduce=True)
        br.wait_stream(main)
        with torch.cuda.stream(br):
            with ph("logits_loss_reduce"):
                ops.logit_head_reduce(self.head_ws, G["out_W"], G["out_b"], self.loss, B, self.zw)
        self._stamp("head_end")
        # MLP backward (relu masks from the saved activations)
        with ph("mlp_bwd"):
            for i in reversed(range(nmlp)):
                self._tower_param_grads(ph, acts, main, i)
                if i > 0:   # dH[i-1] = (dH[i] @ W_i^T) * relu'(h_{i-1}); W_i [in,out] is the K-major B operand
                    ops.gemm(self.dH[i], self._w(f"mlp_W{i}"), self.dH[i - 1], aux=acts[i],
                             epilogue=E.EPI_MUL_RELU_MASK, transB=True)
        self._stamp("mlp_bwd_end")

    def _tower_fused(self, ph, acts, main):
        """The tower (both Dense(relu) layers, head, their backward down to dX) as one launch; the parameter gradients
        and the head's loss are side branches."""
        c, P, G = self.cfg, self.P, self.G
        B = c.batch
        br = self.branch[2]
        with ph("tower"):
            ops.tower_step(acts[0], self.WT16["mlp_W0"], self.WT16["mlp_W1"], self.P16["mlp_W0"], self.P16["mlp_W1"],
                           P["mlp_b0"], P["mlp_b1"], P["out_W"], P["out_b"], self.labels, self.Z, self.p_raw, self.dZ,
                           self.H[0], self.dH[0], self.dX.view(B, -1))
        self._stamp("tower_end")
        br.wait_stream(main)
        with torch.cuda.stream(br):
            with ph("logits_loss_reduce"):
                ops.logit_head_grad(self.Z, self.p_raw, self.labels, self.head_ws)
                ops.logit_head_reduce(self.head_ws, G["out_W"], G["out_b"], self.loss, B, self.zw)
        for i in reversed(range(len(c.mlp_hidden))):
            self._tower_param_grads(ph, acts, main, i)

    def _tower_param_grads(self, ph, acts, main, i):
        # weight / bias gradients are only consumed by the dense Adam at the end of the step: they run as parallel
        # branches off the dgrad -> InteractingLayer-backward chain (two streams, alternating, for the weight-gradient
        # GEMMs of successive layers; one for the column sums)
        # (launched as soon as their inputs exist: deferring them until after the backward leaves the tower's
        # window to the GEMMs — 11 us — but the tail then outlasts the sparse update by 18 us)
        bw, bb, br = self.branch
        sw = bw if (len(self.cfg.mlp_hidden) - 1 - i) % 2 == 0 else br
        sw.wait_stream(main)
        with torch.cuda.stream(sw):
            with ph("mlp_wgrad"):
                ops.gemm(acts[i], self.dH[i], self.G[f"mlp_W{i}"], transA=True)   # x^T dy, operands as they lie
        bb.wait_stream(main)
        with torch.cuda.stream(bb):
            with ph("mlp_bgrad"):
                ops.colsum(self.dH[i], out=self.G[f"mlp_b{i}"])

    def _stamp(self, name):
        """Measurement aid (tools/step_timeline.py): with `self.stamps` set to an int64 device buffer, a one-thread
        kernel stores the GPU's global timer when the CURRENT stream reaches this point of the step."""
        if getattr(self, "stamps", None) is None:
            return
        i = self.stamp_names.setdefault(name, len(self.stamp_names))
        cabi.call("rs_debug_timestamp", self.stamps[i:].data_ptr(), ops._stream())

    # ---- embedding halves of the step (overridden by the row-sharded multi-GPU trainer)
    @contextmanager
    def _backward_keys(self, ph):
        """Around the launch that makes the sort keys for the sparse update (the gather, or the forward with the lookup
        inside): the key sort follows it on the side stream, hidden behind the dense forward / backward (a parallel
        branch of the captured graph)."""
        yield
        self.side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(self.side):
            with ph("sort_keys"):
                ops.sort_keys(self.keys, self.row_bits, out=self.keys_sorted)
            self.sort_done.record(self.side)
            self._stamp("side_sort_end")

    def _lookup_args(self):
        """(address of the W table pointers, W, per-field local row base, sort-key buffer) of the fused lookup."""
        if not hasattr(self, "_tab1"):
            import ctypes
            self._tab1 = (ctypes.c_void_p * 1)(self.table.data_ptr())
        import ctypes
        return ctypes.addressof(self._tab1), 1, self.lookup[1], self.keys.data_ptr()

    def _scatter_args(self):
        """(address of the W receive-buffer pointers, W, rank, inverse, cap) of the fused gradient push; None on one GPU."""
        return None

    def _interacting_bwd_fused(self, dparams, st, T, main):
        c = self.cfg
        F, d, U, B = c.num_fields, c.embed_dim, c.unit_num, c.batch
        P = self.P
        sa = self._scatter_args()
        recv, world, rank, inverse, cap = sa if sa is not None else (None, 1, 0, None, 0)
        cabi.call("rs_interacting_bwd_scatter", self.X.data_ptr(), d, 0, self.saved.data_ptr(), T,
                  P["Wqkvr"].data_ptr(), P["bqkvr"].data_ptr(), P["gamma"].data_ptr(), P["beta"].data_ptr(), c.ln_eps,
                  self.dZ[:, self.n_deep:].data_ptr(), U, self.zw, self.dX.data_ptr(), d, 0, self.dX.data_ptr(),
                  recv, world, rank, inverse, cap, None if dparams is None else dparams.data_ptr(), B, F, d, U,
                  c.head_num, c.layer_num,
                  int(c.use_res), self.ws.data_ptr(), self.ws.numel(), st)

    def _embed_forward(self, ph, st, T):
        """The separate gather: X and the sort keys."""
        c = self.cfg
        n = c.batch * c.num_fields
        ids, base, rows = self.lookup
        if self.bag:
            with ph("embed_bag_fwd"):
                cabi.call("rs_embed_bag_fwd_ld", self.table.data_ptr(), self.table_ld, ids.data_ptr(),
                          self.bag_offsets.data_ptr(), base.data_ptr(), rows.data_ptr(), n, c.num_fields, c.embed_dim,
                          self.X.data_ptr(), T, self.keys.data_ptr(), self.inv_cnt.data_ptr(), st)
            return
        with ph("embed_gather"):
            cabi.call("rs_embed_gather_fwd_ld", self.table.data_ptr(), self.table_ld, ids.data_ptr(),
                      base.data_ptr(), rows.data_ptr(), n, c.num_fields, c.embed_dim, self.X.data_ptr(), T,
                      self.keys.data_ptr(), None, st)

    def _embed_backward(self, ph, st, T, main):
        grad = self.dX.view(-1, self.cfg.embed_dim)
        if self.bag:
            # one gradient row per slot, dX[b, f] / count (padding slots are skipped by the segment sum)
            with ph("embed_bag_grad"):
                cabi.call("rs_embed_bag_grad", self.dX.data_ptr(), T, self.bag_offsets.data_ptr(),
                          self.inv_cnt.data_ptr(), self.cfg.batch * self.cfg.num_fields, self.cfg.embed_dim,
                          self.g_occ.data_ptr(), st)
            grad = self.g_occ
        main.wait_event(self.sort_done)        # sorted keys (not the dense work queued behind them)
        with ph("embed_segsum_adam"):
            self._sparse_update(grad, self.keys_sorted)

    def _sparse_update(self, grad, keys_sorted, grad_scale=1.0):
        """Sorted-segment sum of the gradient rows + sparse Adam on the rows `keys_sorted` names."""
        c = self.cfg
        ops.segsum_adam(self.table, self.table_m, self.table_v, grad, keys_sorted, c.lr_sparse, c.beta1, c.beta2, c.eps,
                        self.adam_scalars, grad_scale=grad_scale)

    def _dense_sync(self, ph):
        """Single GPU: nothing to exchange.  (Multi-GPU: all-reduce of the flat dense gradient.)"""

    def _interacting_bwd(self, dparams, st, T):
        c = self.cfg
        F, d, U, B = c.num_fields, c.embed_dim, c.unit_num, c.batch
        P = self.P
        # dA is read in place from the Z-gradient columns [n_deep:] (sample stride zw)
        cabi.call("rs_interacting_bwd", self.X.data_ptr(), d, 0, self.saved.data_ptr(),
                  T, P["Wqkvr"].data_ptr(), P["bqkvr"].data_ptr(), P["gamma"].data_ptr(), P["beta"].data_ptr(),
                  c.ln_eps, self.dZ[:, self.n_deep:].data_ptr(), U, self.zw, self.dX.data_ptr(), d, 0,
                  dparams.data_ptr(), B, F, d, U, c.head_num, c.layer_num, int(c.use_res),
                  int(self.act_dtype == torch.bfloat16), self.ws.data_ptr(), self.ws.numel(), st)

    def _dense_fwd(self, x, wname, bname, out):
        """out = relu(x @ W + b)  (Dense(relu))."""
        if self.bf16:
            ops.gemm(x, self.WT16[wname], out, bias=self.P[bname], epilogue=cabi.EPI_BIAS_RELU, transB=True)
        else:
            ops.gemm(x, self.P[wname], out, bias=self.P[bname], epilogue=cabi.EPI_BIAS_RELU)

    def evict(self, threshold: float, decay: float = 1.0):
        """Hash mode: show = show * decay for every id, then drop the ids whose show is below `threshold`; their rows
        are freed for new ids (idmap.IdMap.evict).  Runs on the current stream between steps; the buffers stay where
        they are, so a captured step remains valid."""
        threshold, decay = check_evict_args(threshold, decay)
        if self.idmap is None:
            raise ValueError("evict needs id_map='hash' (mod-mode tables have no ids to drop)")
        self.idmap.evict(threshold, decay)

    # --------------------------------------------------------------- frontends
    def _check_ids(self, ids):
        """ids must be [B, S]: S = sum(bag_size) id columns per sample."""
        if tuple(ids.shape) != tuple(self.ids.shape):
            raise ValueError(f"ids of shape {tuple(ids.shape)}: the trainer takes [batch, sum(bag_size)] = "
                             f"{tuple(self.ids.shape)}")

    def step(self, ids: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        """Device-resident inputs -> one train step; returns the loss tensor (device, 1 element).  ids [B, S] int64
        (S = sum(bag_size); field f in the columns [off_f, off_f + K_f)), labels [B, 1]."""
        self._check_ids(ids)
        self.ids.copy_(ids, non_blocking=True)
        self.labels.copy_(labels, non_blocking=True)
        self.run()
        return self.loss

    def run(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self._launch_step()

    # ---- capture: the warm-up launch must not train ---------------------------------------------------
    def _touched_rows(self) -> torch.Tensor:
        """Arena rows the step on the CURRENT static id buffer updates (sorted unique int64); hash mode: the rows of
        the ids already mapped and every row the step's insert may hand out."""
        return self.store.touched_rows([(self.ids, self.slot_fields)])

    def _snapshot(self):
        """Everything one optimizer step changes: the [w|m|v] records of the touched rows, the dense parameters
        with their moments and bf16 shadows, the Adam step scalars."""
        snap = {"arena": self.store.snapshot(self._touched_rows()), "flat": self.flat.clone(),
                "flat_m": self.flat_m.clone(), "flat_v": self.flat_v.clone(), "flat_bf16": self.flat_bf16.clone(),
                "scalars": self.adam_scalars.clone()}
        if self.bf16:
            snap["WT16"] = {k: v.clone() for k, v in self.WT16.items()}
        return snap

    def _restore(self, snap):
        self.store.restore(snap["arena"])
        self.flat.copy_(snap["flat"]); self.flat_m.copy_(snap["flat_m"]); self.flat_v.copy_(snap["flat_v"])
        self.flat_bf16.copy_(snap["flat_bf16"]); self.adam_scalars.copy_(snap["scalars"])
        for k, v in snap.get("WT16", {}).items():
            self.WT16[k].copy_(v)

    def capture(self):
        """Capture the step into a CUDA graph.  The warm-up launch (one real step on whatever the static id / label
        buffers hold) is undone afterwards — tables, optimizer state, dense parameters and the Adam step counter
        are restored bit for bit — so capture() may be called after load_checkpoint / import_keras_autoint
        without changing the loaded weights, and exact resume holds."""
        snap = self._snapshot()
        s = torch.cuda.Stream(device=self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):
            self._launch_step()
        torch.cuda.current_stream(self.dev).wait_stream(s)
        torch.cuda.synchronize(self.dev)
        self._restore(snap)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._launch_step()
        self.graph = g
        return g

    def step_from_host(self, ids_pinned: torch.Tensor, labels_pinned: torch.Tensor) -> float:
        """End-to-end call: pinned host ids/labels -> H2D -> step -> loss read back (D2H)."""
        self._check_ids(ids_pinned)
        self.ids.copy_(ids_pinned, non_blocking=True)
        self.labels.copy_(labels_pinned, non_blocking=True)
        self.run()
        return float(self.loss.item())

    def fit_host(self, batches):
        """End-to-end training loop over an iterable of (ids_pinned [B,S] int64, labels_pinned [B,1] f32) host
        batches; yields one loss (python float) per batch, in order.

        Input pipeline: batch n+1's host->device copy runs on a copy stream into the other half of a
        double buffer while step n computes; step n's loss is copied device->host asynchronously into
        pinned memory and handed out one step later, when it has long arrived.  Every step still moves
        its own inputs H2D and its own loss D2H — they just do not serialise with the compute."""
        def check(ids, labels):
            self._check_ids(ids)
            return self.cfg.batch

        for _, loss in self._pipelined("fit", batches, check, lambda n: self.run(), self.loss):
            yield loss

    def _pipelined(self, key, batches, check, launch, out):
        """The double-buffered input pipeline of fit_host and evaluate: for every (ids [n, S], labels [n, 1]) batch,
        n = check(ids, labels) (raises for a bad batch), the batch is copied into rows [0, n) of the static id / label
        buffers (ids of rows [n, B) = -1), launch(n) runs on the current stream, and (n, float(out)) is yielded, one
        batch late.  Device-resident batches are read on the copy stream after the current stream's earlier work.
        Every caller `key` has its own buffers, events and copy stream: an evaluate() run between two batches of a
        fit_host loop leaves the training batch already uploaded, and the loss not yet handed out, where they are."""
        dev = self.dev
        B = self.cfg.batch
        if not hasattr(self, "_pipes"):
            self._pipes = {}
        if key not in self._pipes:
            self._pipes[key] = {
                "copy": torch.cuda.Stream(device=dev),
                "ids": [torch.empty_like(self.ids) for _ in range(2)],
                "lab": [torch.empty_like(self.labels) for _ in range(2)],
                "ready": [torch.cuda.Event() for _ in range(2)],       # H2D of slot k finished
                "free": [torch.cuda.Event() for _ in range(2)],        # slot k consumed by the step
                "loss": [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)],
                "done": [torch.cuda.Event() for _ in range(2)],        # loss of slot k is on the host
            }
        p = self._pipes[key]
        main = torch.cuda.current_stream(dev)
        it = iter(batches)
        rows = [0, 0]

        def upload(k, batch):
            ids_h, lab_h = batch
            n = rows[k] = check(ids_h, lab_h)
            with torch.cuda.stream(p["copy"]):
                p["copy"].wait_event(p["free"][k])
                if ids_h.is_cuda or lab_h.is_cuda:
                    p["copy"].wait_stream(main)
                for t in (ids_h, lab_h):
                    if t.is_cuda:
                        t.record_stream(p["copy"])
                if n == B:
                    p["ids"][k].copy_(ids_h, non_blocking=True)
                    p["lab"][k].copy_(lab_h, non_blocking=True)
                else:
                    p["ids"][k][:n].copy_(ids_h, non_blocking=True)
                    p["ids"][k][n:].fill_(-1)
                    p["lab"][k][:n].copy_(lab_h, non_blocking=True)
                p["ready"][k].record(p["copy"])

        for k in range(2):
            p["free"][k].record(main)
        nxt = next(it, None)
        if nxt is None:
            return
        upload(0, nxt)
        n = 0
        pending = None
        while nxt is not None:
            k = n & 1
            cur, nxt = nxt, next(it, None)
            main.wait_event(p["ready"][k])
            self.ids.copy_(p["ids"][k], non_blocking=True)          # device-to-device, a few microseconds
            self.labels.copy_(p["lab"][k], non_blocking=True)
            p["free"][k].record(main)
            rows_k = rows[k]
            if nxt is not None:
                upload(k ^ 1, nxt)                                   # overlaps the step below
            launch(rows_k)
            p["loss"][k].copy_(out.reshape(1), non_blocking=True)
            p["done"][k].record(main)
            if pending is not None:
                p["done"][pending[0]].synchronize()
                yield pending[1], float(p["loss"][pending[0]][0])
            pending = (k, rows_k)
            n += 1
        p["done"][pending[0]].synchronize()
        yield pending[1], float(p["loss"][pending[0]][0])

    # ---- evaluation: the train step's forward and the Keras metrics of its p ------------------------------------
    @torch.no_grad()
    def evaluate(self, batches, num_thresholds: int = 200, threshold: float = 0.5) -> dict:
        """Keras `model.evaluate` with `compile(metrics=[AUC(), BinaryAccuracy(), CTR(), COPC()])`: the metrics of
        `api.metrics.BinaryMetrics` (Keras AUC thresholds, accuracy at `threshold`) and the mean loss over every sample
        of `batches`, an iterable of (ids [n, S] int64, labels [n, 1] f32), 1 <= n <= batch, on the host (pinned, for
        overlap) or on the device.  Returns python floats for BinaryMetrics.NAMES and "loss"; the state is fresh per
        call.  Every batch runs the eval step: the train step's forward (its p is bit for bit the p_raw a train step
        from the same state computes) on the static buffers, padded with id -1 rows to the batch size, and the metrics
        and the summed loss of its first n rows.  Nothing the train step updates changes, hash mode inserts and counts
        no id (an unseen id reads as padding), and a captured train graph stays valid.  Full batches replay a CUDA
        graph of the eval step captured on first use; a partial one runs the same launches eagerly."""
        ev = self._eval_state(num_thresholds, threshold)
        ev["metrics"].reset_states()
        count, loss_sum = 0, 0.0
        for n, loss in self._pipelined("eval", batches, self._check_eval_batch, self._eval_run, ev["loss"]):
            count += n
            loss_sum += n * loss                # the batch's fp32 mean times its rows
        totals = torch.tensor([loss_sum, count], dtype=torch.float64, device=self.dev)
        self._eval_reduce(ev, totals)
        out = ev["metrics"].result()
        loss_sum, count = totals.tolist()
        out["loss"] = loss_sum / count if count > 0 else 0.0
        return out

    def _check_eval_batch(self, ids, labels) -> int:
        """n of an (ids [n, S], labels [n, 1]) eval batch; ValueError unless 1 <= n <= batch and the labels are [n, 1]."""
        B, S = self.ids.shape
        if ids.dim() != 2 or ids.shape[1] != S or not 1 <= ids.shape[0] <= B:
            raise ValueError(f"ids of shape {tuple(ids.shape)}: evaluate takes [n, sum(bag_size)] = [n, {S}] with "
                             f"1 <= n <= batch = {B}")
        n = int(ids.shape[0])
        if tuple(labels.shape) != (n, 1):
            raise ValueError(f"labels of shape {tuple(labels.shape)} for {n} rows of ids: evaluate takes [n, 1]")
        return n

    def _eval_state(self, num_thresholds, threshold):
        """The eval step's own buffers: the metric state (BinaryMetrics), the batch loss, scratch for what the forward
        kernels also write (bags: 1 / count; the separate head pass: dZ and its partial sums) and the graph.  Kept
        while num_thresholds and threshold stay the same."""
        key = (int(num_thresholds), float(threshold))
        ev = getattr(self, "_ev", None)
        if ev is not None and ev["key"] == key:
            return ev
        from .api.metrics import BinaryMetrics
        B, F = self.cfg.batch, self.cfg.num_fields
        ev = {"key": key, "metrics": BinaryMetrics(num_thresholds, threshold, self.dev),
              "loss": torch.zeros(1, device=self.dev), "graph": None}
        if self.fused and self.bag:
            ev["inv_cnt"] = torch.empty(B * F, device=self.dev)
        if not self.fuse_tower:
            ev["dZ"] = torch.empty_like(self.dZ)
            ev["head_ws"] = ops.logit_head_workspace(B, self.zw, self.dev)
        self._ev = ev
        return ev

    def _eval_run(self, n):
        """One eval step over the static buffers; a full batch replays the eval graph, captured after its first eager
        launch (no state to restore: the eval step changes none)."""
        ev = self._ev
        full = n == self.cfg.batch
        if full and ev["graph"] is not None:
            ev["graph"].replay()
            return
        self._launch_eval(n)
        if full:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._launch_eval(n)
            ev["graph"] = g

    def _launch_eval(self, n):
        """The eval step on torch's current stream: the train step's forward (same kernels, same arithmetic; no saved
        activations, sort keys or gradients) into p_raw, then the metrics and the summed loss of rows [0, n)."""
        c = self.cfg
        F, d, U, B = c.num_fields, c.embed_dim, c.unit_num, c.batch
        st, T, P = ops._stream(), ops._DT[self.act_dtype], self.P
        ev = self._ev
        if self.fused:
            self.store.lookup(self.ids, self.slot_fields, insert=False, out=self.ids_rows)
            tabs, world, lbase_t, _ = self._lookup_args()
            lk_ids, _, lk_rows = self.lookup
            if self.bag:
                cabi.call("rs_interacting_fwd_gather_bag", self.table.data_ptr(), self.table_ld, lk_ids.data_ptr(),
                          self.slot_off.data_ptr(), lbase_t.data_ptr(), lk_rows.data_ptr(), self.X.data_ptr(), d, 0,
                          None, ev["inv_cnt"].data_ptr(), T, P["Wqkvr"].data_ptr(), P["bqkvr"].data_ptr(),
                          P["gamma"].data_ptr(), P["beta"].data_ptr(), c.ln_eps, self.Z[:, self.n_deep:].data_ptr(), U,
                          self.zw, None, B, F, self.S, d, U, c.head_num, c.layer_num, int(c.use_res), st)
            else:
                cabi.call("rs_interacting_fwd_gather", tabs, self.table_ld, world, lk_ids.data_ptr(), lbase_t.data_ptr(),
                          lk_rows.data_ptr(), self.X.data_ptr(), d, 0, None, T, P["Wqkvr"].data_ptr(),
                          P["bqkvr"].data_ptr(), P["gamma"].data_ptr(), P["beta"].data_ptr(), c.ln_eps,
                          self.Z[:, self.n_deep:].data_ptr(), U, self.zw, None, B, F, d, U, c.head_num, c.layer_num,
                          int(c.use_res), st)
        else:
            self._predict_lookup(st, T)
            cabi.call("rs_interacting_fwd", self.X.data_ptr(), d, 0, T, P["Wqkvr"].data_ptr(), P["bqkvr"].data_ptr(),
                      P["gamma"].data_ptr(), P["beta"].data_ptr(), c.ln_eps, self.Z[:, self.n_deep:].data_ptr(), U,
                      self.zw, None, B, F, d, U, c.head_num, c.layer_num, int(c.use_res), int(self.bf16), st)
        Xf = self.X.view(B, F * d)
        if self.fuse_tower:
            ops.tower_fwd(Xf, self.WT16["mlp_W0"], self.WT16["mlp_W1"], self.P16["mlp_W0"], self.P16["mlp_W1"],
                          P["mlp_b0"], P["mlp_b1"], P["out_W"], P["out_b"], self.Z, self.p_raw)
        else:
            acts = [Xf] + self.H + [self.Z[:, :self.n_deep]]
            for i in range(len(c.mlp_hidden)):
                self._dense_fwd(acts[i], f"mlp_W{i}", f"mlp_b{i}", acts[i + 1])
            # the train step's head pass; its dZ and gradient partials land in the eval step's scratch
            ops.logit_head(self.Z, P["out_W"], P["out_b"], self.labels, ev["dZ"], None, None, p_out=self.p_raw,
                           loss=ev["loss"], relu_cols=self.n_deep, ws=ev["head_ws"], defer_reduce=True)
        m = ev["metrics"]
        ops.binary_metrics_update(m.state, self.p_raw[:n], self.labels[:n], m.thresholds, m.threshold)
        ops.bce_sigmoid_fwd_bwd(self.p_raw[:n], self.labels[:n], want_grad=False, loss=ev["loss"])

    def _eval_reduce(self, ev, totals):
        """One GPU: nothing to merge.  (Sharded: the sum of every rank's metric state and loss totals.)"""

    @torch.no_grad()
    def predict(self, ids: torch.Tensor) -> torch.Tensor:
        """Forward only on this rank's batch (clip(sigmoid) probabilities), eager launches.  Hash mode: ids are looked
        up, never inserted (unseen ids read as zero vectors).  Sharded: the rows are read from the owners' shards."""
        c = self.cfg
        F, d, U, B = c.num_fields, c.embed_dim, c.unit_num, c.batch
        self._check_ids(ids)
        self.ids.copy_(ids)
        T = ops._DT[self.act_dtype]
        st = ops._stream()
        P = self.P
        self._predict_lookup(st, T)
        cabi.call("rs_interacting_fwd", self.X.data_ptr(), d, 0, T, P["Wqkvr"].data_ptr(), P["bqkvr"].data_ptr(),
                  P["gamma"].data_ptr(), P["beta"].data_ptr(), c.ln_eps, self.Z[:, self.n_deep:].data_ptr(), U,
                  self.zw, None, B, F, d, U, c.head_num, c.layer_num, int(c.use_res), 0, st)
        acts = [self.X.view(B, F * d)] + self.H + [self.Z[:, :self.n_deep]]
        for i in range(len(c.mlp_hidden)):
            self._dense_fwd(acts[i], f"mlp_W{i}", f"mlp_b{i}", acts[i + 1])
        # the head kernel also produces gradients; they land in scratch and are ignored here
        ops.logit_head(self.Z, P["out_W"], P["out_b"], self.labels, self.dZ, self.G["out_W"], self.G["out_b"],
                       p_out=self.p_raw, loss=self.loss)
        return self.p_raw.float().clamp(1e-6, 1.0)

    def _predict_lookup(self, st, T):
        """X = the embedding rows (bags: their means) of the static id buffer, inserting no id."""
        c = self.cfg
        ids = self.store.lookup(self.ids, self.slot_fields, insert=False, out=self.ids_rows)[0]
        _, base, rows = self.lookup
        if self.bag:
            cabi.call("rs_embed_bag_fwd_ld", self.table.data_ptr(), self.table_ld, ids.data_ptr(),
                      self.bag_offsets.data_ptr(), base.data_ptr(), rows.data_ptr(), c.batch * c.num_fields,
                      c.num_fields, c.embed_dim, self.X.data_ptr(), T, None, None, st)
            return
        cabi.call("rs_embed_gather_fwd_ld", self.table.data_ptr(), self.table_ld, ids.data_ptr(), base.data_ptr(),
                  rows.data_ptr(), c.batch * c.num_fields, c.num_fields, c.embed_dim, self.X.data_ptr(), T, None, None,
                  st)
