"""Sparse embedding + sparse optimizer surface the reference reaches through `tensornet` (tn):
    tn.feature_column.category_column / embedding_column, tn.layers.EmbeddingFeatures,
    tn.core.Adam / tn.core.AdaGrad
(call sites staytime/VideoDnn.py:217-244, rough_rank/model.py:89-115, rank/ctr/base_model.py:203-217).
TensorNet itself is not vendored by the reference: table storage, the `bucket_size` semantics (ids
are reduced mod bucket_size here) and the exact update rules are this repo's documented choices
(SURVEY.md §8c, DESIGN.md).  All tables of one EmbeddingFeatures layer live in ONE fp32 arena so a
batch is served by a single gather launch and a single sorted-segment update launch.

`id_map="hash"` replaces the modulo rule by a collision-free map (recommendsystem_b200.idmap): every distinct
(column, id) gets its own row of the column's `bucket_size` rows, as TensorNet's hash tables give every feature sign
its own row, and `evict` drops the ids whose decayed show count falls below AdaGrad's `feature_drop_show`."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional

import torch

from .. import cabi, ops
from ..arena import Arena
from ..idmap import check_evict_args


@dataclass
class CategoryColumn:
    key: str
    bucket_size: int


@dataclass
class EmbeddingColumn:
    categorical_column: CategoryColumn
    dimension: int
    combiner: Optional[str] = "mean"
    seq_max_len: Optional[int] = None
    name: Optional[str] = None

    @property
    def key(self):
        return self.name or self.categorical_column.key


def category_column(key, bucket_size):
    return CategoryColumn(str(key), int(bucket_size))


def embedding_column(categorical_column, dimension, combiner="mean", seq_max_len=None, name=None):
    return EmbeddingColumn(categorical_column, int(dimension), combiner, seq_max_len, name)


class Adam:
    """tn.core.Adam(learning_rate, beta1, beta2, epsilon) — sparse rows touched by the batch."""

    def __init__(self, learning_rate=0.001, beta1=0.9, beta2=0.999, epsilon=1e-8):
        self.learning_rate, self.beta1, self.beta2, self.epsilon = learning_rate, beta1, beta2, epsilon


class AdaGrad:
    """tn.core.AdaGrad(learning_rate, initial_g2sum, initial_scale[, feature_drop_show]).
    One g2sum scalar per row (TensorNet style); rows are initialised N(0,1) * initial_scale.  `feature_drop_show` is
    the show threshold EmbeddingFeatures.evict uses by default (id_map="hash"); -1 drops nothing."""

    def __init__(self, learning_rate=0.01, initial_g2sum=0, initial_scale=1, epsilon=1e-8, feature_drop_show=-1,
                 per_element=False):
        self.learning_rate, self.initial_g2sum, self.initial_scale = learning_rate, initial_g2sum, initial_scale
        self.epsilon, self.per_element, self.feature_drop_show = epsilon, per_element, feature_drop_show


class EmbeddingFeatures:
    """EmbeddingFeatures(embedding_columns, sparse_opt, name)(inputs: dict[key -> ids]) ->
    dict[column key -> [B, d]]  (combiner='mean', dense [B] or [B, bag] ids; id < 0 = padding) or
    ([B, T, d], mask [B, T]) for `combiner=None, seq_max_len=T` sequence columns.

    `backward(grads)` applies the fused sorted-segment sparse optimizer to the rows the last
    forward touched (the reference's server-side push); `grads` maps column key -> d(loss)/d(output).

    id_map="mod" (default): row = row_base[column] + id mod bucket_size.  id_map="hash": `bucket_size` is the
    column's row capacity and each distinct id gets its own row the first time a call with gradients enabled
    (training) sees it, initialised N(0, scale) as a function of (seed, column, id); calls under torch.no_grad()
    (the nets' predict) give unseen ids zero vectors and change nothing.  Once a column's rows are used up, new ids
    read as zero vectors and get no update, like padding (`idmap.stats()` counts them).  Training calls also count
    every id's shows; `evict(threshold, decay)` decays them and frees the rows of the ids below the threshold."""

    def __init__(self, embedding_columns: List[EmbeddingColumn], sparse_opt, name="embedding", device="cuda:0",
                 out_dtype=torch.float32, seed=0, id_map="mod"):
        self.id_map = id_map
        self.cols = list(embedding_columns)
        self.opt = sparse_opt
        self.dev = torch.device(device)
        dims = {c.dimension for c in self.cols}
        if len(dims) != 1:
            raise ValueError("one EmbeddingFeatures layer holds columns of a single dimension (one arena)")
        self.d = dims.pop()
        self.out_dtype = out_dtype
        if not isinstance(sparse_opt, (Adam, AdaGrad)):
            raise TypeError("sparse_opt must be api.embedding.Adam or AdaGrad")
        scale = float(getattr(sparse_opt, "initial_scale", 0.1) if isinstance(sparse_opt, AdaGrad) else 0.1)
        adagrad = None if isinstance(sparse_opt, Adam) else (sparse_opt.initial_g2sum, sparse_opt.per_element)
        # every table of the layer in one arena (sharded layer: this rank's rows of it), N(0, scale) from `seed`
        self.store = ar = Arena([c.categorical_column.bucket_size for c in self.cols], self.d, self.dev,
                                shard=self._arena_shard(), adagrad=adagrad, id_map=id_map, seed=seed, scale=scale)
        if ar.idmap is None:                    # (hash mode: a row is initialised when its id is first inserted)
            ar.init_normal(seed, scale)
        self.table, self.arena, self.m, self.v, self.g2sum = ar.w, ar.records, ar.m, ar.v, ar.g2sum
        self.idmap, self.base, self.rows, self.table_ld, self.row_bits = ar.idmap, ar.base, ar.rows, ar.ld, ar.row_bits
        if isinstance(sparse_opt, Adam):
            self.scalars = torch.zeros(4, device=self.dev)
        self._last = None
        self._pending_backward = False

    def _arena_shard(self):
        """(W, rank) of a row-sharded layer; None on one GPU."""
        return None

    def __call__(self, inputs: Dict[str, torch.Tensor]):
        out, plan = {}, []
        # single-valued mean columns (ids [B] / [B,1], the Criteo-shaped case) share ONE gather launch over
        # the stacked ids [B, F'] (per-column row_base / bucket size) and one sorted-segment push
        single = [ci for ci, c in enumerate(self.cols) if c.combiner is not None and
                  not isinstance(inputs[c.categorical_column.key], (tuple, list)) and
                  (inputs[c.categorical_column.key].dim() == 1 or inputs[c.categorical_column.key].shape[1] == 1)]
        if len(single) > 1:
            ids = torch.stack([inputs[self.cols[ci].categorical_column.key].reshape(-1) for ci in single], dim=1)
            ids = ids.to(self.dev, torch.int64).contiguous()
            ids, base, rows = self._lookup(ids, single)
            emb, keys, _ = ops.embed_gather(self.table, ids, base, rows, torch.float32, want_keys=True)
            for j, ci in enumerate(single):
                out[self.cols[ci].key] = emb[:, j, :].to(self.out_dtype)
            plan.append(([self.cols[ci].key for ci in single], keys, 1.0, None))
            # the gather output as it lies: (column keys, [B, F', d]) for consumers that work on the stacked tensor
            self.last_stacked = ([self.cols[ci].key for ci in single], emb.to(self.out_dtype))
        else:
            single = []
            self.last_stacked = None
        for ci, c in enumerate(self.cols):
            if ci in single:
                continue
            raw = inputs[c.categorical_column.key]
            if isinstance(raw, (tuple, list)):
                # variable-length bag in CSR form (values int64 [nnz], offsets int64 [B+1]): the VarLenFeature /
                # SparseTensor input of the reference (staytime/parse.py:22-23), combiner='mean' (VideoDnn.py:224-226)
                if c.combiner is None:
                    raise ValueError("CSR (values, offsets) inputs are for combiner='mean' columns")
                vals, base, rows = self._lookup(raw[0].to(self.dev, torch.int64).contiguous(), (ci,))
                offs = raw[1].to(self.dev, torch.int64).contiguous()
                nb = offs.numel() - 1
                emb = torch.empty(nb, self.d, dtype=torch.float32, device=self.dev)
                keys = torch.empty(vals.numel(), dtype=torch.int64, device=self.dev)
                inv = torch.empty(nb, dtype=torch.float32, device=self.dev)
                cabi.call("rs_embed_bag_fwd_ld", self.table.data_ptr(), self.table_ld, vals.data_ptr(), offs.data_ptr(),
                          base.data_ptr(), rows.data_ptr(), nb, 1, self.d, emb.data_ptr(), cabi.RS_F32, keys.data_ptr(),
                          inv.data_ptr(), ops._stream())
                out[c.key] = emb.to(self.out_dtype)
                plan.append((c.key, keys, None, ("csr", offs, inv)))
                continue
            ids = raw.to(self.dev, torch.int64)
            if c.combiner is None:                               # sequence column -> ([B,T,d], mask)
                T = c.seq_max_len or ids.shape[1]
                seq = ids[:, :T].contiguous()
                lk, base, rows = self._lookup(seq.reshape(-1, 1), (ci,))
                emb, keys, arows = ops.embed_gather(self.table, lk, base, rows, self.out_dtype,
                                                    want_keys=True, want_rows=True)
                out[c.key] = (emb.view(seq.shape[0], T, self.d), (arows.view(seq.shape[0], T) >= 0))
                plan.append((c.key, keys, 1.0, None))
            else:
                if ids.dim() == 1:
                    ids = ids[:, None]
                B, bag = ids.shape
                lk, base, rows = self._lookup(ids.reshape(-1, 1).contiguous(), (ci,))
                emb, keys, arows = ops.embed_gather(self.table, lk, base, rows,
                                                    torch.float32, want_keys=True, want_rows=True)
                if bag == 1:
                    out[c.key] = emb.view(B, self.d).to(self.out_dtype)
                    plan.append((c.key, keys, 1.0, None))
                else:                                            # combiner='mean' over the valid ids of the bag
                    valid = (arows.view(B, bag) >= 0)
                    cnt = valid.sum(1).clamp(min=1).to(torch.float32)
                    out[c.key] = (emb.view(B, bag, self.d).sum(1) / cnt[:, None]).to(self.out_dtype)
                    plan.append((c.key, keys, None, (bag, cnt)))
        self._last = plan
        self._pending_backward = torch.is_grad_enabled()
        return out

    # ---- state one train step changes (GraphedTrainStep undoes its warm-up steps with these) -----------
    def touched_rows(self, inputs: Dict[str, torch.Tensor]) -> torch.Tensor:
        """Sorted unique arena rows a step on `inputs` reads and updates (hash mode: the rows of the ids already
        mapped, and every row the step's inserts may hand out)."""
        return self.store.touched_rows(list(self._column_ids(inputs)))

    def _column_ids(self, inputs):
        """(ids [N, 1], (column,)) of every column: the ids a step on `inputs` looks up (< 0 = padding)."""
        for ci, c in enumerate(self.cols):
            ids = inputs[c.categorical_column.key]
            if isinstance(ids, (tuple, list)):                   # CSR bag: (values, offsets)
                ids = ids[0]
            elif c.combiner is None and c.seq_max_len:
                ids = ids[:, :c.seq_max_len]
            yield ids.to(self.dev, torch.int64).reshape(-1, 1), (ci,)

    def snapshot(self, inputs):
        scalars = self.scalars.clone() if isinstance(self.opt, Adam) else None
        return self.store.snapshot(self.touched_rows(inputs)), scalars

    def restore(self, snap):
        rows, scalars = snap
        self.store.restore(rows)
        if scalars is not None:
            self.scalars.copy_(scalars)

    def _lookup(self, ids, cols):
        """(ids, row_base, rows) the gather kernels read for the columns `cols`; hash mode inserts new ids and counts
        the shows of every id when gradients are enabled (training)."""
        train = torch.is_grad_enabled()
        lk = self.store.lookup(ids, cols, insert=train)
        if train and self.idmap is not None:
            self.idmap.count(lk[0])
        return lk

    def evict(self, threshold: Optional[float] = None, decay: float = 1.0):
        """Hash mode: show = show * decay for every id, then drop the ids whose show is below `threshold` (default:
        AdaGrad's feature_drop_show; with Adam it must be given).  Their rows are freed for new ids; an evicted id
        reads as a zero vector until a training call sees it again.  Call it between steps: not while a training
        forward waits for its backward (its sort keys hold row numbers)."""
        if threshold is None:
            if not isinstance(self.opt, AdaGrad):
                raise ValueError("evict: with Adam the threshold must be given (AdaGrad defaults to feature_drop_show)")
            threshold = self.opt.feature_drop_show
        threshold, decay = check_evict_args(threshold, decay)
        if self.idmap is None:
            raise ValueError("evict needs id_map='hash' (mod-mode tables have no ids to drop)")
        if self._pending_backward:
            raise RuntimeError("evict called between a training forward and its backward")
        self._last = None                          # the plan of an inference call names rows that may move
        self.idmap.evict(threshold, decay)

    def backward(self, grads: Dict[str, torch.Tensor]):
        """Push d(loss)/d(output) of every column: segment-sum per touched row + optimizer update."""
        if self._last is None:
            raise RuntimeError("EmbeddingFeatures.backward called before a forward")
        if isinstance(self.opt, Adam):
            ops.adam_advance(self.scalars, self.opt.beta1, self.opt.beta2)
        for key, keys, scale, bag in self._last:
            if isinstance(key, list):                             # stacked single-valued columns: [B, F', d]
                g = torch.stack([grads[k] for k in key], dim=1)
            else:
                g = grads[key]
            if isinstance(g, tuple):
                g = g[0]
            g = g.reshape(-1, self.d)
            if bag is not None and bag[0] == "csr":               # CSR bag: one gradient row per occurrence
                _, offs, inv = bag
                gc = g.contiguous()
                g = torch.empty(keys.numel(), self.d, dtype=torch.float32, device=self.dev)
                cabi.call("rs_embed_bag_grad", gc.data_ptr(), ops._dt(gc), offs.data_ptr(), inv.data_ptr(),
                          offs.numel() - 1, self.d, g.data_ptr(), ops._stream())
            elif bag is not None:                                 # mean combiner: 1/count per occurrence
                b, cnt = bag
                g = (g.float() / cnt[:, None]).repeat_interleave(b, dim=0)
            g = g.contiguous()
            ks = ops.sort_keys(keys, self.row_bits)
            if isinstance(self.opt, Adam):
                ops.segsum_adam(self.table, self.m, self.v, g, ks, self.opt.learning_rate, self.opt.beta1,
                                self.opt.beta2, self.opt.epsilon, self.scalars)
            else:
                ops.segsum_adagrad(self.table, self.g2sum, g, ks, self.opt.learning_rate, self.opt.epsilon,
                                   self.opt.per_element)
        self._last = None
        self._pending_backward = False
