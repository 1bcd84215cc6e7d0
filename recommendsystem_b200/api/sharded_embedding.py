"""Row-sharded multi-GPU `EmbeddingFeatures` — the sparse side of the composed models on W GPUs.

The reference shards every model's input the same way, `dataset.shard(tn.core.shard_num(), tn.core.self_shard_id())`
(staytime/parse.py:77-79), and leaves the tables to TensorNet's sharded parameter server.  Here: one process per GPU,
each rank holds its own batch (data parallel) and the rows `r mod W == rank` of every table (SURVEY 8e):

    owner(row) = row mod W ;  local row = local_base[column] + row div W

forward   ONE kernel per column group: every rank reads the rows it needs straight out of the owners' HBM over
          NVLink / NVSwitch (CUDA-IPC mappings of all W shards, rs_embed_gather_peer_fwd): bit-exact with the unsharded
          gather.  For the backward the owners need the (row, position) keys of what was read: rs_route_ids_padded
          (fixed-capacity buckets, no host round trip) -> all-to-all(ids) -> keys -> sort.
backward  the gradient rows go straight into the owners' receive buffers with peer stores (rs_scatter_rows_peer),
          a flag barrier over peer memory (rs_peer_barrier) separates the stores from the owners' reads, then the
          owner-local sorted-segment sum + sparse optimizer (Adam or AdaGrad) with grad_scale = 1/W (every rank's
          loss is the mean over ITS batch: the update is that of the global batch), and a second barrier orders every
          owner's update before the next step's peer reads.

Everything is launched on the current stream with fixed buffers: the whole train step — collectives included — is
CUDA-graph capturable (api.graph.GraphedTrainStep).  Buffers of a column group are created at its first use (collective:
every rank runs the same model code), i.e. during the eager warm-up steps, never during capture.
"""
from __future__ import annotations

import ctypes
from typing import Dict, List

import torch
import torch.distributed as dist

from .. import cabi, ops
from ..arena import check_sharded_id_map, field_slices
from ..sharded import bucket_capacity, map_peer_buffers
from .embedding import Adam, AdaGrad, EmbeddingColumn, EmbeddingFeatures


class _Group:
    """Exchange buffers of one column group at a fixed number of lookups."""
    pass


class ShardedEmbeddingFeatures(EmbeddingFeatures):
    def __init__(self, embedding_columns: List[EmbeddingColumn], sparse_opt, name="embedding", device="cuda:0",
                 out_dtype=torch.float32, seed=0, group=None, capacity_factor=None, id_map="mod"):
        check_sharded_id_map(id_map)
        if not dist.is_initialized():
            raise RuntimeError("ShardedEmbeddingFeatures needs torch.distributed (one process per GPU)")
        self.group = group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > 8:
            raise ValueError("peer-memory sharding is built for one NVSwitch domain (<= 8 GPUs)")
        self.capacity_factor = capacity_factor
        self._ipc_opened = {}
        self._groups: Dict[tuple, _Group] = {}
        super().__init__(embedding_columns, sparse_opt, name, device, out_dtype, seed, id_map)
        self.peer_tables = map_peer_buffers(self.table, self.world, self.rank, group, self._ipc_opened)
        self.flags = torch.zeros(16, dtype=torch.int32, device=self.dev)
        torch.cuda.synchronize(self.dev)
        self.peer_flags = map_peer_buffers(self.flags, self.world, self.rank, group, self._ipc_opened)
        self.overflow = torch.zeros(1, dtype=torch.int32, device=self.dev)

    # this rank's rows of every column hold the same values as the unsharded layer with the same seed
    def _arena_shard(self):
        return self.world, self.rank

    # ---- exchange buffers ------------------------------------------------------------------------------------
    def _group(self, gkey, n, cols, padded=False) -> _Group:
        g = self._groups.get((gkey, n))
        if g is not None:
            return g
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("a column group met a new batch shape during CUDA-graph capture: run one eager step first")
        W, d, dev = self.world, self.d, self.dev
        g = _Group()
        g.n, g.F = n, len(cols)
        # Groups that may carry padding (sequence / bag columns) spread it over the owners by a hash of the lookup index
        # (rs_route_ids_padded_spread): the buckets stay balanced and the usual capacity holds.
        g.cap = bucket_capacity(n, W, self.capacity_factor)
        g.pad_spread = bool(padded)
        g.lbase_t, g.rows_t = self.store.geom(cols)
        g.send_rows = torch.empty(W * g.cap, dtype=torch.int32, device=dev)
        g.recv_rows = torch.empty(W * g.cap, dtype=torch.int32, device=dev)
        g.inverse = torch.empty(n, dtype=torch.int32, device=dev)
        g.send_counts = torch.empty(W, dtype=torch.int32, device=dev)
        g.keys = torch.empty(W * g.cap, dtype=torch.int64, device=dev)
        g.keys_sorted = torch.empty_like(g.keys)
        g.g_recv = torch.zeros(W * g.cap, d, dtype=torch.float32, device=dev)
        torch.cuda.synchronize(dev)
        g.peer_grecv = map_peer_buffers(g.g_recv, W, self.rank, self.group, self._ipc_opened)
        self._groups[(gkey, n)] = g
        return g

    def _lookup(self, gkey, ids: torch.Tensor, cols, padded=False) -> torch.Tensor:
        """ids int64 [N, len(cols)] (id < 0 = padding) -> fp32 [N, len(cols), d]; registers the owners' keys."""
        ids = ids.contiguous()
        n = ids.numel()
        g = self._group(gkey, n, tuple(cols), padded)
        out = torch.empty(ids.shape[0], g.F, self.d, dtype=torch.float32, device=self.dev)
        st = ops._stream()
        cabi.call("rs_embed_gather_peer_fwd", ctypes.addressof(self.peer_tables), self.table_ld, self.world, ids.data_ptr(),
                  g.lbase_t.data_ptr(), g.rows_t.data_ptr(), n, g.F, self.d, out.data_ptr(), cabi.RS_F32, st)
        ops.route_ids_padded(ids, g.F, g.rows_t, g.lbase_t, self.world, g.cap, g.send_rows, g.inverse, g.send_counts,
                             self.overflow, pad_spread=g.pad_spread)
        dist.all_to_all_single(g.recv_rows, g.send_rows, group=self.group)
        cabi.call("rs_embed_gather_rows_ld", self.table.data_ptr(), self.table_ld, g.recv_rows.data_ptr(),
                  g.recv_rows.numel(), self.d, None, cabi.RS_F32, None, g.keys.data_ptr(), st)
        ops.sort_keys(g.keys, self.row_bits, out=g.keys_sorted)
        return out, g

    def __call__(self, inputs: Dict[str, torch.Tensor]):
        out, plan = {}, []
        single = [ci for ci, c in enumerate(self.cols) if c.combiner is not None and
                  (inputs[c.categorical_column.key].dim() == 1 or inputs[c.categorical_column.key].shape[1] == 1)]
        if single:
            ids = torch.stack([inputs[self.cols[ci].categorical_column.key].reshape(-1) for ci in single], dim=1)
            emb, g = self._lookup(("single", tuple(single)), ids.to(self.dev, torch.int64), single)
            for j, ci in enumerate(single):
                out[self.cols[ci].key] = emb[:, j, :].to(self.out_dtype)
            plan.append(([self.cols[ci].key for ci in single], g, None))
            self.last_stacked = ([self.cols[ci].key for ci in single], emb.to(self.out_dtype))
        else:
            self.last_stacked = None
        for ci, c in enumerate(self.cols):
            if ci in single:
                continue
            ids = inputs[c.categorical_column.key].to(self.dev, torch.int64)
            if c.combiner is None:                               # sequence column -> ([B,T,d], mask)
                T = c.seq_max_len or ids.shape[1]
                seq = ids[:, :T].contiguous()
                emb, g = self._lookup(("seq", ci), seq.reshape(-1, 1), [ci], padded=True)
                out[c.key] = (emb.view(seq.shape[0], T, self.d).to(self.out_dtype), seq >= 0)
                plan.append((c.key, g, None))
            else:                                                # combiner='mean' over the valid ids of a padded bag
                B, bag = ids.shape
                emb, g = self._lookup(("bag", ci), ids.reshape(-1, 1), [ci], padded=True)
                cnt = (ids >= 0).sum(1).clamp(min=1).to(torch.float32)
                out[c.key] = (emb.view(B, bag, self.d).sum(1) / cnt[:, None]).to(self.out_dtype)
                plan.append((c.key, g, (bag, cnt)))
        self._last = plan
        return out

    def _barrier(self):
        cabi.call("rs_peer_barrier", ctypes.addressof(self.peer_flags), self.world, self.rank, ops._stream())

    def backward(self, grads: Dict[str, torch.Tensor]):
        """Push d(loss)/d(output) of every column to the owners: peer stores -> barrier -> owner-local sorted-segment
        sum + optimizer (grad_scale 1/W) -> barrier."""
        if self._last is None:
            raise RuntimeError("EmbeddingFeatures.backward called before a forward")
        st = ops._stream()
        for key, g, bag in self._last:
            gr = torch.stack([grads[k] for k in key], dim=1) if isinstance(key, list) else grads[key]
            if isinstance(gr, tuple):
                gr = gr[0]
            gr = gr.reshape(-1, self.d).float()
            if bag is not None:
                b, cnt = bag
                gr = (gr / cnt[:, None]).repeat_interleave(b, dim=0)
            gr = gr.contiguous()
            cabi.call("rs_scatter_rows_peer", gr.data_ptr(), ctypes.addressof(g.peer_grecv), self.world, self.rank,
                      g.inverse.data_ptr(), g.n, g.cap, self.d * 4, st)
        self._barrier()                                          # every rank's stores have landed
        if isinstance(self.opt, Adam):
            ops.adam_advance(self.scalars, self.opt.beta1, self.opt.beta2)
        scale = 1.0 / self.world
        for key, g, bag in self._last:
            if isinstance(self.opt, Adam):
                ops.segsum_adam(self.table, self.m, self.v, g.g_recv, g.keys_sorted, self.opt.learning_rate, self.opt.beta1,
                                self.opt.beta2, self.opt.epsilon, self.scalars, grad_scale=scale)
            else:
                ops.segsum_adagrad(self.table, self.g2sum, g.g_recv, g.keys_sorted, self.opt.learning_rate,
                                   self.opt.epsilon, self.opt.per_element, grad_scale=scale)
        self._barrier()                                          # every owner's update precedes the next peer reads
        self._last = None

    def check_overflow(self):
        if int(self.overflow.item()) != 0:
            raise RuntimeError("routing bucket overflow: ids too skewed for the bucket capacity; the step's result is "
                               "invalid — re-create the layer with a larger capacity_factor")

    # ---- state one step changes (GraphedTrainStep) / test helpers -------------------------------------------
    def touched_rows(self, inputs: Dict[str, torch.Tensor]) -> torch.Tensor:
        """LOCAL rows a step on the current inputs of ALL ranks updates on this rank (collective)."""
        groups = []
        for ids, cols in self._column_ids(inputs):
            ids = ids.contiguous()
            everyone = [torch.empty_like(ids) for _ in range(self.world)]
            dist.all_gather(everyone, ids, group=self.group)
            groups.append((torch.cat(everyone), cols))
        return self.store.touched_rows(groups)

    def restore(self, snap):
        super().restore(snap)
        torch.cuda.synchronize(self.dev)
        dist.barrier(group=self.group)                           # nobody gathers rows a peer is still restoring

    def gather_global_table(self) -> torch.Tensor:
        """[sum(rows), d] table in the unsharded arena order, on every rank (tests / small tables only)."""
        mine = self.table.contiguous()
        shards = [torch.empty_like(mine) for _ in range(self.world)]
        dist.all_gather(shards, mine, group=self.group)
        out = torch.empty(self.store.total_rows, self.d, device=self.dev)
        for r in range(self.world):
            for g, loc in field_slices(self.rows, self.world, r):
                out[g] = shards[r][loc]
        return out
