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

The exchange itself (peer mappings, buckets, barriers) is sharded.PeerArena / sharded.Buckets, the same as the
sharded AutoInt trainer's.  Everything is launched on the current stream with fixed buffers: the whole train step —
collectives included — is CUDA-graph capturable (api.graph.GraphedTrainStep).  Buckets of a column group are created at
its first use (collective: every rank runs the same model code), i.e. during the eager warm-up steps, never during
capture.
"""
from __future__ import annotations

from typing import Dict, List

import torch
import torch.distributed as dist

from .. import ops
from ..arena import check_sharded_id_map, field_slices
from ..sharded import Buckets, Exchange, PeerArena
from .embedding import Adam, EmbeddingColumn, EmbeddingFeatures


class ShardedEmbeddingFeatures(EmbeddingFeatures):
    def __init__(self, embedding_columns: List[EmbeddingColumn], sparse_opt, name="embedding", device="cuda:0",
                 out_dtype=torch.float32, seed=0, group=None, capacity_factor=None, id_map="mod"):
        check_sharded_id_map(id_map)
        if not dist.is_initialized():
            raise RuntimeError("ShardedEmbeddingFeatures needs torch.distributed (one process per GPU)")
        self.group = group
        ex = Exchange(group)
        self.world, self.rank = ex.world, ex.rank
        self.capacity_factor = capacity_factor
        self._groups: Dict[tuple, Buckets] = {}
        super().__init__(embedding_columns, sparse_opt, name, device, out_dtype, seed, id_map)
        self.peers = PeerArena(self.store, ex)

    # this rank's rows of every column hold the same values as the unsharded layer with the same seed
    def _arena_shard(self):
        return self.world, self.rank

    # ---- exchange buckets ------------------------------------------------------------------------------------
    def _group(self, gkey, n, cols, padded=False) -> Buckets:
        g = self._groups.get((gkey, n))
        if g is None:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("a column group met a new batch shape during CUDA-graph capture: run one eager step "
                                   "first")
            # Groups that may carry padding (sequence / bag columns) spread it over the owners by a hash of the lookup
            # index (rs_route_ids_padded_spread): the buckets stay balanced and the usual capacity holds.
            g = self._groups[(gkey, n)] = Buckets(self.peers, cols, n, torch.float32, self.capacity_factor,
                                                  pad_spread=padded)
        return g

    def _lookup(self, gkey, ids: torch.Tensor, cols, padded=False) -> torch.Tensor:
        """ids int64 [N, len(cols)] (id < 0 = padding) -> fp32 [N, len(cols), d]; registers the owners' keys."""
        ids = ids.contiguous()
        g = self._group(gkey, ids.numel(), tuple(cols), padded)
        out = torch.empty(ids.shape[0], g.F, self.d, dtype=torch.float32, device=self.dev)
        g.gather(ids, out)
        g.owner_keys(ids)
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
        self._pending_backward = torch.is_grad_enabled()
        return out

    def backward(self, grads: Dict[str, torch.Tensor]):
        """Push d(loss)/d(output) of every column to the owners: peer stores -> barrier -> owner-local sorted-segment
        sum + optimizer (grad_scale 1/W) -> barrier."""
        if self._last is None:
            raise RuntimeError("EmbeddingFeatures.backward called before a forward")
        for key, g, bag in self._last:
            gr = torch.stack([grads[k] for k in key], dim=1) if isinstance(key, list) else grads[key]
            if isinstance(gr, tuple):
                gr = gr[0]
            gr = gr.reshape(-1, self.d).float()
            if bag is not None:
                b, cnt = bag
                gr = (gr / cnt[:, None]).repeat_interleave(b, dim=0)
            g.push(gr.contiguous())
        self.peers.barrier()                                     # every rank's stores have landed
        if isinstance(self.opt, Adam):
            ops.adam_advance(self.scalars, self.opt.beta1, self.opt.beta2)
        for key, g, bag in self._last:
            g.update(self._sparse_update)
        self.peers.barrier()                                     # every owner's update precedes the next peer reads
        self._last = None
        self._pending_backward = False

    def check_overflow(self):
        self.peers.check_overflow()

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
