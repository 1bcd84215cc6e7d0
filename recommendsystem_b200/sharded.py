"""Multi-GPU AutoInt: data-parallel dense part, embedding tables row-sharded across the ranks,
ids / rows / gradients exchanged by NCCL all-to-all over NVLink (one process per GPU).

    owner(row) = row mod W ; local row = local_base[f] + row div W         (SURVEY.md §8e)

    ids [b,F] --route (K7, fixed-capacity buckets)--> all-to-all(ids) --> owner gathers (K1)
        --> all-to-all(rows) --> un-permute --> X [b,F,d] --> dense step (as on one GPU) --> dX
        --> permute --> all-to-all(grads) --> owner: sort + segment-sum + sparse Adam (K3)
    dense gradients: one flat all-reduce (average) before the dense Adam.

`peer_gather=True` (default on NCCL) replaces the forward half by ONE kernel that reads the rows it
needs straight out of the owners' HBM over NVLink / NVSwitch (CUDA-IPC mappings of every rank's shard,
rs_embed_gather_peer_fwd): no id all-to-all, owner gather, row all-to-all or un-permute on the critical
path.  The routing + id all-to-all still run — on a side stream, hidden behind the dense forward — because
the owners need the (row, position) keys for the backward's sorted-segment update.  The backward pushes the
gradient rows into the owners' receive buffers with peer stores (rs_scatter_rows_peer).  Two flag barriers over
peer memory (rs_peer_barrier) order things: stores before the owners' reads, and every owner's sparse update
before the next step's peer reads.

Buckets have a fixed capacity, so there is no host round trip for the counts and the whole
step — collectives included — is one CUDA graph.  A bucket overflow (skewed ids) sets a device
flag that `check_overflow()` turns into an exception; nothing is silently dropped.

This replaces TensorNet's sparse pull/push (only trace in the reference: tn.core.shard_num() /
self_shard_id(), staytime/parse.py:78-79).  The collective plumbing lives in `Exchange`, which
is device-agnostic so that the protocol is tested on CPU with the gloo backend.
"""
from __future__ import annotations

import ctypes
import os
import math

import torch
import torch.distributed as dist

from . import cabi, ops
from .arena import INIT_CHUNK_ROWS, check_sharded_id_map, shard_layout  # noqa: F401  (shard_layout: re-exported)
from .autoint import AutoIntConfig, AutoIntTrainer, _Phase


def bucket_capacity(n_lookups: int, world: int, factor: float | None = None) -> int:
    """Slots per (source, owner) pair.  Default: mean + 8 sigma of a uniform multinomial + 64,
    rounded up to 128 (overflow probability for uniform ids < 1e-14 per bucket)."""
    mean = n_lookups / world
    if factor is not None:
        cap = mean * factor
    else:
        cap = mean + 8.0 * math.sqrt(max(mean * (1 - 1.0 / world), 1.0)) + 64
    return min(n_lookups, int(math.ceil(cap / 128.0) * 128))


def map_peer_buffers(tensor, world, rank, group, opened):
    """Exchange CUDA-IPC handles of `tensor` (one per rank of `group`) and map every rank's copy into this process.
    Returns a ctypes array of `world` device pointers (a kernel argument).  `opened` caches the imported allocations
    (an allocation may be opened once per process).  Collective, host-synchronising: setup time only."""
    handle = (ctypes.c_ubyte * 64)()
    off = ctypes.c_ulonglong(0)
    cabi.call("rs_ipc_export", tensor.data_ptr(), ctypes.addressof(handle), ctypes.addressof(off))
    everyone = [None] * world
    dist.all_gather_object(everyone, (bytes(handle), int(off.value)), group=group)
    ptrs = (ctypes.c_void_p * world)()
    for r, (h, o) in enumerate(everyone):
        if r == rank:
            ptrs[r] = tensor.data_ptr()
            continue
        if (r, h) not in opened:
            hb = (ctypes.c_ubyte * 64).from_buffer_copy(h)
            base = ctypes.c_void_p(0)
            cabi.call("rs_ipc_import", ctypes.addressof(hb), 0, ctypes.addressof(base))
            opened[(r, h)] = base.value
        ptrs[r] = opened[(r, h)] + o
    dist.barrier(group=group)
    return ptrs


class Exchange:
    """The three all-to-alls of a sharded step (equal splits of `cap` slots per peer)."""

    def __init__(self, group=None):
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)

    def all_to_all(self, out: torch.Tensor, inp: torch.Tensor):
        dist.all_to_all_single(out, inp, group=self.group)
        return out

    def all_reduce_mean(self, t: torch.Tensor):
        if dist.get_backend(self.group) == "nccl":
            dist.all_reduce(t, op=dist.ReduceOp.AVG, group=self.group)
        else:   # gloo has no AVG
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
            t.div_(self.world)
        return t


class ShardedAutoIntTrainer(AutoIntTrainer):
    """AutoIntTrainer whose tables are row-sharded over the ranks of `group`.  `cfg.batch` is the
    PER-RANK batch (weak scaling); the loss each rank reports is the mean over its own batch and
    gradients are averaged over ranks, i.e. the update is that of the global batch W * batch."""

    def __init__(self, cfg: AutoIntConfig, device, group=None, global_tables: torch.Tensor | None = None,
                 dense_init: dict | None = None, capacity_factor: float | None = None,
                 peer_gather: bool | None = None, capacity: int | None = None, peer_ids: bool | None = None):
        check_sharded_id_map(cfg.id_map)          # before any collective
        self.ex = Exchange(group)
        self.world, self.rank = self.ex.world, self.ex.rank
        self._capacity_factor = capacity_factor
        super().__init__(cfg, device, tables=global_tables, dense_init=dense_init)
        self.local_rows, self.local_base, self.lbase_t = self.store.local_rows, self.store.local_base, self.store.lbase_t
        W, n, d = self.world, cfg.batch * cfg.num_fields, cfg.embed_dim
        # `capacity` pins the slots per (source, owner) bucket exactly (tests: buckets filled to the brim, forced overflow)
        self.cap = int(capacity) if capacity is not None else bucket_capacity(n, W, capacity_factor)
        T = self.act_dtype
        dev = self.dev
        self.send_rows = torch.empty(W * self.cap, dtype=torch.int32, device=dev)
        self.recv_rows = torch.empty(W * self.cap, dtype=torch.int32, device=dev)
        self.inverse = torch.empty(n, dtype=torch.int32, device=dev)
        self.send_counts = torch.empty(W, dtype=torch.int32, device=dev)
        self.overflow = torch.zeros(1, dtype=torch.int32, device=dev)
        self.rows_out = torch.empty(W * self.cap, d, dtype=T, device=dev)      # gathered for the peers
        self.rows_in = torch.empty(W * self.cap, d, dtype=T, device=dev)       # received for my lookups
        self.g_send = torch.empty(W * self.cap, d, dtype=T, device=dev)
        self.g_recv = torch.empty(W * self.cap, d, dtype=T, device=dev)
        self.keys = torch.empty(W * self.cap, dtype=torch.int64, device=dev)
        self.keys_sorted = torch.empty_like(self.keys)
        if peer_gather is None:
            peer_gather = dist.get_backend(group) == "nccl" and W <= 8
        self.peer_gather = bool(peer_gather)
        # peer_ids: the routed ids reach their owners by peer stores + a flag barrier (rs_peer_all_to_all_i32, 16 us)
        # instead of a NCCL all-to-all (38 us).  Opt-in (argument, or RS_PEER_IDS=1): at W = 2 the owners' key sort
        # still ends with the backward either way (it shares the tower's window with the GEMMs), the step gains 3 us,
        # and only W = 2 was run; the NCCL exchange is the one proven at W = 8.
        if peer_ids is None:
            peer_ids = os.environ.get("RS_PEER_IDS", "0") == "1"
        self.peer_ids = bool(peer_ids) and self.peer_gather
        if self.peer_gather:
            self._map_peer_tables(group)
            self.side2 = torch.cuda.Stream(device=dev)
            self.route_done = torch.cuda.Event()
            self.inverse_done = torch.cuda.Event()
        else:
            self.fused = False                       # the all-NCCL path keeps the separate gather / scatter kernels

    def _map_peers(self, tensor, group):
        """Exchange CUDA-IPC handles of `tensor` (one per rank) and map every rank's copy into this process;
        returns a host array of W device pointers (a kernel argument)."""
        if not hasattr(self, "_ipc_opened"):
            self._ipc_opened = {}
        return map_peer_buffers(tensor, self.world, self.rank, group, self._ipc_opened)

    def _map_peer_tables(self, group):
        self.peer_ptrs = self._map_peers(self.table, group)          # every rank's table shard
        self.peer_grecv = self._map_peers(self.g_recv, group)         # every rank's gradient receive buffer
        self.flags = torch.zeros(16, dtype=torch.int32, device=self.dev)   # RS_MAX_PEERS slots + the epoch
        torch.cuda.synchronize(self.dev)
        self.peer_flags = self._map_peers(self.flags, group)
        if self.peer_ids:
            self.peer_recv_rows = self._map_peers(self.recv_rows, group)  # every rank's routed-id receive buffer
            # its barrier runs on the owners' side stream, unordered with the main stream's push barrier: own flags
            self.flags_ids = torch.zeros(16, dtype=torch.int32, device=self.dev)
            torch.cuda.synchronize(self.dev)
            self.peer_flags_ids = self._map_peers(self.flags_ids, group)

    def _barrier(self, ph, name):
        """Cross-rank barrier on the current stream: a flag kernel over peer memory (rs_peer_barrier)."""
        with ph(name):
            cabi.call("rs_peer_barrier", ctypes.addressof(self.peer_flags), self.world, self.rank, ops._stream())

    def _arena_shard(self):
        return self.world, self.rank

    def _init_tables(self, tables):
        """This rank's rows of the global tables given (parity tests), or its own N(0, table_init_scale) draw in local
        row order from seed + 7919 rank (not the single-GPU trainer's tables)."""
        if tables is not None:
            return super()._init_tables(tables)
        gen = torch.Generator(device=self.dev).manual_seed(self.cfg.seed + 7919 * self.rank)
        n_local, d = self.store.n_local, self.cfg.embed_dim
        for r0 in range(0, n_local, INIT_CHUNK_ROWS):
            r1 = min(n_local, r0 + INIT_CHUNK_ROWS)
            self.table[r0:r1] = torch.empty(r1 - r0, d, device=self.dev).normal_(0.0, self.cfg.table_init_scale,
                                                                                 generator=gen)

    # ---- embedding halves of the step -----------------------------------------------------
    def _lookup_args(self):
        return ctypes.addressof(self.peer_ptrs), self.world, self.lbase_t, None      # the owners make the keys

    def _scatter_args(self):
        return ctypes.addressof(self.peer_grecv), self.world, self.rank, self.inverse.data_ptr(), self.cap

    def _interacting_bwd_fused(self, dparams, st, T, main):
        main.wait_event(self.inverse_done)          # this step's slots (rs_route_ids_padded on the side stream)
        super()._interacting_bwd_fused(dparams, st, T, main)

    def _embed_forward(self, ph, st, T, gather=True):
        c = self.cfg
        F, d = c.num_fields, c.embed_dim
        if not gather and not self.peer_gather:
            raise RuntimeError("the fused lookup needs peer_gather=True (rows are read from the owners' HBM)")
        if self.peer_gather:
            main = torch.cuda.current_stream(self.dev)
            # owners' view of the step (keys for the backward): routing, id all-to-all, key sort — all on a
            # side stream; the peer reads below need none of it
            self.side2.wait_stream(main)
            with torch.cuda.stream(self.side2):
                with ph("route_ids"):
                    ops.route_ids_padded(self.ids, F, self.rows_t, self.lbase_t, self.world, self.cap, self.send_rows,
                                         self.inverse, self.send_counts, self.overflow)
                self.inverse_done.record(self.side2)
                self._stamp("owners_route_end")
                with ph("a2a_ids"):
                    if self.peer_ids:
                        cabi.call("rs_peer_all_to_all_i32", self.send_rows.data_ptr(), ctypes.addressof(self.peer_recv_rows),
                                  self.world, self.rank, self.cap, ops._stream())
                        cabi.call("rs_peer_barrier", ctypes.addressof(self.peer_flags_ids), self.world, self.rank,
                                  ops._stream())
                    else:
                        self.ex.all_to_all(self.recv_rows, self.send_rows)
                self._stamp("owners_a2a_ids_end")
                with ph("sort_keys"):
                    cabi.call("rs_embed_keys_from_rows", self.recv_rows.data_ptr(), self.recv_rows.numel(),
                              self.keys.data_ptr(), ops._stream())
                    ops.sort_keys(self.keys, self.row_bits, out=self.keys_sorted)
                self.route_done.record(self.side2)
                self._stamp("owners_sort_end")
            if not gather:
                return
            with ph("embed_gather_peer"):
                cabi.call("rs_embed_gather_peer_fwd", ctypes.addressof(self.peer_ptrs), self.table_ld, self.world,
                          self.ids.data_ptr(), self.lbase_t.data_ptr(), self.rows_t.data_ptr(),
                          c.batch * F, F, d, self.X.data_ptr(), T, st)
            return
        with ph("route_ids"):
            ops.route_ids_padded(self.ids, F, self.rows_t, self.lbase_t, self.world, self.cap, self.send_rows,
                                 self.inverse, self.send_counts, self.overflow)
        with ph("a2a_ids"):
            self.ex.all_to_all(self.recv_rows, self.send_rows)
        with ph("embed_gather"):
            cabi.call("rs_embed_gather_rows_ld", self.table.data_ptr(), self.table_ld, self.recv_rows.data_ptr(),
                      self.recv_rows.numel(), d, self.rows_out.data_ptr(), T, None, self.keys.data_ptr(), st)
        with ph("a2a_rows"):
            self.ex.all_to_all(self.rows_in, self.rows_out)
        with ph("unpermute"):
            ops.permute_rows(self.rows_in, self.inverse, scatter=False, out=self.X.view(-1, d))

    def _sort_keys(self, ph):
        if not self.peer_gather:            # peer mode sorts on its own side stream (see _embed_forward)
            super()._sort_keys(ph)

    def _embed_backward(self, ph, st, T, main):
        c = self.cfg
        d = c.embed_dim
        if self.peer_gather:
            # gradient rows go straight into the owners' receive buffers (peer stores over NVLink): the permute
            # and the all-to-all in one kernel; a flag barrier separates the stores from the owners' reads
            if not self.fused:                 # (fused: the InteractingLayer backward already stored the rows)
                main.wait_event(self.inverse_done)
                with ph("scatter_grads_peer"):
                    row_bytes = d * self.dX.element_size()
                    cabi.call("rs_scatter_rows_peer", self.dX.data_ptr(), ctypes.addressof(self.peer_grecv), self.world,
                              self.rank, self.inverse.data_ptr(), c.batch * c.num_fields, self.cap, row_bytes, st)
            self._barrier(ph, "peer_barrier")
            self._stamp("push_barrier_end")
            # the owners' sorted keys of this step (side stream: behind the forward it often finishes only now, while
            # the barrier above — which does not need them — is already under way)
            main.wait_event(self.route_done)
        else:
            with ph("permute_grads"):
                self.g_send.zero_()
                ops.permute_rows(self.dX.view(-1, d), self.inverse, scatter=True, out=self.g_send)
            with ph("a2a_grads"):
                self.ex.all_to_all(self.g_recv, self.g_send)
        if not self.peer_gather:
            main.wait_event(self.sort_done)    # sorted keys (the dense all-reduce / Adam stay on the side stream)
        with ph("embed_segsum_adam"):
            # local losses are means over the local batch: 1/W makes it the global-batch mean
            ops.segsum_adam(self.table, self.table_m, self.table_v, self.g_recv, self.keys_sorted, c.lr_sparse,
                            c.beta1, c.beta2, c.eps, self.adam_scalars, grad_scale=1.0 / self.world)
        if self.peer_gather:
            # cross-rank barrier: every owner's update is complete before any rank's next peer gather;
            # runs beside the dense Adam
            self.side2.wait_stream(main)
            with torch.cuda.stream(self.side2):
                self._barrier(ph, "peer_barrier_end")
                self._stamp("update_barrier_end")
            self._join_side2 = True

    def _dense_sync(self, ph):
        self._stamp("allreduce_begin")
        with ph("allreduce_dense"):
            self.ex.all_reduce_mean(self.flat_g)
        self._stamp("allreduce_end")

    def _touched_rows(self) -> torch.Tensor:
        """LOCAL arena rows the step on the current static id buffers of ALL ranks updates on this rank."""
        everyone = [torch.empty_like(self.ids) for _ in range(self.world)]
        dist.all_gather(everyone, self.ids, group=self.ex.group)
        return self.store.touched_rows([(torch.cat(everyone, 0), self.fields)])

    def capture(self):
        """Capture the sharded step (collectives included).  The warm-up launch runs on whatever the static id
        buffer holds (zeros unless the caller filled it), which may legitimately overflow the buckets; the flag is
        cleared afterwards so it reports real steps only.  As in the single-GPU trainer the warm-up's optimizer
        step is undone (every rank restores the rows it owns); a barrier keeps any rank from gathering rows of a
        peer that is still restoring."""
        g = super().capture()
        self.overflow.zero_()
        torch.cuda.synchronize(self.dev)
        dist.barrier(group=self.ex.group)
        return g

    def _predict_lookup(self, st, T):
        """The sharded gather (_embed_forward: peer reads, or route + all-to-alls), never the local shard with global
        row numbers."""
        self._embed_forward(lambda name: _Phase(None, name), st, T)
        if self.peer_gather:       # the owners' key work of _embed_forward is not needed here
            torch.cuda.current_stream(self.dev).wait_stream(self.side2)

    def check_overflow(self):
        """Raise if any routing bucket ever exceeded its capacity (ids too skewed for `capacity_factor`)."""
        if int(self.overflow.item()) != 0:
            raise RuntimeError(f"routing bucket overflow: some owner received more than {self.cap} lookups from "
                               "one rank; the step's result is invalid — re-create the trainer with a larger "
                               "capacity_factor")
