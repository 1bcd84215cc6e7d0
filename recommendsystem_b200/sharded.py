"""Multi-GPU AutoInt: data-parallel dense part, embedding tables row-sharded across the ranks of one NVSwitch domain
(one process per GPU, at most RS_MAX_PEERS = 8 of them, NCCL).

    owner(row) = row mod W ; local row = local_base[f] + row div W         (SURVEY.md §8e)

Every rank maps every rank's table shard into its address space (CUDA IPC) and reads the rows it needs straight out of
the owners' HBM over NVLink / NVSwitch (rs_embed_gather_peer_fwd, or the fused InteractingLayer forward).  The owners
still need the (row, position) keys of what was read for the backward's sorted-segment update: the ids are routed into
fixed-capacity buckets (rs_route_ids_padded), exchanged by one NCCL all-to-all and turned into sorted keys — on a
side stream, hidden behind the dense forward.  The backward pushes the gradient rows into the owners' receive buffers
with peer stores (rs_scatter_rows_peer, or the fused InteractingLayer backward).  Two flag barriers over peer memory
(rs_peer_barrier) order things: stores before the owners' reads, and every owner's sparse update before the next
step's peer reads.  Dense gradients: one flat all-reduce (average) before the dense Adam.

Buckets have a fixed capacity, so there is no host round trip for the counts and the whole
step — collectives included — is one CUDA graph.  A bucket overflow (skewed ids) sets a device
flag that `check_overflow()` turns into an exception; nothing is silently dropped.

`PeerArena` and `Buckets` are this exchange, shared by ShardedAutoIntTrainer and api.sharded_embedding.
ShardedEmbeddingFeatures.  This replaces TensorNet's sparse pull/push (only trace in the reference:
tn.core.shard_num() / self_shard_id(), staytime/parse.py:78-79).  The collective plumbing lives in `Exchange`, which
is device-agnostic so that the protocol is tested on CPU with the gloo backend.
"""
from __future__ import annotations

import ctypes
import math
from contextlib import contextmanager

import torch
import torch.distributed as dist

from . import cabi, ops
from .arena import INIT_CHUNK_ROWS, check_sharded_id_map, shard_layout  # noqa: F401  (shard_layout: re-exported)
from .autoint import AutoIntConfig, AutoIntTrainer


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
    """The collectives of a sharded step: all-to-all of equal splits, mean all-reduce."""

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


class PeerArena:
    """The peer-memory side of one row-sharded arena (arena.Arena `store` on every rank of `ex`'s group): every rank's
    table shard mapped into this process, the flag array of the cross-rank barrier and the bucket-overflow flag.
    Collective at construction."""

    def __init__(self, store, ex: Exchange):
        backend = dist.get_backend(ex.group)
        if backend != "nccl" or ex.world > cabi.RS_MAX_PEERS:
            raise ValueError(f"row-sharded tables are read and updated over peer memory: they need an NCCL group of at "
                             f"most {cabi.RS_MAX_PEERS} GPUs (one NVSwitch domain), not {ex.world} ranks on {backend}")
        self.store, self.ex = store, ex
        self.world, self.rank, self.dev = ex.world, ex.rank, store.dev
        self._opened = {}
        self.tables = self.map(store.w)
        self.flags = torch.zeros(cabi.RS_MAX_PEERS + 1, dtype=torch.int32, device=self.dev)   # a slot per rank + epoch
        self.overflow = torch.zeros(1, dtype=torch.int32, device=self.dev)
        torch.cuda.synchronize(self.dev)            # the flags are zero before any peer stores into them
        self.peer_flags = self.map(self.flags)

    def map(self, tensor):
        """Every rank's copy of `tensor`, mapped into this process: a host array of W device pointers (collective)."""
        return map_peer_buffers(tensor, self.world, self.rank, self.ex.group, self._opened)

    def barrier(self):
        """Cross-rank barrier on the current stream: a flag kernel over peer memory; every rank's earlier writes (peer
        stores included) are visible to the others once they leave it."""
        cabi.call("rs_peer_barrier", ctypes.addressof(self.peer_flags), self.world, self.rank, ops._stream())

    def check_overflow(self):
        """Raise if any routing bucket ever exceeded its capacity (ids too skewed for the bucket capacity)."""
        if int(self.overflow.item()) != 0:
            raise RuntimeError("routing bucket overflow: some owner received more lookups from one rank than a bucket "
                               "holds; the step's result is invalid — re-create it with a larger capacity_factor")


class Buckets:
    """The exchange of one lookup group: `n` lookups of the fields `cols` (ids int64 [n / len(cols), len(cols)], < 0 =
    padding) in fixed-capacity (source, owner) buckets, and the gradient receive buffer (`dtype` rows), mapped on every
    rank.  Every operation launches on the current stream.  `capacity` pins the slots per bucket exactly; otherwise
    bucket_capacity(n, W, capacity_factor).  `pad_spread`: padding ids take a slot at owner hash(i) mod W instead of
    owner 0 (groups that are mostly padding keep balanced buckets).  Collective at construction."""

    def __init__(self, peers: PeerArena, cols, n: int, dtype, capacity_factor=None, capacity=None, pad_spread=False):
        W, dev, d = peers.world, peers.dev, peers.store.d
        self.peers, self.n, self.F, self.pad_spread = peers, int(n), len(cols), bool(pad_spread)
        self.lbase_t, self.rows_t = peers.store.geom(cols)
        self.cap = int(capacity) if capacity is not None else bucket_capacity(self.n, W, capacity_factor)
        self.send_rows = torch.empty(W * self.cap, dtype=torch.int32, device=dev)
        self.recv_rows = torch.empty(W * self.cap, dtype=torch.int32, device=dev)
        self.inverse = torch.empty(self.n, dtype=torch.int32, device=dev)
        self.send_counts = torch.empty(W, dtype=torch.int32, device=dev)
        self.keys = torch.empty(W * self.cap, dtype=torch.int64, device=dev)
        self.keys_sorted = torch.empty_like(self.keys)
        self.g_recv = torch.zeros(W * self.cap, d, dtype=dtype, device=dev)
        torch.cuda.synchronize(dev)
        self.peer_grecv = peers.map(self.g_recv)

    def gather(self, ids, out):
        """out [n / F, F, d] = the rows of `ids`, read from the owners' shards (bit-exact with the unsharded gather)."""
        p = self.peers
        cabi.call("rs_embed_gather_peer_fwd", ctypes.addressof(p.tables), p.store.ld, p.world, ids.data_ptr(),
                  self.lbase_t.data_ptr(), self.rows_t.data_ptr(), self.n, self.F, p.store.d, out.data_ptr(),
                  ops._dt(out), ops._stream())

    # ---- the owners' keys for the backward: route -> all-to-all(ids) -> sorted keys
    def route(self, ids):
        """The lookups of `ids` into the send buckets; `inverse` = every lookup's slot (owner * cap + k)."""
        p = self.peers
        ops.route_ids_padded(ids, self.F, self.rows_t, self.lbase_t, p.world, self.cap, self.send_rows, self.inverse,
                             self.send_counts, p.overflow, pad_spread=self.pad_spread)

    def exchange_ids(self):
        self.peers.ex.all_to_all(self.recv_rows, self.send_rows)

    def sort_keys(self):
        """keys_sorted: the owner's received rows as (row << 32 | slot) sort keys, sorted."""
        cabi.call("rs_embed_keys_from_rows", self.recv_rows.data_ptr(), self.recv_rows.numel(), self.keys.data_ptr(),
                  ops._stream())
        ops.sort_keys(self.keys, self.peers.store.row_bits, out=self.keys_sorted)

    def owner_keys(self, ids):
        self.route(ids)
        self.exchange_ids()
        self.sort_keys()

    # ---- backward: push -> barrier -> update -> barrier
    def push(self, grad):
        """Store this rank's gradient rows (grad [n, d] in the lookups' order) into the owners' receive buffers."""
        p = self.peers
        cabi.call("rs_scatter_rows_peer", grad.data_ptr(), ctypes.addressof(self.peer_grecv), p.world, p.rank,
                  self.inverse.data_ptr(), self.n, self.cap, grad.shape[-1] * grad.element_size(), ops._stream())

    def scatter_args(self):
        """(address of the W receive-buffer pointers, W, rank, inverse, cap): the push fused into
        rs_interacting_bwd_scatter."""
        p = self.peers
        return ctypes.addressof(self.peer_grecv), p.world, p.rank, self.inverse.data_ptr(), self.cap

    def update(self, step):
        """The owner's sparse update: step(received gradient rows, sorted keys, grad_scale).  Every rank's loss is the
        mean over its own batch: grad_scale = 1/W makes the update that of the global batch."""
        step(self.g_recv, self.keys_sorted, grad_scale=1.0 / self.peers.world)


class ShardedAutoIntTrainer(AutoIntTrainer):
    """AutoIntTrainer whose tables are row-sharded over the ranks of `group`.  `cfg.batch` is the
    PER-RANK batch (weak scaling); the loss each rank reports is the mean over its own batch and
    gradients are averaged over ranks, i.e. the update is that of the global batch W * batch."""

    def __init__(self, cfg: AutoIntConfig, device, group=None, global_tables: torch.Tensor | None = None,
                 dense_init: dict | None = None, capacity_factor: float | None = None, capacity: int | None = None):
        check_sharded_id_map(cfg.id_map)          # before any collective
        if any(k > 1 for k in cfg.bags()):
            # the fused gradient push sends one row per (sample, field): bags would need one per slot
            raise ValueError("row-sharded bag fields are not built")
        self.ex = Exchange(group)
        self.world, self.rank = self.ex.world, self.ex.rank
        super().__init__(cfg, device, tables=global_tables, dense_init=dense_init)
        self.local_rows, self.local_base, self.lbase_t = self.store.local_rows, self.store.local_base, self.store.lbase_t
        self.peers = PeerArena(self.store, self.ex)
        # `capacity` pins the slots per (source, owner) bucket exactly (tests: buckets filled to the brim, forced overflow)
        self.buckets = Buckets(self.peers, self.fields, cfg.batch * cfg.num_fields, self.act_dtype, capacity_factor,
                               capacity)
        self.side2 = torch.cuda.Stream(device=self.dev)       # the owners' keys, then the update barrier
        self.route_done = torch.cuda.Event()
        self.inverse_done = torch.cuda.Event()

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
    def _launch_step(self):
        super()._launch_step()
        torch.cuda.current_stream(self.dev).wait_stream(self.side2)     # the update barrier (_embed_backward)

    def _lookup_args(self):
        return ctypes.addressof(self.peers.tables), self.world, self.lbase_t, None      # the owners make the keys

    def _scatter_args(self):
        return self.buckets.scatter_args()

    def _interacting_bwd_fused(self, dparams, st, T, main):
        main.wait_event(self.inverse_done)          # this step's slots (rs_route_ids_padded on the side stream)
        super()._interacting_bwd_fused(dparams, st, T, main)

    @contextmanager
    def _backward_keys(self, ph):
        """The owners' view of the step: routing, id all-to-all and key sort need only the ids, so they run on a side
        stream that forks BEFORE the forward; the peer reads need none of it."""
        b = self.buckets
        self.side2.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(self.side2):
            with ph("route_ids"):
                b.route(self.ids)
            self.inverse_done.record(self.side2)
            self._stamp("owners_route_end")
            with ph("a2a_ids"):
                b.exchange_ids()
            self._stamp("owners_a2a_ids_end")
            with ph("sort_keys"):
                b.sort_keys()
            self.route_done.record(self.side2)
            self._stamp("owners_sort_end")
        yield

    def _embed_forward(self, ph, st, T):
        with ph("embed_gather_peer"):
            self.buckets.gather(self.ids, self.X)

    def _embed_backward(self, ph, st, T, main):
        if not self.fused:                 # (fused: the InteractingLayer backward already stored the rows)
            main.wait_event(self.inverse_done)
            with ph("scatter_grads_peer"):
                self.buckets.push(self.dX)
        with ph("peer_barrier"):           # every rank's stores have landed
            self.peers.barrier()
        self._stamp("push_barrier_end")
        # the owners' sorted keys of this step (side stream: behind the forward it often finishes only now, while
        # the barrier above — which does not need them — is already under way)
        main.wait_event(self.route_done)
        with ph("embed_segsum_adam"):
            self.buckets.update(self._sparse_update)
        # cross-rank barrier: every owner's update is complete before any rank's next peer gather; runs beside the
        # dense Adam and joins the step at its end (_launch_step)
        self.side2.wait_stream(main)
        with torch.cuda.stream(self.side2):
            with ph("peer_barrier_end"):
                self.peers.barrier()
            self._stamp("update_barrier_end")

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
        self.peers.overflow.zero_()
        torch.cuda.synchronize(self.dev)
        dist.barrier(group=self.ex.group)
        return g

    def _predict_lookup(self, st, T):
        """The peer gather, never the local shard with global row numbers."""
        self.buckets.gather(self.ids, self.X)

    def evaluate(self, batches, num_thresholds: int = 200, threshold: float = 0.5) -> dict:
        """AutoIntTrainer.evaluate over this rank's `batches`, collective: every rank calls it with its own stream (the
        number of batches, zero included, may differ) and every rank returns the metrics and mean loss of all of them.

        The eval step reads rows straight from the owners' shards (the fused loader over the peer table pointers, or
        the peer gather) and needs no routing, id exchange or barrier: this rank's last train step ended behind the
        update barrier (every owner's update of that step is complete), and no owner updates a row again before its
        next train step's push barrier, which every rank enters only after the eval launches queued before it."""
        return super().evaluate(batches, num_thresholds, threshold)

    def _eval_reduce(self, ev, totals):
        """One all-reduce (sum) of every rank's metric state and [loss sum, count].  The integer words travel as
        float64, exact below 2^53; NCCL hands every rank the same sums, so every rank returns the same dict."""
        T = ev["metrics"].num_thresholds
        state = ev["metrics"].state
        n_int = 2 * T + 4                    # integer words; the last two hold float64 bit patterns
        buf = torch.cat([state[:n_int].double(), state[n_int:].view(torch.float64), totals])
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=self.ex.group)
        state[:n_int].copy_(buf[:n_int].to(torch.int64))
        state[n_int:].view(torch.float64).copy_(buf[n_int:n_int + 2])
        totals.copy_(buf[n_int + 2:])

    def check_overflow(self):
        """Raise if any routing bucket ever exceeded its capacity (ids too skewed for `capacity_factor`)."""
        self.peers.check_overflow()
