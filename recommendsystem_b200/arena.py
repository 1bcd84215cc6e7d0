"""The embedding arena: the tables of one set of fields and their sparse-optimizer state, as one array on one rank.

This module is the only code that knows the arena's layout (DESIGN.md §2):
    field f owns R_f rows; row_base = exclusive cumsum of R
    mod mode     global row = row_base[f] + id mod R_f
    W ranks      owner = (id mod R_f) mod W ; local row = local_base[f] + (id mod R_f) div W,
                 each rank holding ceil(R_f / W) rows of every field (shard_layout); W = 1 is the unsharded arena
    storage      Adam: one [w | m | v] record of 3d floats per row (the sparse update touches ONE contiguous block
                 per row); AdaGrad: w [n, d] and g2sum [n] or [n, d]
    hash mode    (recommendsystem_b200.idmap, one rank only) ids are first mapped to rows, which the kernels read
                 through the identity geometry (row_base 0, rows = total rows)
The arena issues no collective: the sharded classes gather the ids of every rank before asking it for touched rows.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops

INIT_CHUNK_ROWS = 1 << 22        # the initial draw goes through temporaries of at most this many rows


def shard_layout(rows_per_field, world: int = 1):
    """(local_rows[F], local_base[F]) of every rank of a `world`-way row-sharded arena: ceil(R_f / W) rows of field f
    per rank.  At W = 1: (rows, row_base)."""
    rows = np.asarray(rows_per_field, np.int64)
    local_rows = (rows + world - 1) // world
    local_base = np.concatenate([[0], np.cumsum(local_rows)[:-1]]).astype(np.int64)
    return local_rows, local_base


def field_slices(rows_per_field, world: int, rank: int):
    """Per field, (global slice, local slice): the rows of the global arena that rank `rank` of a `world`-way arena
    holds (global rows row_base[f] + rank, + rank + W, ...), and where they lie in its shard."""
    rows = np.asarray(rows_per_field, np.int64)
    _, base = shard_layout(rows, 1)
    _, local_base = shard_layout(rows, world)
    for R, b, lb in zip(rows.tolist(), base.tolist(), local_base.tolist()):
        n = len(range(rank, R, world))
        yield slice(b + rank, b + R, world), slice(lb, lb + n)


def check_sharded_id_map(id_map: str):
    """Row-sharded arenas support id_map='mod' only."""
    if id_map != "mod":
        # the owners would have to map the routed ids before the peers read rows by index: not built yet
        raise NotImplementedError("row-sharded tables support id_map='mod' only (row-sharded id maps are not built)")


class Arena:
    """Tables + sparse-optimizer state of the fields `rows_per_field` on one rank.

    `shard=(W, rank)` holds that rank's rows of a row-sharded arena; None holds them all.  `adagrad=(initial_g2sum,
    per_element)` keeps AdaGrad state instead of Adam's.  With id_map="hash" a row is initialised by the insert that
    first hands it out (N(0, scale) from `seed`); otherwise the caller initialises w (init_normal, load_global)."""

    def __init__(self, rows_per_field, d: int, device, shard=None, adagrad=None, id_map="mod", seed=0, scale=0.1):
        from .idmap import IdMap, check_id_map          # (idmap builds on this module's layout)
        check_id_map(id_map)
        if shard is not None:
            check_sharded_id_map(id_map)
        self.dev = torch.device(device)
        self.world, self.rank = shard if shard is not None else (1, 0)
        self.d = int(d)
        self.rows = np.asarray(rows_per_field, np.int64)
        _, self.base = shard_layout(self.rows, 1)
        self.local_rows, self.local_base = shard_layout(self.rows, self.world)
        self.total_rows = int(self.rows.sum())
        if self.total_rows >= 2 ** 31 - 1:
            raise ValueError("arena rows must fit int32")
        self.n_local = int(self.local_rows.sum())
        self.row_bits = ops.row_bits(self.n_local)
        self.rows_t = torch.from_numpy(self.rows).to(self.dev)
        self.base_t = torch.from_numpy(self.base).to(self.dev)
        self.lbase_t = self.base_t if self.world == 1 else torch.from_numpy(self.local_base).to(self.dev)
        n = self.n_local
        self.records = self.m = self.v = self.g2sum = None
        if adagrad is None:
            self.records = torch.zeros(n, 3, self.d, device=self.dev)
            self.w, self.m, self.v = self.records[:, 0, :], self.records[:, 1, :], self.records[:, 2, :]
            states = [(self.m, 0.0), (self.v, 0.0)]
        else:
            g2sum0, per_element = float(adagrad[0]), bool(adagrad[1])
            self.w = torch.zeros(n, self.d, device=self.dev)
            self.g2sum = torch.full((n, self.d) if per_element else (n,), g2sum0, device=self.dev)
            states = [(self.g2sum, g2sum0)]
        self.ld = self.w.stride(0)
        self.state = [self.records] if adagrad is None else [self.w, self.g2sum]     # what an update changes per row
        self.idmap = IdMap(self.rows, self.dev, seed, scale, self.w, states) if id_map == "hash" else None
        all_cols = tuple(range(len(self.rows)))
        self._geom = {} if self.idmap is not None else {all_cols: (self.lbase_t, self.rows_t)}

    # ---- initial values
    def init_normal(self, seed: int, scale: float):
        """w = N(0, scale), drawn from ONE generator seeded with `seed` in global arena order, INIT_CHUNK_ROWS rows at
        a time; every rank keeps its own rows, so the shards of a W-way arena reassemble into the W = 1 draw."""
        gen = torch.Generator(device=self.dev).manual_seed(int(seed))
        W, total = self.world, self.total_rows
        for r0 in range(0, total, INIT_CHUNK_ROWS):
            r1 = min(total, r0 + INIT_CHUNK_ROWS)
            vals = torch.empty(r1 - r0, self.d, device=self.dev).normal_(0.0, scale, generator=gen)
            if W == 1:
                self.w[r0:r1] = vals
            else:
                r = torch.arange(r0, r1, device=self.dev)
                f = torch.searchsorted(self.base_t, r, right=True) - 1
                i = r - self.base_t[f]
                mine = torch.remainder(i, W) == self.rank
                self.w[(self.lbase_t[f] + torch.div(i, W, rounding_mode="floor"))[mine]] = vals[mine]
            del vals                # one chunk alive at a time: the next one reuses its memory

    def load_global(self, tables: torch.Tensor):
        """w = this rank's rows of a global table [total rows, d] in arena order (any device)."""
        assert tuple(tables.shape) == (self.total_rows, self.d)
        src = tables.to(torch.float32)
        for g, loc in field_slices(self.rows, self.world, self.rank):
            self.w[loc] = src[g].to(self.dev)

    # ---- lookups
    def geom(self, cols):
        """(row_base, rows) device tensors the lookup kernels read for the fields `cols`, created once (no host ->
        device copy per call: capturable): the local row base and row counts, or (hash mode) the identity geometry."""
        cols = [int(c) for c in cols]
        key = len(cols) if self.idmap is not None else tuple(cols)
        if key not in self._geom:
            g = (np.zeros(len(cols), np.int64), np.full(len(cols), self.total_rows, np.int64)) if self.idmap is not None \
                else (self.local_base[cols], self.rows[cols])
            self._geom[key] = tuple(torch.as_tensor(a, device=self.dev) for a in g)
        return self._geom[key]

    def lookup(self, ids: torch.Tensor, cols, insert: bool, out=None):
        """(ids, row_base, rows) the lookup kernels read for ids int64 [..., len(cols)] of the fields `cols`: the raw
        ids, or (hash mode) the rows they map to (-1 = padding or unseen; insert=True first gives new ids rows; `out`
        receives them)."""
        if self.idmap is not None:
            ids = self.idmap.resolve(ids, self.idmap.fields(cols), insert=insert, out=out)
        return (ids, *self.geom(cols))

    # ---- the rows a step updates, and undo
    def touched_rows(self, groups) -> torch.Tensor:
        """Sorted unique LOCAL rows that a step looking up `groups` = [(ids [..., len(cols)], cols), ...] updates on
        this rank (ids of every rank when sharded; < 0 = padding).  Hash mode: the rows of the ids already mapped and
        every row the step's inserts may hand out."""
        rows = []
        lookups = np.zeros(len(self.rows), np.int64)
        for ids, cols in groups:
            ids = ids.reshape(-1, len(cols))
            if self.idmap is not None:
                r = self.idmap.resolve(ids.contiguous(), self.idmap.fields(cols), insert=False)
                rows.append(r[r >= 0])
                np.add.at(lookups, list(cols), (ids >= 0).sum(0).cpu().numpy())
                continue
            lbase, nrows = self.geom(cols)
            g = torch.remainder(ids, nrows[None, :])
            mine = ids >= 0
            if self.world > 1:                 # owner g mod W, local offset g div W (identities at W = 1)
                mine &= torch.remainder(g, self.world) == self.rank
                g = torch.div(g, self.world, rounding_mode="floor")
            rows.append((lbase[None, :] + g)[mine])
        if self.idmap is not None:
            rows.append(self.idmap.pending_rows(lookups))
        return torch.unique(torch.cat(rows)) if rows else torch.empty(0, dtype=torch.int64, device=self.dev)

    def _undo_state(self):
        """Per-row arrays a train step changes: the optimizer records and (hash mode) the show counts."""
        return self.state if self.idmap is None else self.state + [self.idmap.show]

    def snapshot(self, rows: torch.Tensor):
        """The weights, optimizer state and (hash mode) show counts of `rows`, and the id map's counters."""
        return rows, [t[rows].clone() for t in self._undo_state()], None if self.idmap is None else self.idmap.snapshot()

    def restore(self, snap):
        rows, saved, idmap = snap
        for t, v in zip(self._undo_state(), saved):
            t[rows] = v
        if idmap is not None:
            self.idmap.restore(idmap)
