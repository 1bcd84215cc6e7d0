"""Collision-free id -> arena-row map: the `id_map="hash"` mode of api.embedding.EmbeddingFeatures and
autoint.AutoIntTrainer.

The reference's sparse inputs are feature signs (64-bit hashes) that TensorNet keeps in sharded hash tables, one row
per distinct sign.  The default `"mod"` mode reads row `row_base[f] + id mod rows[f]`, so ids congruent modulo the
table size share a row and its optimizer state.  An IdMap gives every distinct (field, id) its own row of the field's
range [row_base[f], row_base[f] + R_f) the first time a training step sees it (R_f = the field's `bucket_size` /
`rows_per_field`, a fixed capacity).  After `resolve` the existing gather / fused-lookup / sorted-segment kernels run
unchanged on the resolved rows with an identity geometry (row_base = 0, rows = total rows).

This module is the only code that knows the map's format (include/rs_b200.h, K9):
    slots        int64 [n_slots, 2]   {key, row | pad << 32}, field f owns next_pow2(2 R_f) of them
    key_of_row   int64 [total rows]   the id that owns each arena row, -1 = unused
    counters     int64 [2, n_fields]  live rows, overflowed lookups (ids that found their field full)
    show         fp32  [total rows]   show count of each row (training lookups; 0 for a row no key owns)
    evicted      int64 [n_fields]     keys dropped by `evict` so far
A new row's record is written by the insert kernel itself: w = scale * N(0,1) as a pure function of
(seed, field, id, k), optimizer state at its initial values.  Row numbers depend on the order in which the insert
threads win their atomics, but nothing computed depends on them, so hash mode is bit-reproducible per key.

Eviction (TensorNet's show decay and `feature_drop_show`) keeps long runs on new ids: every training lookup adds 1 to
its row's show count (`count`), and `evict(threshold, decay)` multiplies every live row's show by `decay` and drops the
keys whose show is then below `threshold`.  Each field's live rows are compacted back to the front of its range, so
the insert kernel keeps handing out rows from one counter.  An evicted id is like one never seen: it reads zeros in
inference and, trained again, gets a fresh record from the init rule with show 0.  Show increments all add 1.0f and
decay is per-row fp32, so the set of evicted keys is a pure function of the key history (DESIGN.md §5).
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops
from .arena import shard_layout

ID_MAPS = ("mod", "hash")


def check_id_map(id_map: str) -> str:
    if id_map not in ID_MAPS:
        raise ValueError(f"id_map must be one of {ID_MAPS}, not {id_map!r}")
    return id_map


def check_evict_args(threshold, decay):
    """(threshold, decay) as the fp32 values the eviction uses; ValueError unless 0 < decay <= 1 and the threshold is
    finite."""
    with np.errstate(over="ignore", invalid="ignore"):
        t, dc = np.float32(threshold), np.float32(decay)
    if not np.isfinite(t):
        raise ValueError(f"evict: threshold must be finite, not {threshold!r}")
    if not (0.0 < dc <= 1.0):
        raise ValueError(f"evict: decay must be in (0, 1], not {decay!r}")
    return float(t), float(dc)


def slots_per_field(rows_per_field) -> np.ndarray:
    """next power of two >= 2 R_f (load factor <= 1/2)."""
    rows = np.asarray(rows_per_field, np.int64)
    return np.asarray([1 << int(max(2 * int(r), 2) - 1).bit_length() for r in rows], np.int64)


class IdMap:
    """Map of the fields of one arena.  `w` is the arena's [total_rows, d] weight view (row stride allowed);
    `states` are up to two (view, initial value) pairs of per-row optimizer state ([R] or [R, k] fp32) that a new
    row gets."""

    def __init__(self, rows_per_field, device, seed: int, scale: float, w: torch.Tensor, states=()):
        self.dev = torch.device(device)
        self.rows = np.asarray(rows_per_field, np.int64)
        _, self.base = shard_layout(self.rows, 1)
        self.total_rows = int(self.rows.sum())
        if w.shape[0] != self.total_rows:
            raise ValueError(f"IdMap: weight view has {w.shape[0]} rows, the fields {self.total_rows}")
        slots = slots_per_field(self.rows)
        slot_base = np.concatenate([[0], np.cumsum(slots)[:-1]]).astype(np.int64)
        self.n_fields = len(self.rows)
        self.geom = torch.from_numpy(np.stack([self.base, self.rows, slot_base, slots - 1], 1).copy()).to(self.dev)
        self.slots = torch.empty(int(slots.sum()), 2, dtype=torch.int64, device=self.dev)
        self.key_of_row = torch.empty(self.total_rows, dtype=torch.int64, device=self.dev)
        self.counters = torch.zeros(2, self.n_fields, dtype=torch.int64, device=self.dev)
        self.show = torch.zeros(self.total_rows, dtype=torch.float32, device=self.dev)
        self.evicted = torch.zeros(self.n_fields, dtype=torch.int64, device=self.dev)
        self.seed, self.scale, self.w, self.states = int(seed), float(scale), w, list(states)
        self._fields = {}
        self._rebuild()                                  # empty slots, key_of_row = -1

    def _rebuild(self):
        ops.idmap_rebuild(self.slots, self.key_of_row, self.counters, self.geom, int(self.rows.max()))

    def fields(self, fields) -> torch.Tensor:
        """int32 device tensor of a column -> field list, created once (graph-capturable callers)."""
        key = tuple(int(f) for f in fields)
        t = self._fields.get(key)
        if t is None:
            t = torch.tensor(key, dtype=torch.int32, device=self.dev)
            self._fields[key] = t
        return t

    def resolve(self, ids: torch.Tensor, field_of_col: torch.Tensor, insert: bool, out=None) -> torch.Tensor:
        """ids int64 [..., F] (column j of field field_of_col[j]; < 0 = padding) -> int64 arena rows of the same shape,
        -1 for padding, unseen (insert=False) and overflowed keys.  insert=True first gives new keys rows."""
        if insert:
            ops.idmap_insert(self.slots, self.key_of_row, self.counters, self.geom, ids, field_of_col, self.seed,
                             self.scale, self.w, self.states)
        return ops.idmap_lookup(self.slots, self.counters, self.geom, ids, field_of_col, out=out, after_insert=insert)

    def count(self, rows: torch.Tensor) -> None:
        """show[r] += 1 for every row r >= 0 of `rows` (the output of a training `resolve`)."""
        ops.idmap_count(self.show, rows)

    def evict(self, threshold: float, decay: float = 1.0) -> None:
        """show = fp32(show * decay) on every live row, then drop the keys whose show is < threshold, compact every
        field's live rows and rebuild the slots.  Asynchronous on the current stream; no buffer moves, so captured
        graphs stay valid."""
        threshold, decay = check_evict_args(threshold, decay)
        ops.idmap_evict(self.slots, self.key_of_row, self.counters, self.geom, self.show, self.evicted, threshold,
                        decay, self.w, [t for t, _ in self.states])

    def stats(self) -> dict:
        """Live rows, overflowed lookups and evicted keys per field (device -> host copies)."""
        c = self.counters.cpu().numpy()
        return {"rows_used": c[0].tolist(), "overflow": c[1].tolist(), "evicted": self.evicted.cpu().tolist(),
                "capacity": self.rows.tolist()}

    # ---- checkpoints
    def state(self) -> dict:
        """Host arrays: the owners of the live rows of every field and their show counts (field after field),
        counters, evicted keys, capacities."""
        c = self.counters.cpu().numpy()
        live = lambda t: np.concatenate([t[int(b): int(b) + int(n)].cpu().numpy() for b, n in zip(self.base, c[0])])
        return {"key_of_row": live(self.key_of_row), "show": live(self.show), "rows_used": c[0].copy(),
                "overflow": c[1].copy(), "evicted": self.evicted.cpu().numpy(), "rows_per_field": self.rows.copy()}

    def load_state(self, st) -> None:
        if [int(x) for x in st["rows_per_field"]] != [int(x) for x in self.rows]:
            raise ValueError("id map: the checkpoint's rows per field differ from this map's")
        used = np.asarray(st["rows_used"], np.int64)
        keys = np.asarray(st["key_of_row"], np.int64)
        if (used > self.rows).any() or keys.size != int(used.sum()):
            raise ValueError("id map: inconsistent checkpoint (rows used vs key_of_row)")
        # show / evicted: absent from maps saved before eviction existed (zero shows, nothing evicted)
        show = np.asarray(st["show"], np.float32) if "show" in st else np.zeros(keys.size, np.float32)
        if show.size != keys.size:
            raise ValueError("id map: inconsistent checkpoint (show vs key_of_row)")
        self.show.zero_()
        o = 0
        for b, n in zip(self.base, used):
            if n:
                self.key_of_row[int(b): int(b) + int(n)].copy_(torch.from_numpy(keys[o:o + int(n)].copy()))
                self.show[int(b): int(b) + int(n)].copy_(torch.from_numpy(show[o:o + int(n)].copy()))
            o += int(n)
        self.counters.copy_(torch.from_numpy(np.stack([used, np.asarray(st["overflow"], np.int64)])))
        ev = np.asarray(st["evicted"], np.int64) if "evicted" in st else np.zeros(self.n_fields, np.int64)
        self.evicted.copy_(torch.from_numpy(ev.copy()))
        self._rebuild()

    # ---- undo (GraphedTrainStep / AutoIntTrainer.capture warm-up steps)
    def snapshot(self) -> torch.Tensor:
        return self.counters.clone()

    def restore(self, snap: torch.Tensor) -> None:
        """Back to the counters of `snap`: rows handed out since are forgotten (show 0, as rows no key owns) and the
        slots rebuilt.  The show counts of the rows kept are the caller's (Arena.snapshot / restore)."""
        self.counters.copy_(snap)
        for b, u, r in zip(self.base, snap[0].cpu().numpy(), self.rows):
            self.show[int(b) + int(u): int(b) + int(r)].zero_()
        self._rebuild()

    def pending_rows(self, lookups_per_field) -> torch.Tensor:
        """Rows the next insert of at most lookups_per_field[f] keys per field can hand out (sorted int64)."""
        used = self.counters[0].cpu().numpy()
        out = [np.arange(b + u, b + min(u + int(n), r), dtype=np.int64)
               for b, u, r, n in zip(self.base, used, self.rows, lookups_per_field)]
        return torch.from_numpy(np.concatenate(out) if out else np.zeros(0, np.int64)).to(self.dev)
