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
    counters     int64 [2, n_fields]  rows used, overflowed lookups (ids that found their field full)
A new row's record is written by the insert kernel itself: w = scale * N(0,1) as a pure function of
(seed, field, id, k), optimizer state at its initial values.  Row numbers depend on the order in which the insert
threads win their atomics, but nothing computed depends on them, so hash mode is bit-reproducible per key.
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

    def stats(self) -> dict:
        """Rows used and overflowed lookups per field (one device -> host copy)."""
        c = self.counters.cpu().numpy()
        return {"rows_used": c[0].tolist(), "overflow": c[1].tolist(), "capacity": self.rows.tolist()}

    # ---- checkpoints
    def state(self) -> dict:
        """Host arrays: the owners of the used rows of every field (field after field), counters, capacities."""
        c = self.counters.cpu().numpy()
        kor = [self.key_of_row[int(b): int(b) + int(n)].cpu().numpy() for b, n in zip(self.base, c[0])]
        return {"key_of_row": np.concatenate(kor) if kor else np.zeros(0, np.int64), "rows_used": c[0].copy(),
                "overflow": c[1].copy(), "rows_per_field": self.rows.copy()}

    def load_state(self, st) -> None:
        if [int(x) for x in st["rows_per_field"]] != [int(x) for x in self.rows]:
            raise ValueError("id map: the checkpoint's rows per field differ from this map's")
        used = np.asarray(st["rows_used"], np.int64)
        keys = np.asarray(st["key_of_row"], np.int64)
        if (used > self.rows).any() or keys.size != int(used.sum()):
            raise ValueError("id map: inconsistent checkpoint (rows used vs key_of_row)")
        o = 0
        for b, n in zip(self.base, used):
            if n:
                self.key_of_row[int(b): int(b) + int(n)].copy_(torch.from_numpy(keys[o:o + int(n)].copy()))
            o += int(n)
        self.counters.copy_(torch.from_numpy(np.stack([used, np.asarray(st["overflow"], np.int64)])))
        self._rebuild()

    # ---- undo (GraphedTrainStep / AutoIntTrainer.capture warm-up steps)
    def snapshot(self) -> torch.Tensor:
        return self.counters.clone()

    def restore(self, snap: torch.Tensor) -> None:
        """Back to the counters of `snap`: rows handed out since are forgotten and the slots rebuilt."""
        self.counters.copy_(snap)
        self._rebuild()

    def pending_rows(self, lookups_per_field) -> torch.Tensor:
        """Rows the next insert of at most lookups_per_field[f] keys per field can hand out (sorted int64)."""
        used = self.counters[0].cpu().numpy()
        out = [np.arange(b + u, b + min(u + int(n), r), dtype=np.int64)
               for b, u, r, n in zip(self.base, used, self.rows, lookups_per_field)]
        return torch.from_numpy(np.concatenate(out) if out else np.zeros(0, np.int64)).to(self.dev)
