"""Checkpoint records of the composed nets on CPU: arena.Arena pack / unpack for the three sparse-optimizer layouts, and
resharding of [n, record_floats] shards between world sizes."""
import itertools
import json

import numpy as np
import pytest
import torch

from recommendsystem_b200 import checkpoint as ck
from recommendsystem_b200.arena import Arena

KINDS = {"adam": None, "adagrad_row": (0.1, False), "adagrad_element": (0.1, True)}


def _fill(arena, seed):
    g = torch.Generator().manual_seed(seed)
    for t in arena.state:
        t.copy_(torch.randn(t.shape, generator=g))


@pytest.mark.parametrize("kind", list(KINDS))
def test_pack_unpack_round_trip(kind):
    rows, d = [13, 1, 40], 4
    a = Arena(rows, d, "cpu", adagrad=KINDS[kind])
    _fill(a, 1)
    rf = {"adam": 3 * d, "adagrad_row": d + 1, "adagrad_element": 2 * d}[kind]
    assert a.record_floats == rf
    rec = a.pack(slice(0, a.n_local))
    assert rec.shape == (a.n_local, rf) and rec.dtype == torch.float32
    assert torch.equal(rec[:, :d], a.w)                               # w leads every record
    if kind == "adam":
        assert torch.equal(rec, a.records.reshape(a.n_local, 3 * d))  # the Adam record is the arena itself
    else:
        assert torch.equal(rec[:, d:], a.g2sum.reshape(a.n_local, -1))
    b = Arena(rows, d, "cpu", adagrad=KINDS[kind])
    w_id = b.w.data_ptr()
    b.unpack(slice(0, 20), rec[:20])                                  # a slice ...
    idx = torch.arange(20, a.n_local)[torch.randperm(a.n_local - 20, generator=torch.Generator().manual_seed(2))]
    b.unpack(idx, rec[idx])                                           # ... and scattered rows
    assert b.w.data_ptr() == w_id                                     # in place
    for x, y in zip(a.state, b.state):
        assert torch.equal(x, y)
    assert torch.equal(b.pack(idx), rec[idx])


def _write_world(path, glob, rows, W):
    """The shards a W-way job writes: shard s holds global rows s, s+W, ... of every field (records of any width)."""
    local_rows, local_base = ck.shard_rows(rows, W)
    _, base = ck.shard_rows(rows, 1)
    for s in range(W):
        shard = np.zeros((int(local_rows.sum()), glob.shape[1]), np.float32)
        for f, R in enumerate(rows):
            part = glob[base[f]: base[f] + R][s::W]
            shard[local_base[f]: local_base[f] + part.shape[0]] = part
        assert ck.write_shard(ck.shard_path(path, s, W), iter([shard[:3], shard[3:]])) == shard.shape[0]
    meta = {"format": ck.FORMAT, "world": W, "embed_dim": 4, "record_floats": int(glob.shape[1]),
            "rows_per_field": [int(r) for r in rows]}
    (path / "meta.json").write_text(json.dumps(meta))
    return meta


@pytest.mark.parametrize("width", ["d+1", "2d"])
@pytest.mark.parametrize("old_w,new_w", list(itertools.product([1, 2, 3, 8], repeat=2)))
def test_reshard_records_of_any_width(tmp_path, width, old_w, new_w):
    rows, d = [17, 1, 64, 9, 2], 4           # ragged, with fields of fewer rows than ranks
    rf = d + 1 if width == "d+1" else 2 * d
    glob = np.random.default_rng(old_w * 10 + new_w).standard_normal((sum(rows), rf)).astype(np.float32)
    meta = _write_world(tmp_path, glob, rows, old_w)
    new_rows, new_base = ck.shard_rows(rows, new_w)
    _, base = ck.shard_rows(rows, 1)
    seen = np.zeros(sum(rows), np.int64)
    for r in range(new_w):
        shard = np.full((int(new_rows.sum()), rf), np.nan, np.float32)
        for dst, rec in ck.load_shard_rows(tmp_path, meta, new_w, r, chunk_rows=5):
            assert rec.shape == (dst.size, rf)
            assert np.isnan(shard[dst]).all()                 # every destination row written once
            shard[dst] = rec
        for f, R in enumerate(rows):
            g = np.arange(r, R, new_w)
            np.testing.assert_array_equal(shard[new_base[f]: new_base[f] + g.size], glob[base[f] + g])
            seen[base[f] + g] += 1
    assert (seen == 1).all()                                  # every global row reassembled exactly once
