"""The embedding arena's index math (recommendsystem_b200.arena) on CPU tensors, and the initial tables of the GPU
classes built on it against the chunked N(0, scale) draw restated here."""
import numpy as np
import pytest
import torch

from recommendsystem_b200.arena import Arena, field_slices, shard_layout

CHUNK = 1 << 22


def _chunked_draw(total, d, seed, scale, device):
    """The initial table: one generator seeded with `seed`, N(0, scale) over the rows in arena order, 2^22 at a time."""
    gen = torch.Generator(device=device).manual_seed(seed)
    out = torch.empty(total, d, device=device)
    for r0 in range(0, total, CHUNK):
        r1 = min(total, r0 + CHUNK)
        out[r0:r1] = torch.empty(r1 - r0, d, device=device).normal_(0.0, scale, generator=gen)
    return out


def _global_of_local(rows, world, rank):
    """global arena row of every local row of rank `rank`"""
    local_rows, _ = shard_layout(rows, world)
    out = np.full(int(local_rows.sum()), -1, np.int64)
    everything = np.arange(int(np.sum(rows)), dtype=np.int64)
    for g, loc in field_slices(rows, world, rank):
        out[loc] = everything[g]
    return out


def test_shard_layout_at_one_rank_is_the_arena_layout():
    rows = [1000, 7, 33, 1]
    local_rows, local_base = shard_layout(rows, 1)
    assert local_rows.tolist() == rows
    assert local_base.tolist() == [0, 1000, 1007, 1040]


def test_touched_rows_over_ranks_reassemble_the_one_rank_set():
    rows, F = [97, 5, 1, 300, 64], 5
    rng = np.random.default_rng(0)
    ids = rng.integers(0, 10 ** 9, size=(256, F)).astype(np.int64)
    ids[rng.random(ids.shape) < 0.2] = -1                      # padding
    groups = [(torch.from_numpy(ids), range(F)), (torch.from_numpy(ids[:, 3:4].copy()), (3,))]
    one = Arena(rows, 2, "cpu").touched_rows(groups)
    base = np.cumsum([0] + rows[:-1])
    want = np.unique(np.concatenate([base[f] + ids[ids[:, f] >= 0, f] % rows[f] for f in range(F)]))
    assert one.tolist() == want.tolist()
    for W in (1, 2, 3, 8):
        got = []
        for r in range(W):
            loc = Arena(rows, 2, "cpu", shard=(W, r)).touched_rows(groups).numpy()
            assert (np.diff(loc) > 0).all()                       # sorted, unique
            got.append(_global_of_local(rows, W, r)[loc])
        got = np.concatenate(got)
        assert (got >= 0).all() and np.unique(got).size == got.size
        assert np.sort(got).tolist() == one.tolist()


@pytest.mark.parametrize("W", [2, 3])
def test_sharded_draw_reassembles_the_one_rank_draw(W):
    rows, d, seed, scale = [CHUNK - 5, 3, 11], 2, 7, 0.25      # just over 2^22 rows: the draw spans two chunks
    one = Arena(rows, d, "cpu", adagrad=(0.0, False))
    one.init_normal(seed, scale)
    out = torch.full_like(one.w, float("nan"))
    for r in range(W):
        shard = Arena(rows, d, "cpu", shard=(W, r), adagrad=(0.0, False))
        shard.init_normal(seed, scale)
        for g, loc in field_slices(rows, W, r):
            out[g] = shard.w[loc]
    assert torch.equal(out, one.w)


def test_one_rank_draw_is_the_chunked_loop():
    rows, d, seed, scale = [CHUNK, 9], 3, 3, 0.1
    a = Arena(rows, d, "cpu")
    a.init_normal(seed, scale)
    assert torch.equal(a.w, _chunked_draw(sum(rows), d, seed, scale, "cpu"))
    assert not a.m.any() and not a.v.any()


@pytest.mark.gpu
def test_initial_tables_are_the_chunked_draw(cuda_dev):
    from recommendsystem_b200.api.embedding import Adam, AdaGrad, EmbeddingFeatures, category_column, embedding_column
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    rows = [CHUNK - 100, 1000, 357]
    cfg = AutoIntConfig(num_fields=3, rows_per_field=rows, batch=64, mlp_hidden=(32, 16))
    tr = AutoIntTrainer(cfg, cuda_dev)
    assert torch.equal(tr.table, _chunked_draw(sum(rows), 16, cfg.seed, cfg.table_init_scale, cuda_dev))
    del tr
    cols = [embedding_column(category_column(f"c{i}", r), 8) for i, r in enumerate(rows)]
    for opt, scale in ((Adam(), 0.1), (AdaGrad(initial_scale=0.3), 0.3), (AdaGrad(initial_scale=0.3, per_element=True), 0.3)):
        e = EmbeddingFeatures(cols, opt, device=cuda_dev, seed=11)
        assert torch.equal(e.table, _chunked_draw(sum(rows), 8, 11, scale, cuda_dev)), type(opt).__name__
        del e
