"""Checkpoint layout / resharding logic on CPU (no GPU, no CUDA library calls)."""
import json

import numpy as np
import pytest

from recommendsystem_b200 import checkpoint as ck


def _global_tables(rows, d, seed=3):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal((int(r), 3, d)).astype(np.float32) for r in rows]


def _write_world(tmp_path, tabs, rows, d, W):
    """Write the shards a W-way job would: shard s holds global rows s, s+W, ... of every field."""
    local_rows, local_base = ck.shard_rows(rows, W)
    for s in range(W):
        arena = np.zeros((int(local_rows.sum()), 3, d), np.float32)
        for f, t in enumerate(tabs):
            part = t[s::W]
            arena[local_base[f]: local_base[f] + part.shape[0]] = part
        n = ck.write_shard(ck.shard_path(tmp_path, s, W), iter([arena[:5], arena[5:]]))
        assert n == arena.shape[0]
    meta = {"format": ck.FORMAT, "world": W, "embed_dim": d, "rows_per_field": [int(r) for r in rows]}
    (tmp_path / "meta.json").write_text(json.dumps(meta))
    return meta


@pytest.mark.parametrize("old_w,new_w", [(1, 1), (1, 2), (2, 1), (2, 3), (3, 2), (4, 8), (8, 2)])
def test_reshard_any_world(tmp_path, old_w, new_w):
    rows, d = [17, 1, 64, 9, 2], 4          # ragged, includes fields with fewer rows than ranks
    tabs = _global_tables(rows, d)
    meta = _write_world(tmp_path, tabs, rows, d, old_w)
    assert ck.read_meta(tmp_path)["world"] == old_w
    new_rows, new_base = ck.shard_rows(rows, new_w)
    for r in range(new_w):
        arena = np.full((int(new_rows.sum()), 3, d), np.nan, np.float32)
        for dst, rec in ck.load_shard_rows(tmp_path, meta, new_w, r, chunk_rows=7):
            assert np.isnan(arena[dst]).all()             # every destination row written once
            arena[dst] = rec
        for f, t in enumerate(tabs):
            want = t[r::new_w]
            got = arena[new_base[f]: new_base[f] + want.shape[0]]
            np.testing.assert_array_equal(got, want)      # bit-exact


def test_bad_format_raises(tmp_path):
    (tmp_path / "meta.json").write_text(json.dumps({"format": "something else"}))
    with pytest.raises(ValueError):
        ck.read_meta(tmp_path)


def test_load_keras_state_names():
    import torch

    class M(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.din_nn_0 = torch.nn.ParameterDict({"kernel": torch.nn.Parameter(torch.zeros(3, 2))})
            self.kernel0 = torch.nn.Parameter(torch.zeros(2, 2))

    m = M()
    w = {"din_nn_0/kernel:0": np.arange(6, dtype=np.float32).reshape(3, 2), "kernel0:0": np.eye(2, dtype=np.float32)}
    assert sorted(ck.load_keras_state(m, w)) == ["din_nn_0_kernel", "kernel0"]
    assert m.din_nn_0["kernel"][2, 1].item() == 5.0
    with pytest.raises(KeyError):
        ck.load_keras_state(m, {"nope/kernel:0": np.zeros((1,))})
    with pytest.raises(ValueError):
        ck.load_keras_state(m, {"kernel0:0": np.zeros((3, 3), np.float32)})


def test_reshard_plan_partitions_every_row_exactly_once():
    """Property (hypothesis): for any ragged table set and any W -> W', the plans of the W' new ranks together
    read every saved row exactly once and write every destination row exactly once."""
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=60, deadline=None)
    @given(rows=st.lists(st.integers(1, 200), min_size=1, max_size=6), old_w=st.integers(1, 9), new_w=st.integers(1, 9),
           chunk=st.integers(1, 64))
    def prop(rows, old_w, new_w, chunk):
        _, old_base = ck.shard_rows(rows, old_w)
        new_rows, new_base = ck.shard_rows(rows, new_w)
        seen_src = set()
        for r in range(new_w):
            seen_dst = set()
            for s, src, dst in ck.reshard_plan(rows, old_w, new_w, r, chunk_rows=chunk):
                assert len(src) == len(dst) > 0
                for a, b in zip(src.tolist(), dst.tolist()):
                    assert (s, a) not in seen_src and b not in seen_dst
                    seen_src.add((s, a)); seen_dst.add(b)
                    # the pair addresses the same global row of the same field
                    f = int(np.searchsorted(old_base, a, side="right") - 1)
                    g_old = (a - old_base[f]) * old_w + s
                    f2 = int(np.searchsorted(new_base, b, side="right") - 1)
                    g_new = (b - new_base[f2]) * new_w + r
                    assert f == f2 and g_old == g_new < rows[f]
            assert len(seen_dst) == sum(len(range(r, R, new_w)) for R in rows)
        assert len(seen_src) == sum(rows)

    prop()


def test_keras_import_export_host_logic():
    """Name mapping of import_keras_autoint / export_keras_autoint on a stub trainer (CPU tensors): packing of the four
    projections into Wqkvr, `use_res=False`, the ':0' suffix and prefix handling, error cases."""
    import types

    import torch
    d = U = 4
    spec = {"Wqkvr": (d, 4 * U), "bqkvr": (4 * U,), "gamma": (U,), "beta": (U,), "mlp_W0": (3 * d, 8), "mlp_b0": (8,),
            "out_W": (8 + 3 * U, 1), "out_b": (1,)}

    def stub(use_res=True):
        cfg = types.SimpleNamespace(use_res=use_res, unit_num=U, embed_dim=d, mlp_hidden=(8,))
        return types.SimpleNamespace(cfg=cfg, P={k: torch.zeros(s) for k, s in spec.items()})

    rng = np.random.default_rng(0)
    w = {}
    for nm in ("query", "key", "value", "res"):
        w[f"model/{nm}_dense/kernel:0"] = rng.standard_normal((d, U)).astype(np.float32)
        w[f"model/{nm}_dense/bias:0"] = rng.standard_normal(U).astype(np.float32)
    w["model/layer_normalization/gamma:0"] = rng.standard_normal(U).astype(np.float32)
    w["model/layer_normalization/beta:0"] = rng.standard_normal(U).astype(np.float32)
    w["model/dense_0/kernel"] = rng.standard_normal((3 * d, 8)).astype(np.float32)       # MultiLayerDense default names, no ':0'
    w["model/dense_0/bias"] = rng.standard_normal(8).astype(np.float32)
    w["model/logits/kernel:0"] = rng.standard_normal((8 + 3 * U, 1)).astype(np.float32)
    w["model/logits/bias:0"] = rng.standard_normal(1).astype(np.float32)
    tr = stub()
    rep = ck.import_keras_autoint(tr, w, prefix="model/")
    assert rep["mlp_W0"] == "dense_0/kernel" and rep["gamma"] == "layer_normalization/gamma"
    for i, nm in enumerate(("query", "key", "value", "res")):
        np.testing.assert_array_equal(tr.P["Wqkvr"][:, i * U:(i + 1) * U].numpy(), w[f"model/{nm}_dense/kernel:0"])
        np.testing.assert_array_equal(tr.P["bqkvr"][i * U:(i + 1) * U].numpy(), w[f"model/{nm}_dense/bias:0"])
    back = ck.export_keras_autoint(tr)
    np.testing.assert_array_equal(back["res_dense/kernel:0"], w["model/res_dense/kernel:0"])
    np.testing.assert_array_equal(back["mlp_0/kernel:0"], w["model/dense_0/kernel"])

    # use_res=False: no res_dense weights expected, the packed block stays zero and is not exported
    w2 = {k: v for k, v in w.items() if "res_dense" not in k}
    tr2 = stub(use_res=False)
    ck.import_keras_autoint(tr2, w2, prefix="model/")
    assert float(tr2.P["Wqkvr"][:, 3 * U:].abs().sum()) == 0.0
    assert "res_dense/kernel:0" not in ck.export_keras_autoint(tr2)
    with pytest.raises(KeyError):
        ck.import_keras_autoint(stub(use_res=False), w, prefix="model/")        # stray res_dense weights
    with pytest.raises(KeyError):
        ck.import_keras_autoint(stub(), w2, prefix="model/")                     # res_dense missing
