"""The fused tower launch (rs_tower_step) against the 4 GEMMs + head pass it replaces: the same bf16 train step from
the same state and batch with AutoIntConfig.fuse_tower on and off."""
import numpy as np
import pytest

from util import REL_BF16, assert_close

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _trainer(B, fuse, hidden=(256, 128)):
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    cfg = AutoIntConfig(num_fields=39, rows_per_field=5000, embed_dim=16, unit_num=16, head_num=2, layer_num=3,
                        mlp_hidden=hidden, batch=B, dtype="bf16", lr_dense=1e-3, lr_sparse=1e-2, fuse_tower=fuse)
    return AutoIntTrainer(cfg, "cuda:0")


@pytest.mark.parametrize("B", [8192, 1000])
def test_fused_tower_matches_separate_kernels(B):
    rng = np.random.default_rng(B)
    ids = torch.from_numpy(rng.integers(0, 2 ** 40, size=(B, 39)).astype(np.int64)).cuda()
    y = torch.from_numpy((rng.random((B, 1)) < 0.25).astype(np.float32)).cuda()
    tf, ts = _trainer(B, True), _trainer(B, False)
    assert tf.fuse_tower and not ts.fuse_tower
    lf, ls = tf.step(ids, y), ts.step(ids, y)
    torch.cuda.synchronize()
    g = lambda t: t.float().cpu().numpy()
    assert_close(g(tf.X), g(ts.X), 0.0, "X")
    assert_close(g(tf.H[0]), g(ts.H[0]), REL_BF16, "H0")
    assert_close(g(tf.Z), g(ts.Z), REL_BF16, "Z")
    assert_close(g(tf.p_raw), g(ts.p_raw), REL_BF16, "p_raw")
    assert abs(float(lf) - float(ls)) <= 1e-3 * abs(float(ls))
    assert_close(g(tf.dZ), g(ts.dZ), REL_BF16, "dZ")
    for i in range(2):
        assert_close(g(tf.dH[i]), g(ts.dH[i]), REL_BF16, f"dH{i}")
    assert_close(g(tf.dX), g(ts.dX), 2 * REL_BF16, "dX")
    for k in tf.G:
        assert_close(g(tf.G[k]), g(ts.G[k]), 2 * REL_BF16, f"grad {k}")
    assert_close(g(tf.flat), g(ts.flat), REL_BF16, "dense parameters after the step")
    # (the tables are not compared: a first Adam step moves a row element by ~lr * sign(g), so gradient elements near
    # zero may differ by 2 lr between the two paths; their input, dX, is compared above)


def test_fused_tower_in_graph_trains_like_separate_kernels():
    B = 2048
    rng = np.random.default_rng(3)
    tf, ts = _trainer(B, True), _trainer(B, False)
    losses = {True: [], False: []}
    for tr in (tf, ts):
        tr.capture()
    for _ in range(20):
        ids = torch.from_numpy(rng.integers(0, 2 ** 40, size=(B, 39)).astype(np.int64)).cuda()
        y = torch.from_numpy((rng.random((B, 1)) < 0.25).astype(np.float32)).cuda()
        for tr in (tf, ts):
            losses[tr.fuse_tower].append(float(tr.step(ids, y)))
    np.testing.assert_allclose(losses[True], losses[False], rtol=1e-2)


def test_unsupported_tower_takes_separate_path():
    tr = _trainer(256, True, hidden=(256, 128, 64))
    assert not tr.fuse_tower
    tr = _trainer(256, True, hidden=(128, 64))
    assert not tr.fuse_tower
    rng = np.random.default_rng(0)
    ids = torch.from_numpy(rng.integers(0, 2 ** 40, size=(256, 39)).astype(np.int64)).cuda()
    y = torch.from_numpy((rng.random((256, 1)) < 0.25).astype(np.float32)).cuda()
    assert np.isfinite(float(tr.step(ids, y)))
