"""GPU: checkpoints of the composed nets (an object with `emb`, `sub_model` and optionally `opt`).

Resuming is exact: train(2) -> save -> load into a net built from another seed -> train(2) equals train(4) bit for
bit (losses, sub_model parameters, DenseAdam moments and scalars, the arena records, the sparse Adam scalars and the
dropout counters), eagerly and through api.graph.GraphedTrainStep built after / captured before the load.  None of
these nets draws from torch's RNG in a train step; one that did would fail here rather than drift."""
import os
import subprocess
import sys

import numpy as np
import pytest

import util_models as um

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
from torch import nn  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
B = 48


# ------------------------------------------------------------------ a small net over AdaGrad per element
class _Tower(nn.Module):
    def __init__(self, hidden, dropout=False):
        super().__init__()
        from recommendsystem_b200.api import InteractingLayer
        from recommendsystem_b200.api.builders import _KerasDense
        self.hidden = _KerasDense(hidden, "relu")
        self.out = _KerasDense(1, "sigmoid")
        # attention dropout over the columns: a counter every train step advances
        self.interact = InteractingLayer(unit_num=8, head_num=2, use_dropout=True) if dropout else None

    def forward(self, embs):
        x = torch.cat(embs, dim=1)
        if self.interact is not None:
            x = torch.cat([x, self.interact(torch.stack(embs, dim=1)).flatten(1)], dim=1)
        return self.out(self.hidden(x))


class ElementNet:
    """Three single-valued columns and one padded bag column over EmbeddingFeatures(AdaGrad(per_element=True)), a
    two-layer tower (dropout=True: beside an InteractingLayer with attention dropout), dense Adam.  A user's net: no
    subclass of api.net.ComposedNet."""

    def __init__(self, dev, seed, bucket=300, d=8, opt="adagrad_element", id_map="mod", hidden=16, dropout=False):
        from recommendsystem_b200.api.embedding import (Adam, AdaGrad, EmbeddingFeatures, category_column,
                                                        embedding_column)
        self.keys = ["c0", "c1", "c2", "bag"]
        cols = [embedding_column(category_column(k, bucket), d) for k in self.keys]
        sparse = Adam(1e-2) if opt == "adam" else AdaGrad(0.05, 0.1, 0.1, per_element=opt == "adagrad_element")
        self.emb = EmbeddingFeatures(cols, sparse, device=dev, seed=seed, id_map=id_map)
        self.sub_model = _Tower(hidden, dropout).to(dev)
        self.opt = None

    def predict(self, inputs):
        with torch.no_grad():
            e = self.emb(inputs)
            return self.sub_model([e[k] for k in self.keys])

    def dense_optimizer(self):
        from recommendsystem_b200.api.optim import DenseAdam
        if self.opt is None:
            self.opt = DenseAdam(self.sub_model.parameters(), lr=1e-3)
        return self.opt

    def train_step(self, inputs, labels):
        e = self.emb(inputs)
        leaves = {k: e[k].detach().requires_grad_(True) for k in self.keys}
        p = self.sub_model([leaves[k] for k in self.keys])
        opt = self.dense_optimizer()
        y = labels["y"]
        loss = -(y * torch.log(p + 1e-6) + (1 - y) * torch.log(1 - p + 1e-6)).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        self.emb.backward({k: v.grad for k, v in leaves.items()})
        return loss.detach(), {"p": p.detach()}


class OtherElementNet(ElementNet):
    pass


def _element_batch(g, dev):
    inp = {k: torch.randint(0, 10 ** 9, (B,), generator=g) for k in ("c0", "c1", "c2")}
    bag = torch.randint(0, 10 ** 9, (B, 3), generator=g)
    bag[torch.rand(B, 3, generator=g) < 0.3] = -1
    inp["bag"] = bag
    return ({k: v.to(dev) for k, v in inp.items()}, {"y": (torch.rand(B, 1, generator=g) < 0.3).float().to(dev)})


# ------------------------------------------------------------------ the four nets
def _case(kind, dev):
    """(build(seed) -> net with its lazy layers built, four (inputs, labels) batches)."""
    from recommendsystem_b200.api.builders import AUTOINT, AUTOINT_LABELS
    from recommendsystem_b200.api.rank_ctr import TASK_NAMES, Model, parse_feature_slots
    from recommendsystem_b200.api.rough_rank_model import DSSM, config as RC
    from recommendsystem_b200.api.staytime_config import Config as C
    from recommendsystem_b200.api.video_dnn import TASK_KEYS, mtl_net
    g = torch.Generator().manual_seed(7)
    d = str(dev)
    ids = lambda keys: {k: torch.randint(0, 10 ** 9, (B,), generator=g).to(dev) for k in keys}
    flag = lambda: (torch.rand(B, 1, generator=g) < 0.3).float().to(dev)
    if kind == "mtl":
        T = 6
        make = lambda seed: mtl_net(C.SLOTS, C.SEQ_SLOTS, T, dnn_hidden_units=(64, 32), bucket_size=500, device=d,
                                    seed=seed)["net"]

        def batch():
            inp = ids(C.SLOTS)
            for s in C.SEQ_SLOTS:
                x = torch.randint(0, 10 ** 9, (B, T), generator=g)
                lens = torch.randint(0, T + 1, (B,), generator=g)
                x[torch.arange(T)[None, :] >= lens[:, None]] = -1
                inp[s] = x.to(dev)
            y0 = torch.softmax(torch.randn(B, 400, generator=g), -1)
            return inp, {TASK_KEYS[0]: torch.cat([y0, torch.zeros(B, 1)], 1).to(dev), TASK_KEYS[1]: flag(),
                         TASK_KEYS[2]: flag()}
    elif kind == "dssm":
        make = lambda seed: DSSM(bucket_size=500, device=d, seed=seed)["net"]

        def batch():
            inp = ids(RC.USER_FEATURE_IDS + RC.ITEM_FEATURE_IDS)
            inp[RC.DENSE_MASK_ID] = flag()
            return inp, {"student": flag(), "teacher": flag()}
    elif kind == "rank_ctr":
        cfg = um.rank_ctr_config(np.random.default_rng(0))
        make = lambda seed: Model(cfg, bucket_size=500, device=d, seed=seed).run()["net"]
        slots = parse_feature_slots(cfg).sparse_slots

        def batch():
            return ids(slots), {t: flag() for t in TASK_NAMES}
    elif kind == "autoint":
        slots = [str(3000 + i) for i in range(13)]
        make = lambda seed: AUTOINT(slots, [], True, dnn_hidden_units=(32, 16), bucket_size=500, device=d,
                                    seed=seed).model

        def batch():
            return ids(slots), {k: flag() for k in AUTOINT_LABELS}
    else:
        make = lambda seed: ElementNet(dev, seed, dropout=kind == "element_dropout")

        def batch():
            return _element_batch(g, dev)
    batches = [batch() for _ in range(4)]

    def build(seed):
        net = make(seed)
        torch.manual_seed(seed)              # the lazily-built layers draw their weights at the first call
        net.predict(batches[0][0])
        return net
    return build, batches


def _dropout_layers(net):
    return [(p, m) for p, m in net.sub_model.named_modules() if hasattr(m, "_drop_step")]


def _state(net, host_counters=True):
    """Everything a train step changes, on the host."""
    torch.cuda.synchronize()
    st = {"records": net.emb.store.pack(slice(0, net.emb.store.n_local)).cpu()}
    names = {id(p): k for k, p in net.sub_model.named_parameters()}
    for k, p in net.sub_model.named_parameters():
        st["p/" + k] = p.detach().cpu().clone()
    for p, m, v in net.opt.moments():
        st["m/" + names[id(p)]], st["v/" + names[id(p)]] = m.cpu().clone(), v.cpu().clone()
    st["adam_scalars"] = net.opt.scalars.cpu().clone()
    if getattr(net.emb, "scalars", None) is not None:
        st["sparse_scalars"] = net.emb.scalars.cpu().clone()
    for path, layer in _dropout_layers(net):
        st["drop/" + path] = layer._drop_step.cpu().clone()
        if host_counters:
            st["calls/" + path] = torch.tensor(layer._dropout_calls)
    return st


def _assert_same(x, y):
    assert sorted(x) == sorted(y)
    bad = [k for k in x if not torch.equal(x[k], y[k])]
    assert not bad, bad[:10]


CASES = [(k, "eager") for k in ("mtl", "dssm", "rank_ctr", "autoint", "element")] + \
        [(k, m) for k in ("mtl", "dssm", "rank_ctr", "autoint", "element_dropout")
         for m in ("graph_after", "graph_before")]


@pytest.mark.parametrize("kind,mode", CASES)
def test_resume_is_exact(cuda_dev, tmp_path, kind, mode):
    from recommendsystem_b200 import checkpoint as ck
    from recommendsystem_b200.api.graph import GraphedTrainStep
    build, batches = _case(kind, cuda_dev)
    a = build(1)
    la = [float(a.train_step(*bt)[0]) for bt in batches]
    b = build(1)
    lb = [float(b.train_step(*bt)[0]) for bt in batches[:2]]
    assert lb == la[:2]
    ck.save_checkpoint(b, tmp_path / "ck", step=2)
    meta = ck.read_meta(tmp_path / "ck")
    assert meta["model"] == type(b).__name__ and meta["step"] == 2 and meta["world"] == 1
    assert meta["record_floats"] == b.emb.store.record_floats

    c = build(2)                                      # other tables and dense weights: the load overwrites them all
    if mode == "graph_before":
        gs = GraphedTrainStep(c, *batches[2], warmup=3)
    ck.load_checkpoint(c, tmp_path / "ck")
    _assert_same(_state(b), _state(c))
    if mode == "graph_after":
        gs = GraphedTrainStep(c, *batches[2], warmup=3)
    step = c.train_step if mode == "eager" else gs
    lc = [float(step(*bt)[0]) for bt in batches[2:]]
    assert la[2:] == lc, (la, lc)
    # a graph replay does not advance the host mirror of the dropout counter (the device counter is compared)
    _assert_same(_state(a, mode == "eager"), _state(c, mode == "eager"))
    assert any(not torch.equal(x, y) for x, y in zip(_state(b).values(), _state(c).values()))


# ------------------------------------------------------------------ hash mode
def _rows_of(idmap, field, keys, dev):
    t = torch.as_tensor(keys, dtype=torch.int64).reshape(-1, 1).to(dev)
    return idmap.resolve(t, idmap.fields([field]), insert=False).reshape(-1)


def test_hash_mode_resume_per_key(cuda_dev, tmp_path):
    """AUTOINT(id_map="hash"): train, evict, save, load, train against an uninterrupted run, per key (row numbers
    are not reproducible): the record and the show count of every key, the map's counters, the dense state.  The
    resumed net has other dense weights but the same id-map seed: the seed is the init rule of the ids a later step
    inserts, and a net built with another one is refused."""
    from recommendsystem_b200 import checkpoint as ck
    from recommendsystem_b200.api.builders import AUTOINT, AUTOINT_LABELS
    dev = cuda_dev
    slots = [str(3000 + i) for i in range(8)]
    g = torch.Generator().manual_seed(16)
    pools = torch.randint(0, 2 ** 62, (len(slots), 150), generator=g)
    batches = []
    for _ in range(4):
        inp = {s: pools[i][torch.randint(0, 150, (B,), generator=g)].to(dev) for i, s in enumerate(slots)}
        batches.append((inp, {k: (torch.rand(B, 1, generator=g) < 0.3).float().to(dev) for k in AUTOINT_LABELS}))

    def build(seed, id_map="hash", weight_seed=None):
        net = AUTOINT(slots, [], True, dnn_hidden_units=(32, 16), bucket_size=120, device=str(dev), seed=seed,
                      id_map=id_map).model
        torch.manual_seed(seed if weight_seed is None else weight_seed)
        net.predict(batches[0][0])
        return net

    def run(net, part):
        out = []
        for i in part:
            out.append(float(net.train_step(*batches[i])[0]))
            if i == 1:
                net.emb.evict(1.5, 0.75)
        return out

    a, b = build(3), build(3)
    la, lb = run(a, range(4)), run(b, range(2))
    assert sum(b.emb.idmap.stats()["evicted"]) > 0
    ck.save_checkpoint(b, tmp_path / "h", step=2)
    with pytest.raises(ValueError, match="id_map_seed"):
        ck.load_checkpoint(build(4), tmp_path / "h")
    c = build(3, weight_seed=4)
    assert any(not torch.equal(x, y) for x, y in zip(b.sub_model.parameters(), c.sub_model.parameters()))
    ck.load_checkpoint(c, tmp_path / "h")
    assert c.emb.idmap.stats() == b.emb.idmap.stats()
    assert la[2:] == run(c, range(2, 4))
    assert a.emb.idmap.stats() == c.emb.idmap.stats()
    for x, y in zip(a.sub_model.parameters(), c.sub_model.parameters()):
        assert torch.equal(x, y)
    assert torch.equal(a.opt.flat_m, c.opt.flat_m) and torch.equal(a.opt.scalars, c.opt.scalars)
    assert torch.equal(a.emb.scalars, c.emb.scalars)
    for f in range(len(slots)):
        ra, rc = _rows_of(a.emb.idmap, f, pools[f], dev), _rows_of(c.emb.idmap, f, pools[f], dev)
        assert torch.equal(ra >= 0, rc >= 0)
        ok = ra >= 0
        assert torch.equal(a.emb.store.pack(ra[ok]), c.emb.store.pack(rc[ok])), "per-key [w|m|v]"
        assert torch.equal(a.emb.idmap.show[ra[ok]], c.emb.idmap.show[rc[ok]]), "per-key show"
    with pytest.raises(ValueError, match="id_map"):
        ck.load_checkpoint(build(4, "mod"), tmp_path / "h")
    ck.save_checkpoint(build(4, "mod"), tmp_path / "m")
    with pytest.raises(ValueError, match="id_map"):
        ck.load_checkpoint(build(4), tmp_path / "m")


# ------------------------------------------------------------------ refusals
def test_load_and_save_refusals(cuda_dev, tmp_path):
    from recommendsystem_b200 import checkpoint as ck
    dev = cuda_dev
    g = torch.Generator().manual_seed(3)
    inp, lab = _element_batch(g, dev)

    def built(cls=ElementNet, **kw):
        net = cls(dev, 9, **kw)
        net.predict(inp)
        return net

    src = built()
    src.train_step(inp, lab)
    ck.save_checkpoint(src, tmp_path)
    for what, net in (("model", built(OtherElementNet)), ("columns", built(bucket=301)), ("embed_dim", built(d=4)),
                      ("sparse_optimizer", built(opt="adam")), ("per_element", built(opt="adagrad_row")),
                      ("id_map", built(id_map="hash"))):
        with pytest.raises(ValueError, match=what):
            ck.load_checkpoint(net, tmp_path)
    other = built(hidden=12)
    with pytest.raises(ValueError, match="dense"):
        ck.load_checkpoint(other, tmp_path)
    ck.load_checkpoint(other, tmp_path, dense=False)           # the tables alone still load
    assert torch.equal(other.emb.store.pack(slice(0, None)), src.emb.store.pack(slice(0, None)))
    with pytest.raises(ValueError, match="predict"):
        ck.load_checkpoint(ElementNet(dev, 9), tmp_path)         # lazily-built layers not built yet
    src.emb(inp)                                                 # a training forward waiting for its backward
    with pytest.raises(RuntimeError):
        ck.save_checkpoint(src, tmp_path / "x")
    from recommendsystem_b200.autoint import AutoIntConfig, AutoIntTrainer
    tr = AutoIntTrainer(AutoIntConfig(num_fields=3, rows_per_field=[300, 200, 100], batch=64, mlp_hidden=(32, 16)), dev)
    ck.save_checkpoint(tr, tmp_path / "t")
    with pytest.raises(ValueError, match="model"):
        ck.load_checkpoint(built(), tmp_path / "t")               # a trainer's checkpoint is not a net's
    with pytest.raises(ValueError, match="net"):
        ck.load_checkpoint(tr, tmp_path)                         # and the other way round


# ------------------------------------------------------------------ two GPUs
@pytest.mark.parametrize("which", ["autoint", "video_dnn"])
def test_sharded_round_trips(tmp_path, which):
    """W = 2 ShardedEmbeddingFeatures nets: W -> W, W -> 1 and 1 -> W give back every record, the dense state and the
    optimizer state bit for bit (tests/net_checkpoint_worker.py)."""
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29841", os.path.join(HERE, "net_checkpoint_worker.py"), which, str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=400)
    print(r.stdout[-4000:])
    print(r.stderr[-3000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "FAIL" not in r.stdout and "PASS" in r.stdout
