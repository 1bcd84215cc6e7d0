"""Table / optimizer / dense-weight checkpoints and Keras-weight import (SURVEY §8f rank 3).

The reference delegates persistence to TensorNet (`model.save_weights` on every shard; sparse
tables and their optimizer state live on the parameter shards) and exposes the dense part as a
sub-model whose Keras weight names are the serving contract (`rank/multi_head/autoint:53-54`,
`rough_rank/model.py:62-63`, `staytime/VideoDnn.py:193-215`).

Two kinds of object are saved and loaded:
  * an AutoIntTrainer / ShardedAutoIntTrainer (`arena`, `spec`, `flat`, `flat_m`, ...);
  * a composed net: any object with `emb` (api.embedding.EmbeddingFeatures or api.sharded_embedding.
    ShardedEmbeddingFeatures), `sub_model` (an nn.Module) and optionally `opt` (api.optim.DenseAdam, created through
    the net's `dense_optimizer()` when a load finds none) - MtlNet, DssmNet, RankCtrNet, the AUTOINT model, or a
    user's net that follows the same protocol as api.graph.GraphedTrainStep.

A checkpoint is a directory:

    meta.json                      format, world size, rows per field, dense spec, step; trainer: its config; net:
                                   model class, columns (key, bucket_size), embed_dim, sparse optimizer
                                   (adam | adagrad, per_element), record_floats, id_map (hash mode: id_map_seed,
                                   id_map_scale, which a load must match)
    dense.npz                      fp32 master weights by name, `m/<name>`, `v/<name>`, `adam_scalars`; net: the
                                   sub_model.state_dict() entries, the moments of the parameters DenseAdam owns,
                                   `sparse_scalars` (sparse Adam step scalars) and `dropout/<module path>` = [host
                                   call count, device call count] of every layer with a dropout counter
    tables.rank<r>of<W>.bin        that rank's arena as it lies in HBM: fp32 records, field f at rows local_base[f]...
                                   trainer [n_local, 3, d] = [w | m | v] (DESIGN.md §2); net [n_local, record_floats]
                                   from arena.Arena.pack: Adam [w | m | v] (3d), AdaGrad [w | g2sum] (d + 1 per row,
                                   2d per element)
    idmap.npz                      id_map="hash" trainers and nets only (meta.json "id_map": "hash"): the ids
                                   owning the live rows of every field and their show counts (`key_of_row`, `show`,
                                   field after field), `rows_used`, `overflow`, `evicted`, `rows_per_field`; loading copies the
                                   arena and rebuilds the map from it (a file without `show` / `evicted`, written
                                   before eviction existed, loads with zero shows and zero evictions)

Every rank writes its own shard (device -> pinned host -> file in bounded chunks); rank 0 also
writes meta.json and dense.npz (dense state is replicated).  Loading works for ANY world size:
global row g of a field lives in shard g % W at local row g // W (`arena.shard_layout`), so a
rank of a W'-way job collects the rows g = r', r'+W', ... from whichever old shards hold them.
State is copied INTO the model's existing buffers: captured CUDA graphs (AutoIntTrainer.capture, a
GraphedTrainStep captured before the load) and peer (IPC) mappings stay valid.  Resuming is exact: train(2) -> save
-> load -> train(2) equals train(4) bit for bit (tests/test_gpu_checkpoint.py, tests/test_gpu_net_checkpoint.py).
A net is loaded after its lazily-built layers exist (one `predict`); a save between a training forward and its
backward raises RuntimeError.
"""
from __future__ import annotations

import dataclasses
import json
import os
from pathlib import Path
from typing import Dict, Iterator

import numpy as np
import torch

from .api.interacting_layer import dropout_layers
from .arena import shard_layout as shard_rows     # (local_rows[F], local_base[F]) of a W-way job

FORMAT = "rs_b200.checkpoint.v1"
CHUNK_ROWS = 1 << 20                     # rows per host staging chunk (192 MB at d = 16)


# ------------------------------------------------------------------ layout (pure numpy, CPU-testable)
def shard_path(directory, rank: int, world: int) -> Path:
    return Path(directory) / f"tables.rank{rank}of{world}.bin"


def write_shard(path, chunks: Iterator[np.ndarray]) -> int:
    """Append the chunks (fp32 records of any width, [n, 3, d] for the trainer, [n, record_floats] for a net) to
    `path`; returns the rows written."""
    n = 0
    tmp = str(path) + ".tmp"
    with open(tmp, "wb") as f:
        for c in chunks:
            a = np.ascontiguousarray(c, np.float32)
            f.write(a.tobytes() if a.nbytes < (1 << 20) else memoryview(a).cast("B"))
            n += a.shape[0]
    os.replace(tmp, path)
    return n


def reshard_plan(rows_per_field, old_world: int, new_world: int, new_rank: int, chunk_rows: int = CHUNK_ROWS):
    """Yield (old_rank, src_rows, dst_rows): int64 index arrays saying which local rows of old shard
    `old_rank` become which local rows of rank `new_rank` in a `new_world`-way job (whole records: any width)."""
    rows = np.asarray(rows_per_field, np.int64)
    _, old_base = shard_rows(rows, old_world)
    _, new_base = shard_rows(rows, new_world)
    for f, R in enumerate(rows):
        for s in range(old_world):
            n_s = (int(R) - s + old_world - 1) // old_world if R > s else 0      # rows of field f in shard s
            for j0 in range(0, n_s, chunk_rows):
                j = np.arange(j0, min(n_s, j0 + chunk_rows), dtype=np.int64)
                g = j * old_world + s                                            # global row in the field
                keep = (g % new_world) == new_rank
                if not keep.any():
                    continue
                yield s, old_base[f] + j[keep], new_base[f] + g[keep] // new_world


def load_shard_rows(directory, meta: dict, new_world: int, new_rank: int, chunk_rows: int = CHUNK_ROWS):
    """Yield (dst_rows int64[n], records) for rank `new_rank` of a `new_world`-way job: records float32
    [n, record_floats] when meta.json names `record_floats` (a net's checkpoint), else the trainer's [n, 3, d]."""
    d, W = int(meta["embed_dim"]), int(meta["world"])
    rec_shape = (int(meta["record_floats"]),) if "record_floats" in meta else (3, d)
    maps = {}
    for s, src, dst in reshard_plan(meta["rows_per_field"], W, new_world, new_rank, chunk_rows):
        if s not in maps:
            p = shard_path(directory, s, W)
            n = os.path.getsize(p) // (int(np.prod(rec_shape)) * 4)
            maps[s] = np.memmap(p, dtype=np.float32, mode="r", shape=(n,) + rec_shape)
        if src.size and (np.diff(src) == 1).all():
            rec = np.asarray(maps[s][int(src[0]): int(src[-1]) + 1])
        elif src.size > 1 and (np.diff(src) == (src[1] - src[0])).all():
            rec = np.asarray(maps[s][int(src[0]): int(src[-1]) + 1: int(src[1] - src[0])])
        else:
            rec = np.asarray(maps[s][src])
        yield dst, rec


# ------------------------------------------------------------------ trainer save / load
def _cfg_dict(cfg) -> dict:
    out = dataclasses.asdict(cfg)
    for k, v in out.items():
        if isinstance(v, tuple):
            out[k] = list(v)
    return out


def _id_map(trainer) -> str:
    return "hash" if trainer.store.idmap is not None else "mod"


def save_checkpoint(obj, directory, step: int | None = None) -> Path:
    """Write the tables, sparse-optimizer state, dense weights and dense-Adam state of `obj`: an (Sharded)AutoIntTrainer
    or a composed net (an object with `emb` and `sub_model`, see the module docstring).  Collective when the tables
    are row-sharded: every rank calls it; the caller barriers before reading."""
    if _is_net(obj):
        return _save_net(obj, directory, step)
    return _save_trainer(obj, directory, step)


def load_checkpoint(obj, directory, tables: bool = True, dense: bool = True) -> dict:
    """Restore `obj` (a trainer or a composed net) in place from `directory` (any world size); returns meta.json.
    Raises ValueError when the checkpoint was written by another kind of model or its geometry differs."""
    meta = (_load_net if _is_net(obj) else _load_trainer)(obj, directory, tables, dense)
    store = obj.emb.store if _is_net(obj) else obj.store
    torch.cuda.synchronize(store.dev)
    if store.world > 1:
        # the next step's peer gather reads the OTHER ranks' shards at its very start: nobody may run ahead of a
        # rank that is still copying its shard in
        import torch.distributed as dist
        dist.barrier(group=obj.emb.group if _is_net(obj) else obj.ex.group)
    return meta


def _save_trainer(trainer, directory, step: int | None = None) -> Path:
    directory = Path(directory)
    directory.mkdir(parents=True, exist_ok=True)
    store = trainer.store
    _save_tables(store, directory)
    if store.rank == 0:
        dense = {}
        for name, shape, off in trainer.spec:
            k = int(np.prod(shape))
            dense[name] = trainer.flat[off:off + k].view(shape).cpu().numpy()
            dense["m/" + name] = trainer.flat_m[off:off + k].view(shape).cpu().numpy()
            dense["v/" + name] = trainer.flat_v[off:off + k].view(shape).cpu().numpy()
        dense["adam_scalars"] = trainer.adam_scalars.cpu().numpy()
        np.savez(directory / "dense.npz", **dense)
        meta = {
            "format": FORMAT, "world": store.world, "embed_dim": store.d,
            "rows_per_field": [int(x) for x in store.rows],
            "record": "[w|m|v] fp32, row stride 3*embed_dim",
            "dense_spec": [[nm, list(sh)] for nm, sh, _ in trainer.spec],
            "config": _cfg_dict(trainer.cfg), "step": step,
        }
        if _id_map(trainer) == "hash":
            meta["id_map"] = "hash"
        _write_meta(directory, meta)
    return directory


def _save_tables(store, directory: Path):
    """This rank's shard of the arena `store`: its Arena.pack records, device -> pinned host -> file in bounded chunks.
    Rank 0 also writes (hash mode) or removes idmap.npz."""
    torch.cuda.synchronize(store.dev)
    n = store.n_local
    stage = torch.empty(min(n, CHUNK_ROWS), store.record_floats, dtype=torch.float32, pin_memory=True)

    def chunks():
        for r0 in range(0, n, CHUNK_ROWS):
            r1 = min(n, r0 + CHUNK_ROWS)
            stage[: r1 - r0].copy_(store.pack(slice(r0, r1)))
            torch.cuda.synchronize(store.dev)
            yield stage[: r1 - r0].numpy()

    write_shard(shard_path(directory, store.rank, store.world), chunks())
    if store.rank == 0:
        # a reused directory may hold table shards of an earlier save at another world size: remove them so
        # that the directory only ever describes ONE checkpoint (meta.json names the world size that counts)
        for stale in directory.glob("tables.rank*of*.bin"):
            if not stale.name.endswith(f"of{store.world}.bin"):
                stale.unlink()
        if store.idmap is not None:
            np.savez(directory / "idmap.npz", **store.idmap.state())
        elif (directory / "idmap.npz").exists():           # left by an earlier hash-mode save into this directory
            (directory / "idmap.npz").unlink()


def _load_tables(store, directory: Path, meta: dict):
    """This rank's rows of the checkpoint's tables (any world size) and, in hash mode, the id map, into `store` in
    place (Arena.unpack)."""
    for s in range(meta["world"]):
        if not shard_path(directory, s, meta["world"]).exists():
            raise FileNotFoundError(shard_path(directory, s, meta["world"]))
    for dst, rec in load_shard_rows(directory, meta, store.world, store.rank):
        t = torch.from_numpy(np.array(rec, np.float32, copy=True)).reshape(dst.size, -1)     # trainer: [n, 3, d]
        contiguous = dst.size and (np.diff(dst) == 1).all()
        store.unpack(slice(int(dst[0]), int(dst[-1]) + 1) if contiguous else torch.from_numpy(dst).to(store.dev), t)
    if store.idmap is not None:
        with np.load(directory / "idmap.npz") as z:
            store.idmap.load_state({k: z[k] for k in z.files})


def _write_meta(directory: Path, meta: dict):
    tmp = directory / "meta.json.tmp"
    tmp.write_text(json.dumps(meta, indent=1))
    os.replace(tmp, directory / "meta.json")


def read_meta(directory) -> dict:
    meta = json.loads((Path(directory) / "meta.json").read_text())
    if meta.get("format") != FORMAT:
        raise ValueError(f"{directory}: not a {FORMAT} checkpoint (format = {meta.get('format')!r})")
    return meta


def _load_trainer(trainer, directory, tables: bool = True, dense: bool = True) -> dict:
    directory = Path(directory)
    meta = read_meta(directory)
    store = trainer.store
    if "model" in meta:
        raise ValueError(f"{directory}: a checkpoint of a {meta['model']} net, not of an AutoInt trainer")
    if meta.get("id_map", "mod") != _id_map(trainer):
        raise ValueError(f"checkpoint id_map={meta.get('id_map', 'mod')!r} does not match the trainer's "
                         f"id_map={_id_map(trainer)!r}")
    if tables:
        if [int(x) for x in store.rows] != meta["rows_per_field"] or store.d != meta["embed_dim"]:
            raise ValueError("checkpoint tables do not match the trainer's rows_per_field / embed_dim")
        _load_tables(store, directory, meta)
    if dense:
        with np.load(directory / "dense.npz") as z:
            for name, shape, off in trainer.spec:
                if name not in z.files or tuple(z[name].shape) != tuple(shape):
                    raise ValueError(f"checkpoint has no dense parameter {name!r} of shape {tuple(shape)}")
                k = int(np.prod(shape))
                for buf, key in ((trainer.flat, name), (trainer.flat_m, "m/" + name), (trainer.flat_v, "v/" + name)):
                    buf[off:off + k].copy_(torch.from_numpy(np.ascontiguousarray(z[key], np.float32)).reshape(-1))
            trainer.adam_scalars.copy_(torch.from_numpy(z["adam_scalars"]))
        _refresh_dense_shadows(trainer)
    return meta


def _refresh_dense_shadows(trainer):
    if hasattr(trainer, "flat_bf16"):
        trainer.flat_bf16.copy_(trainer.flat)
    if hasattr(trainer, "WT16"):                 # bf16 activations: transposed bf16 weight shadows
        trainer._refresh_wt()


# ------------------------------------------------------------------ composed nets (emb + sub_model [+ opt])
def _is_net(obj) -> bool:
    return hasattr(obj, "emb") and hasattr(obj, "sub_model")


def _net_geometry(net) -> dict:
    """What a net's checkpoint must agree with to load: model class, columns, record layout, id map and, in hash mode,
    the init rule of the rows the map hands out after the load (N(0, scale) from the seed)."""
    emb, store = net.emb, net.emb.store
    geom = {"model": type(net).__name__,
            "columns": [[c.key, int(c.categorical_column.bucket_size)] for c in emb.cols],
            "embed_dim": int(emb.d),
            "sparse_optimizer": "adam" if store.g2sum is None else "adagrad",
            "per_element": store.g2sum is not None and store.g2sum.dim() == 2,
            "record_floats": int(store.record_floats),
            "id_map": "hash" if store.idmap is not None else "mod"}
    if store.idmap is not None:
        # the seed and scale are launch arguments of the insert kernel (frozen into captured graphs): a load cannot
        # change them in place, so a net that would initialise new ids differently is refused
        geom["id_map_seed"], geom["id_map_scale"] = int(store.idmap.seed), float(store.idmap.scale)
    return geom


def _dense_spec(net):
    return [[k, list(v.shape)] for k, v in net.sub_model.state_dict().items()]


def _unbuilt_layers(module):
    """Paths of lazily-built layers (Keras `build` at the first call) that have no parameters yet."""
    return [p for p, m in module.named_modules()
            if getattr(m, "built", True) is False or (hasattr(m, "kernel") and m.kernel is None)]


def _dense_opt(net, create: bool):
    """The net's DenseAdam; `create` builds it through the net's dense_optimizer() when it does not exist yet."""
    opt = net.dense_optimizer() if create and hasattr(net, "dense_optimizer") else getattr(net, "opt", None)
    if opt is not None and not hasattr(opt, "moments"):
        raise TypeError(f"checkpoints hold the dense state of api.optim.DenseAdam, not of {type(opt).__name__}")
    return opt


def _save_net(net, directory, step):
    directory = Path(directory)
    emb, store = net.emb, net.emb.store
    if getattr(emb, "_pending_backward", False):
        raise RuntimeError("save_checkpoint called between a training forward and its backward")
    directory.mkdir(parents=True, exist_ok=True)
    _save_tables(store, directory)
    if store.rank == 0:
        sub = net.sub_model
        dense = {k: v.detach().cpu().numpy() for k, v in sub.state_dict().items()}
        names = {id(p): k for k, p in sub.named_parameters()}
        opt = _dense_opt(net, create=False)
        if opt is None:                                  # not trained yet: the state a new DenseAdam starts from
            for k, p in sub.named_parameters():
                if p.requires_grad:
                    dense["m/" + k] = dense["v/" + k] = np.zeros(tuple(p.shape), np.float32)
            dense["adam_scalars"] = np.zeros(4, np.float32)
        else:
            for p, m, v in opt.moments():
                dense["m/" + names[id(p)]] = m.cpu().numpy()
                dense["v/" + names[id(p)]] = v.cpu().numpy()
            dense["adam_scalars"] = opt.scalars.cpu().numpy()
        for path, layer in dropout_layers(sub):
            dense["dropout/" + path] = np.array(layer.dropout_state(), np.int64)
        if getattr(emb, "scalars", None) is not None:
            dense["sparse_scalars"] = emb.scalars.cpu().numpy()
        np.savez(directory / "dense.npz", **dense)
        meta = {"format": FORMAT, "world": store.world, "rows_per_field": [int(x) for x in store.rows],
                "record": "fp32 [w|m|v] (adam) or [w|g2sum] (adagrad), row stride record_floats",
                **_net_geometry(net), "dense_spec": _dense_spec(net), "step": step}
        _write_meta(directory, meta)
    return directory


def _load_net(net, directory, tables: bool, dense: bool) -> dict:
    directory = Path(directory)
    meta = read_meta(directory)
    emb, store = net.emb, net.emb.store
    for k, want in _net_geometry(net).items():
        got = meta.get(k, "mod" if k == "id_map" else None)
        if got != want:
            raise ValueError(f"checkpoint {k} = {got!r} does not match the net's {want!r}")
    if dense:
        unbuilt = _unbuilt_layers(net.sub_model)
        if unbuilt:
            raise ValueError(f"layers {unbuilt[:4]} of the net have no parameters yet: run one predict first")
        if _dense_spec(net) != meta["dense_spec"]:
            raise ValueError("checkpoint dense parameters (names / shapes) do not match the net's sub_model")
    if tables:
        _load_tables(store, directory, meta)
    with np.load(directory / "dense.npz") as z:
        if tables and "sparse_scalars" in z.files:
            emb.scalars.copy_(torch.from_numpy(z["sparse_scalars"]))
        if dense:
            sub = net.sub_model
            opt = _dense_opt(net, create=True)           # a GraphedTrainStep made after the load keeps its state
            with torch.no_grad():
                for k, v in sub.state_dict().items():    # views of the live tensors: copied in place
                    v.copy_(torch.from_numpy(z[k]))
                if opt is not None:
                    names = {id(p): k for k, p in sub.named_parameters()}
                    for p, m, v in opt.moments():
                        m.copy_(torch.from_numpy(z["m/" + names[id(p)]]))
                        v.copy_(torch.from_numpy(z["v/" + names[id(p)]]))
                    opt.scalars.copy_(torch.from_numpy(z["adam_scalars"]))
            for path, layer in dropout_layers(sub):
                layer.load_dropout_state(z["dropout/" + path])
    return meta


# ------------------------------------------------------------------ Keras weights
# Keras variable names of the reference's AutoInt graph -> trainer parameters.  `Dense.kernel` is
# [in, out] like ours (SURVEY §8b), so no transposes; the four InteractingLayer projections are
# packed side by side as Wqkvr = [Wq | Wk | Wv | Wr] (InteractingLayer.py:24-31).
_INTERACT_ORDER = ("query", "key", "value", "res")


def _strip(name: str) -> str:
    return name[:-2] if name.endswith(":0") else name


def import_keras_autoint(trainer, weights: Dict[str, np.ndarray], prefix: str = "") -> Dict[str, str]:
    """Copy TF/Keras weights of the reference AutoInt graph into `trainer`.

    `weights` maps Keras variable names (`{w.name: w.numpy() for w in model.weights}`, or an .npz of
    the same made on the TF side - h5py is not needed) to arrays.  Accepted names (optionally under
    `prefix`, with or without the ':0' suffix):

        <query|key|value|res>_dense/kernel, .../bias        InteractingLayer.py:24-31
        layer_normalization/gamma, /beta                     InteractingLayer.py:31
        mlp_<i>/kernel, /bias      or dense_<i>/...          MultiLayerDense of the deep tower (autoint:36-41)
        logits/kernel, /bias                                 autoint:47-50
    Returns {trainer parameter: source names}.  Unknown names raise KeyError, shape mismatches ValueError."""
    w = {_strip(k)[len(prefix):] if _strip(k).startswith(prefix) else _strip(k): np.asarray(v) for k, v in weights.items()}
    cfg = trainer.cfg
    used, report = set(), {}

    def take(*names):
        for nme in names:
            if nme in w:
                used.add(nme)
                return nme, w[nme].astype(np.float32)
        raise KeyError(f"none of {names} in the Keras weights ({sorted(w)[:8]} ...)")

    def put(param, value, src):
        dst = trainer.P[param]
        if tuple(value.shape) != tuple(dst.shape):
            raise ValueError(f"{src}: shape {tuple(value.shape)} != {param} {tuple(dst.shape)}")
        dst.copy_(torch.from_numpy(np.ascontiguousarray(value)))
        report[param] = src

    ks, bs, src = [], [], []
    for nm in _INTERACT_ORDER:
        if nm == "res" and not cfg.use_res:
            U = cfg.unit_num
            ks.append(np.zeros((cfg.embed_dim, U), np.float32)); bs.append(np.zeros(U, np.float32))
            continue
        a, k = take(f"{nm}_dense/kernel", f"{nm}_dense_kernel")
        b, bv = take(f"{nm}_dense/bias", f"{nm}_dense_bias")
        ks.append(k); bs.append(bv); src += [a, b]
    put("Wqkvr", np.concatenate(ks, axis=1), "|".join(src[0::2]))
    put("bqkvr", np.concatenate(bs, axis=0), "|".join(src[1::2]))
    a, g = take("layer_normalization/gamma", "ln/gamma"); put("gamma", g, a)
    a, bt = take("layer_normalization/beta", "ln/beta"); put("beta", bt, a)
    for i in range(len(cfg.mlp_hidden)):
        a, k = take(f"mlp_{i}/kernel", f"dense_{i}/kernel"); put(f"mlp_W{i}", k, a)
        a, bv = take(f"mlp_{i}/bias", f"dense_{i}/bias"); put(f"mlp_b{i}", bv, a)
    a, k = take("logits/kernel"); put("out_W", k, a)
    a, bv = take("logits/bias"); put("out_b", bv, a)
    extra = set(w) - used
    if extra:
        raise KeyError(f"Keras weights not consumed: {sorted(extra)}")
    _refresh_dense_shadows(trainer)
    return report


def export_keras_autoint(trainer) -> Dict[str, np.ndarray]:
    """Inverse of import_keras_autoint: the dense sub-model under the Keras variable names."""
    cfg, U = trainer.cfg, trainer.cfg.unit_num
    P = {k: v.detach().cpu().numpy() for k, v in trainer.P.items()}
    out = {}
    for i, nm in enumerate(_INTERACT_ORDER):
        if nm == "res" and not cfg.use_res:
            continue
        out[f"{nm}_dense/kernel:0"] = P["Wqkvr"][:, i * U:(i + 1) * U].copy()
        out[f"{nm}_dense/bias:0"] = P["bqkvr"][i * U:(i + 1) * U].copy()
    out["layer_normalization/gamma:0"] = P["gamma"].copy()
    out["layer_normalization/beta:0"] = P["beta"].copy()
    for i in range(len(cfg.mlp_hidden)):
        out[f"mlp_{i}/kernel:0"] = P[f"mlp_W{i}"].copy()
        out[f"mlp_{i}/bias:0"] = P[f"mlp_b{i}"].copy()
    out["logits/kernel:0"] = P["out_W"].copy()
    out["logits/bias:0"] = P["out_b"].copy()
    return out


def load_keras_state(module: torch.nn.Module, weights: Dict[str, np.ndarray], strict: bool = True) -> list:
    """Keras-named weights -> a drop-in layer / model of `recommendsystem_b200.api` (whose parameter
    names already mirror the reference's `add_weight(name=...)` / Dense names with '/' -> '_').
    `a/b/kernel:0` matches the parameter whose dotted name, with '.' and '/' folded to '_', is
    `a_b_kernel`.  Returns the list of parameters set."""
    def fold(s):
        return _strip(s).replace("/", "_").replace(".", "_")

    params = {fold(k): p for k, p in module.named_parameters()}
    done = []
    with torch.no_grad():
        for k, v in weights.items():
            key = fold(k)
            if key not in params:
                if strict:
                    raise KeyError(f"{k}: no parameter named {key} in {type(module).__name__}")
                continue
            p = params[key]
            a = np.asarray(v, np.float32)
            if tuple(a.shape) != tuple(p.shape):
                raise ValueError(f"{k}: shape {tuple(a.shape)} != parameter {tuple(p.shape)}")
            p.copy_(torch.from_numpy(a).to(p.device))
            done.append(key)
    return done
