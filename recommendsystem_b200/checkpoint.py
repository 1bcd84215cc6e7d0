"""Table / optimizer / dense-weight checkpoints and Keras-weight import (SURVEY §8f rank 3).

The reference delegates persistence to TensorNet (`model.save_weights` on every shard; sparse
tables and their optimizer state live on the parameter shards) and exposes the dense part as a
sub-model whose Keras weight names are the serving contract (`rank/multi_head/autoint:53-54`,
`rough_rank/model.py:62-63`, `staytime/VideoDnn.py:193-215`).  Here a checkpoint is a directory:

    meta.json                      format, config, world size, rows per field, dense spec, step
    dense.npz                      fp32 master weights by name, `m/<name>`, `v/<name>`, `adam_scalars`
    tables.rank<r>of<W>.bin        that rank's arena as it lies in HBM: [n_local, 3, d] fp32 records
                                   [w | m | v] (DESIGN.md §2), field f at rows local_base[f]...
    idmap.npz                      id_map="hash" trainers only (meta.json "id_map": "hash"): the ids owning the live
                                   rows of every field and their show counts (`key_of_row`, `show`, field after
                                   field), `rows_used`, `overflow`, `evicted`, `rows_per_field`; loading copies the
                                   arena and rebuilds the map from it (a file without `show` / `evicted`, written
                                   before eviction existed, loads with zero shows and zero evictions)

Every rank writes its own shard (device -> pinned host -> file in bounded chunks); rank 0 also
writes meta.json and dense.npz (dense state is replicated).  Loading works for ANY world size:
global row g of a field lives in shard g % W at local row g // W (`arena.shard_layout`), so a
rank of a W'-way job collects the rows g = r', r'+W', ... from whichever old shards hold them.
State is copied INTO the trainer's existing buffers: captured CUDA graphs and peer (IPC) mappings
stay valid.  Resuming is exact: train(2) -> save -> load -> train(2) equals train(4) bit for bit
(tests/test_gpu_checkpoint.py).
"""
from __future__ import annotations

import dataclasses
import json
import os
from pathlib import Path
from typing import Dict, Iterator, Tuple

import numpy as np
import torch

from .arena import shard_layout as shard_rows     # (local_rows[F], local_base[F]) of a W-way job

FORMAT = "rs_b200.checkpoint.v1"
CHUNK_ROWS = 1 << 20                     # rows per host staging chunk (192 MB at d = 16)


# ------------------------------------------------------------------ layout (pure numpy, CPU-testable)
def shard_path(directory, rank: int, world: int) -> Path:
    return Path(directory) / f"tables.rank{rank}of{world}.bin"


def write_shard(path, chunks: Iterator[np.ndarray]) -> int:
    """Append the chunks ([n, 3, d] fp32, C-contiguous) to `path`; returns the rows written."""
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
    `old_rank` become which local rows of rank `new_rank` in a `new_world`-way job."""
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
    """Yield (dst_rows int64[n], records float32[n, 3, d]) for rank `new_rank` of a `new_world`-way job."""
    d, W = int(meta["embed_dim"]), int(meta["world"])
    maps = {}
    for s, src, dst in reshard_plan(meta["rows_per_field"], W, new_world, new_rank, chunk_rows):
        if s not in maps:
            p = shard_path(directory, s, W)
            n = os.path.getsize(p) // (3 * d * 4)
            maps[s] = np.memmap(p, dtype=np.float32, mode="r", shape=(n, 3, d))
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


def _world_rank(trainer) -> Tuple[int, int]:
    return int(getattr(trainer, "world", 1)), int(getattr(trainer, "rank", 0))


def _id_map(trainer) -> str:
    return "hash" if getattr(trainer, "idmap", None) is not None else "mod"


def save_checkpoint(trainer, directory, step: int | None = None) -> Path:
    """Write `trainer`'s tables, sparse-Adam state, dense weights and dense-Adam state.  Collective
    for a ShardedAutoIntTrainer: every rank calls it; the caller barriers before reading."""
    directory = Path(directory)
    directory.mkdir(parents=True, exist_ok=True)
    W, r = _world_rank(trainer)
    torch.cuda.synchronize(trainer.dev)
    arena = trainer.arena                                    # [n_local, 3, d]
    n, d = arena.shape[0], arena.shape[2]
    stage = torch.empty(min(n, CHUNK_ROWS), 3, d, dtype=torch.float32, pin_memory=True)

    def chunks():
        for r0 in range(0, n, CHUNK_ROWS):
            r1 = min(n, r0 + CHUNK_ROWS)
            stage[: r1 - r0].copy_(arena[r0:r1])
            torch.cuda.synchronize(trainer.dev)
            yield stage[: r1 - r0].numpy()

    write_shard(shard_path(directory, r, W), chunks())
    if r == 0:
        # a reused directory may hold table shards of an earlier save at another world size: remove them so
        # that the directory only ever describes ONE checkpoint (meta.json names the world size that counts)
        for stale in directory.glob("tables.rank*of*.bin"):
            if not stale.name.endswith(f"of{W}.bin"):
                stale.unlink()
        dense = {}
        for name, shape, off in trainer.spec:
            k = int(np.prod(shape))
            dense[name] = trainer.flat[off:off + k].view(shape).cpu().numpy()
            dense["m/" + name] = trainer.flat_m[off:off + k].view(shape).cpu().numpy()
            dense["v/" + name] = trainer.flat_v[off:off + k].view(shape).cpu().numpy()
        dense["adam_scalars"] = trainer.adam_scalars.cpu().numpy()
        np.savez(directory / "dense.npz", **dense)
        if _id_map(trainer) == "hash":
            np.savez(directory / "idmap.npz", **trainer.idmap.state())
        elif (directory / "idmap.npz").exists():           # left by an earlier hash-mode save into this directory
            (directory / "idmap.npz").unlink()
        meta = {
            "format": FORMAT, "world": W, "embed_dim": int(d),
            "rows_per_field": [int(x) for x in trainer.rows_host],
            "record": "[w|m|v] fp32, row stride 3*embed_dim",
            "dense_spec": [[nm, list(sh)] for nm, sh, _ in trainer.spec],
            "config": _cfg_dict(trainer.cfg), "step": step,
        }
        if _id_map(trainer) == "hash":
            meta["id_map"] = "hash"
        tmp = directory / "meta.json.tmp"
        tmp.write_text(json.dumps(meta, indent=1))
        os.replace(tmp, directory / "meta.json")
    return directory


def read_meta(directory) -> dict:
    meta = json.loads((Path(directory) / "meta.json").read_text())
    if meta.get("format") != FORMAT:
        raise ValueError(f"{directory}: not a {FORMAT} checkpoint (format = {meta.get('format')!r})")
    return meta


def load_checkpoint(trainer, directory, tables: bool = True, dense: bool = True) -> dict:
    """Restore `trainer` in place from `directory` (any world size).  Raises ValueError when the
    table geometry or the dense parameter shapes differ."""
    directory = Path(directory)
    meta = read_meta(directory)
    W, r = _world_rank(trainer)
    if meta.get("id_map", "mod") != _id_map(trainer):
        raise ValueError(f"checkpoint id_map={meta.get('id_map', 'mod')!r} does not match the trainer's "
                         f"id_map={_id_map(trainer)!r}")
    if tables:
        if [int(x) for x in trainer.rows_host] != meta["rows_per_field"] or trainer.arena.shape[2] != meta["embed_dim"]:
            raise ValueError("checkpoint tables do not match the trainer's rows_per_field / embed_dim")
        for s in range(meta["world"]):
            if not shard_path(directory, s, meta["world"]).exists():
                raise FileNotFoundError(shard_path(directory, s, meta["world"]))
        arena = trainer.arena
        for dst, rec in load_shard_rows(directory, meta, W, r):
            t = torch.from_numpy(np.array(rec, np.float32, copy=True)).to(trainer.dev)
            if dst.size and (np.diff(dst) == 1).all():
                arena[int(dst[0]): int(dst[-1]) + 1].copy_(t)
            else:
                arena.index_copy_(0, torch.from_numpy(dst).to(trainer.dev), t)
        if _id_map(trainer) == "hash":
            with np.load(directory / "idmap.npz") as z:
                trainer.idmap.load_state({k: z[k] for k in z.files})
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
    torch.cuda.synchronize(trainer.dev)
    if W > 1:
        # the next step's peer gather reads the OTHER ranks' shards at its very start: nobody may run ahead of a
        # rank that is still copying its shard in
        import torch.distributed as dist
        dist.barrier(group=getattr(getattr(trainer, "ex", None), "group", None))
    return meta


def _refresh_dense_shadows(trainer):
    if hasattr(trainer, "flat_bf16"):
        trainer.flat_bf16.copy_(trainer.flat)
    if hasattr(trainer, "WT16"):                 # bf16 activations: transposed bf16 weight shadows
        trainer._refresh_wt()


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
