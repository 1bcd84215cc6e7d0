"""ctypes binding of the C-ABI in include/rs_b200.h (librs_b200.so, sm_100a only).

There is no CPU fallback and no alternative backend: if the shared library is
missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "_lib" / "librs_b200.so"

RS_F32, RS_BF16 = 0, 1
(EPI_NONE, EPI_BIAS, EPI_BIAS_RELU, EPI_BIAS_SIGMOID, EPI_MUL_RELU_MASK, EPI_MUL_DSIGMOID,
 EPI_ACCUM) = range(7)
DIN_A, DIN_B = 0, 1
PATH_NONE, PATH_FFMA, PATH_TCGEN05 = 0, 1, 2
RS_MAX_PEERS = 8          # ranks a peer-memory kernel addresses (one NVSwitch domain)

_p, _i, _i64, _f, _sz, _u64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t, C.c_uint64

# name -> (restype, argtypes); mirrors include/rs_b200.h one to one.
PROTOTYPES = {
    "rs_abi_version": (_i, []),
    "rs_debug_timestamp": (_i, [_p, _p]),
    "rs_last_error": (C.c_char_p, []),
    "rs_launch_count": (_u64, []),
    "rs_built_for_sm100a": (_i, []),
    "rs_embed_gather_fwd": (_i, [_p, _p, _p, _p, _i64, _i, _i, _p, _i, _p, _p, _p]),
    "rs_embed_gather_fwd_ld": (_i, [_p, _i64, _p, _p, _p, _i64, _i, _i, _p, _i, _p, _p, _p]),
    "rs_embed_gather_rows": (_i, [_p, _p, _i64, _i, _p, _i, _p, _p, _p]),
    "rs_embed_gather_rows_ld": (_i, [_p, _i64, _p, _i64, _i, _p, _i, _p, _p, _p]),
    "rs_embed_gather_bag_mean": (_i, [_p, _p, _p, _p, _p, _i64, _i, _i, _p, _i, _p]),
    "rs_embed_bag_fwd_ld": (_i, [_p, _i64, _p, _p, _p, _p, _i64, _i, _i, _p, _i, _p, _p, _p]),
    "rs_embed_bag_grad": (_i, [_p, _i, _p, _p, _i64, _i, _p, _p]),
    "rs_embed_sort_workspace_bytes": (_sz, [_i64]),
    "rs_embed_gather_peer_fwd": (_i, [_p, _i64, _i, _p, _p, _p, _i64, _i, _i, _p, _i, _p]),
    "rs_scatter_rows_peer": (_i, [_p, _p, _i, _i, _p, _i64, _i, _i, _p]),
    "rs_peer_barrier": (_i, [_p, _i, _i, _p]),
    "rs_embed_keys_from_rows": (_i, [_p, _i64, _p, _p]),
    "rs_ipc_export": (_i, [_p, _p, _p]),
    "rs_ipc_import": (_i, [_p, _u64, _p]),
    "rs_embed_sort_keys": (_i, [_p, _p, _i64, _i, _p, _sz, _p]),
    "rs_embed_segsum_adam": (_i, [_p, _p, _p, _p, _i, _p, _i64, _i, _f, _f, _f, _f, _p, _f, _p]),
    "rs_embed_segsum_adam_ld": (_i, [_p, _p, _p, _i64, _p, _i, _p, _i64, _i, _f, _f, _f, _f, _p, _f, _p]),
    "rs_embed_segsum_adagrad": (_i, [_p, _p, _p, _i, _p, _i64, _i, _f, _f, _i, _f, _p]),
    "rs_embed_segsum": (_i, [_p, _i, _p, _i64, _i, _p, _p, _p]),
    "rs_adam_advance": (_i, [_p, _f, _f, _p]),
    "rs_dense_adam": (_i, [_p, _p, _p, _p, _i64, _f, _f, _f, _f, _p, _p, _p]),
    "rs_route_workspace_bytes": (_sz, [_i64, _i]),
    "rs_route_ids": (_i, [_p, _i64, _i, _p, _p, _i, _p, _p, _p, _p, _p, _sz, _p]),
    "rs_route_ids_padded": (_i, [_p, _i64, _i, _p, _p, _i, _i, _p, _p, _p, _p, _p, _sz, _p]),
    "rs_route_ids_padded_spread": (_i, [_p, _i64, _i, _p, _p, _i, _i, _p, _p, _p, _p, _p, _sz, _p]),
    "rs_permute_rows": (_i, [_p, _p, _p, _i64, _i, _i, _i, _p]),
    "rs_idmap_insert": (_i, [_p, _p, _p, _p, _i, _p, _i64, _i, _p, _u64, _f, _p, _i64, _i, _p, _i64, _i, _f,
                             _p, _i64, _i, _f, _p]),
    "rs_idmap_lookup": (_i, [_p, _p, _p, _i, _p, _i64, _i, _p, _p, _i, _p]),
    "rs_idmap_rebuild": (_i, [_p, _i64, _p, _p, _p, _i, _i64, _p]),
    "rs_idmap_count": (_i, [_p, _p, _i64, _p]),
    "rs_idmap_evict_workspace_bytes": (_sz, [_i64]),
    "rs_idmap_evict": (_i, [_p, _i64, _p, _p, _p, _i, _i64, _p, _f, _f, _p, _i64, _i, _p, _i64, _i, _p, _i64, _i, _p,
                            _p, _sz, _p]),
    "rs_interacting_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "rs_interacting_saved_bytes": (_sz, [_i, _i, _i, _i]),
    "rs_interacting_path": (_i, [_i, _i, _i, _i, _i, _i, _f]),
    "rs_interacting_fwd_gather": (_i, [_p, _i64, _i, _p, _p, _p, _p, _i64, _i64, _p, _i, _p, _p, _p, _p, _f, _p, _i64, _i64, _p,
                                       _i, _i, _i, _i, _i, _i, _i, _p]),
    "rs_interacting_fwd_gather_bag": (_i, [_p, _i64, _p, _p, _p, _p, _p, _i64, _i64, _p, _p, _i, _p, _p, _p, _p, _f, _p,
                                           _i64, _i64, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "rs_interacting_bwd_scatter": (_i, [_p, _i64, _i64, _p, _i, _p, _p, _p, _p, _f, _p, _i64, _i64, _p, _i64, _i64, _p,
                                        _p, _i, _i, _p, _i, _p, _i, _i, _i, _i, _i, _i, _i, _p, _sz, _p]),
    "rs_interacting_bwd_reduce": (_i, [_p, _sz, _p, _i, _i, _i, _i, _i, _p]),
    "rs_interacting_fwd": (_i, [_p, _i64, _i64, _i, _p, _p, _p, _p, _f, _p, _i64, _i64, _p,
                                _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "rs_interacting_fwd_dropout": (_i, [_p, _i64, _i64, _i, _p, _p, _p, _p, _f, _p, _i64, _i64, _p,
                                        _i, _i, _i, _i, _i, _i, _i, _i, _f, _u64, _p, _p]),
    "rs_interacting_bwd_dropout": (_i, [_p, _i64, _i64, _p, _i, _p, _p, _p, _p, _f, _p, _i64, _i64, _p, _i64, _i64, _p,
                                        _i, _i, _i, _i, _i, _i, _i, _i, _f, _u64, _p, _p, _sz, _p]),
    "rs_interacting_bwd": (_i, [_p, _i64, _i64, _p, _i, _p, _p, _p, _p, _f, _p, _i64, _i64, _p, _i64, _i64, _p,
                                _i, _i, _i, _i, _i, _i, _i, _i, _p, _sz, _p]),
    "rs_din_fwd": (_i, [_i, _p, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "rs_din_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "rs_din_bwd": (_i, [_i, _p, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p,
                        _i, _i, _i, _i, _p, _sz, _p]),
    "rs_gemm_workspace_bytes": (_sz, []),
    "rs_gemm": (_i, [_p, _i64, _i, _p, _i64, _i, _p, _i64, _p, _p, _i64, _i, _i, _i, _i, _i, _i, _p, _sz, _p]),
    "rs_colsum_workspace_bytes": (_sz, [_i, _i]),
    "rs_colsum": (_i, [_p, _i64, _i, _p, _i, _i, _p, _sz, _p]),
    "rs_act_bwd": (_i, [_p, _i64, _p, _i64, _p, _i64, _i, _i, _i, _i, _p]),
    "rs_copy2d": (_i, [_p, _i64, _i, _p, _i64, _i, _i, _i, _p]),
    "rs_add2d": (_i, [_p, _i64, _p, _i64, _p, _i64, _i, _i, _i, _p]),
    "rs_bce_sigmoid_fwd_bwd": (_i, [_p, _i, _p, _f, _p, _p, _i, _i, _p]),
    "rs_logit_head_workspace_bytes": (_sz, [_i, _i]),
    "rs_logit_head_fwd_bwd": (_i, [_p, _i64, _i, _p, _p, _p, _f, _p, _p, _p, _i64, _p, _p, _i, _i, _p, _sz, _p]),
    "rs_logit_head_fwd_bwd_relu": (_i, [_p, _i64, _i, _p, _p, _p, _f, _p, _p, _p, _i64, _p, _p, _i, _i, _i, _p, _sz, _p]),
    "rs_logit_head_reduce": (_i, [_p, _sz, _p, _p, _p, _i, _i, _p]),
    "rs_logit_head_grad": (_i, [_p, _i64, _i, _p, _p, _f, _i, _i, _p, _sz, _p]),
    "rs_tower_supported": (_i, [_i, _i, _i, _i]),
    "rs_tower_step": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _f, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "rs_tower_fwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "rs_cross_workspace_bytes": (_sz, [_i, _i, _i]),
    "rs_cross_fwd": (_i, [_p, _i64, _i, _p, _p, _p, _i64, _i, _i, _i, _p, _sz, _p]),
    "rs_cross_bwd": (_i, [_p, _i64, _p, _i64, _i, _p, _p, _p, _i64, _p, _p, _i, _i, _i, _p, _sz, _p]),
    "rs_transpose2d": (_i, [_p, _i64, _p, _i64, _i, _i, _i, _p]),
    "rs_set_fp32_gemm_mode": (_i, [_i]),
    "rs_staytime_labels": (_i, [_p, _p, _p, _i, _i, _p, _p, _p, _p, _i64, _i64, _f, _f, _f, _f, _f, _p]),
    "rs_binary_metrics_state_bytes": (_sz, [_i]),
    "rs_binary_metrics_workspace_bytes": (_sz, [_i64]),
    "rs_binary_metrics_update": (_i, [_p, _i, _p, _i64, _p, _i, _f, _p, _p, _sz, _p]),
    "rs_binary_metrics_result": (_i, [_p, _i, _p, _p]),
}

_lib = None
MISSING: list[str] = []


class RsError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load librs_b200.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RsError(
            f"{LIB_PATH} is missing: build it with `python -m recommendsystem_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            MISSING.append(name)  # tests assert this stays empty; calling it raises
            continue
        fn.restype = res
        fn.argtypes = args
    if lib.rs_built_for_sm100a() != 1:
        raise RsError("librs_b200.so was not built for sm_100a")
    _lib = lib
    return lib


def call(name: str, *args):
    """Call an int-returning entry point; raise RsError(rs_last_error()) on failure."""
    lib = load()
    if name in MISSING:
        raise RsError(f"{name} is declared in include/rs_b200.h but missing from {LIB_PATH}")
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RsError(f"{name} failed ({rc}): {lib.rs_last_error().decode(errors='replace')}")
    return rc


def launch_count() -> int:
    return int(load().rs_launch_count())
