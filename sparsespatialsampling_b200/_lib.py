"""
ctypes binding of ``libs3b200.so`` (the C-ABI declared in ``include/s3b200.h``).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C sparsespatialsampling_b200/csrc``.
There is no CPU fallback: if the shared library is missing or no CUDA device is present, every compute
call raises.
"""
import ctypes
import os
from ctypes import c_int, c_int32, c_int64, c_void_p, c_char_p, c_double, POINTER

import torch as pt

_HERE = os.path.dirname(os.path.abspath(__file__))
# S3B200_LIB: alternative build of the same library (A/B measurements of kernel changes)
LIB_PATH = os.environ.get("S3B200_LIB") or os.path.join(_HERE, "libs3b200.so")

S3_F32 = 0
S3_F64 = 1

_lib = None


class S3Error(RuntimeError):
    pass


# name -> (restype, argtypes); mirrors include/s3b200.h one to one
_SIGNATURES = {
    "s3_last_error": (c_char_p, []),
    "s3_version": (c_int, []),
    "s3_launch_count": (c_int64, []),
    "s3_knn_build": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, POINTER(c_void_p)]),
    "s3_knn_free": (c_int, [c_void_p]),
    "s3_knn_query": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "s3_knn_predict": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "s3_knn_tables": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "s3_morton_order": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "s3_cells_refine": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_double, c_void_p]),
    "s3_cells_gain": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_double, c_double, c_int,
                              c_void_p, c_void_p, c_void_p]),
    "s3_cells_mask": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_double, c_void_p, c_void_p, c_int,
                              c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "s3_nodes_mask": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                              c_int, c_void_p, c_void_p]),
    "s3_points_inside": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                 c_void_p]),
    "s3_select_topk": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "s3_select_set_fused": (c_int, [c_int]),
    "s3_topo_create": (c_int, [c_int, c_void_p, c_double, c_int, POINTER(c_void_p)]),
    "s3_topo_sync": (c_int, [c_void_p]),
    "s3_topo_free": (c_int, [c_void_p]),
    "s3_topo_n_cells": (c_int64, [c_void_p]),
    "s3_topo_n_nodes": (c_int64, [c_void_p]),
    "s3_topo_refine": (c_int, [c_void_p, c_void_p, c_int64]),
    "s3_topo_refresh": (c_int, [c_void_p, c_void_p, c_int64, c_int]),
    "s3_topo_mark_invalid": (c_int, [c_void_p, c_void_p, c_int64]),
    "s3_topo_check_nb": (c_int64, [c_void_p, c_int64, c_void_p]),
    "s3_topo_cell": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "s3_topo_final": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64), c_void_p, c_void_p, c_void_p]),
    "s3_leaf_sumsq": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "s3_sumsq": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "s3_interp_gather": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_int, c_void_p,
                                 c_void_p, c_int, c_void_p]),
    "s3_interp_gather_strided": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, c_int64, c_int64, c_void_p, c_void_p,
                                         c_int64, c_int, c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p]),
    "s3_recon_error": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, c_int64, c_int64, c_void_p, c_int, c_int64,
                               c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p]),
    "s3_copy2d_async": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p]),
    "s3_gather_rows": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int, c_void_p]),
    "s3_svd_row_means": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "s3_svd_gram": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int64, c_int, c_void_p, c_void_p]),
    "s3_svd_project": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p]),
    "s3_svd_project_tc": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int64, c_int, c_int,
                                  c_void_p, c_void_p]),
}


def exported_symbols():
    """Names of all entry points declared in include/s3b200.h."""
    return sorted(_SIGNATURES)


def load():
    """Load the shared library (no CUDA call is made here)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise S3Error(f"{LIB_PATH} not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          f"or `make -C sparsespatialsampling_b200/csrc`. There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        # A/B harness hook of the kernels (s3x_tune, not part of include/s3b200.h): S3B200_TUNE="key=value,..."
        lib.s3x_tune.restype, lib.s3x_tune.argtypes = c_int, [c_int, c_int]
        for kv in [t for t in os.environ.get("S3B200_TUNE", "").split(",") if t]:
            key, value = kv.split("=")
            check(lib.s3x_tune(int(key), int(value)))
    return _lib


def check(rc: int):
    if rc != 0:
        msg = load().s3_last_error()
        raise S3Error(f"s3b200 error {rc}: {msg.decode() if msg else '?'}")


def require_cuda():
    if not pt.cuda.is_available():
        raise S3Error("s3b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback.")


def ptr(t, strided: bool = False):
    """Device pointer of a (contiguous) tensor, or NULL for None; ``strided``: the call passes the strides itself."""
    if t is None:
        return None
    assert strided or t.is_contiguous(), "tensor passed to the C-ABI must be contiguous"
    return c_void_p(t.data_ptr())


def stream_ptr():
    return c_void_p(pt.cuda.current_stream().cuda_stream)


def tune(key: int, value: int) -> None:
    """A/B harness hook (scripts/interp_lab.py): kernel launch knobs, see csrc/interp.cu."""
    check(load().s3x_tune(int(key), int(value)))


def launch_count() -> int:
    return int(load().s3_launch_count())
