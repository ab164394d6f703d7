"""ctypes binding of ``libagx_b200.so`` - the only way the Python host layer reaches the GPU kernels.

Signatures mirror ``include/agx_b200.h`` one to one.  There is NO CPU fallback: if the shared library
has not been built, or no CUDA device is present, every compute call raises.
"""

from __future__ import annotations

import ctypes
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_void_p
from pathlib import Path

import torch

LIB_PATH = Path(__file__).resolve().parent / "lib" / "libagx_b200.so"

ABI_VERSION = 4
AGX_OK = 0
AGX_ERR_CUDA = -1
AGX_ERR_ARG = -2
AGX_ERR_UNSUPPORTED = -3
AGX_ERR_OVERFLOW = -4

NORM_CODES = {None: 0, "l1": 1, "l2": 2, "unit-max": 3, "unit-range": 4, "unit-std": 5}

# name -> (restype, argtypes); must list every symbol include/agx_b200.h declares
SIGNATURES = {
    "agx_last_error": (c_char_p, []),
    "agx_abi_version": (c_int, []),
    "agx_launch_count": (c_int64, []),
    "agx_index_build": (c_int, [c_void_p, c_int64, c_int, c_int, c_double, c_void_p, POINTER(c_void_p)]),
    "agx_index_free": (c_int, [c_void_p, c_void_p]),
    "agx_index_info": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int)]),
    "agx_search_vectors": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "agx_knn": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_int, c_double, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p],
    ),
    "agx_knn_flagged": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_int, c_double, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "agx_knn_redecide": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_double, c_void_p, c_void_p, c_void_p]),
    "agx_knn_redecide_ranked": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_int, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "agx_knn_redecide_list": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_int, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "agx_compact_flags": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "agx_set_query_order_mode": (None, [c_int]),
    "agx_last_query_order": (c_int, []),
    "agx_radius_count": (c_int, [c_void_p, c_void_p, c_int64, c_double, c_void_p, c_void_p]),
    "agx_exclusive_scan": (c_int, [c_void_p, c_int64, c_void_p, POINTER(c_int64), c_void_p]),
    "agx_radius_fill": (c_int, [c_void_p, c_void_p, c_int64, c_double, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "agx_max_positive": (c_int, [c_void_p, c_int64, POINTER(c_double), POINTER(c_int64), c_void_p]),
    "agx_host_reference_rdist": (c_int, [c_void_p, c_void_p, c_int64, c_int, POINTER(c_double)]),
    "agx_order_resolve": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "agx_gate_supported": (c_int, []),
    "agx_gate_wait": (c_int, [c_void_p, c_void_p]),
    "agx_gate_open": (c_int, [c_void_p, c_void_p]),
    "agx_mark_nodes": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "agx_relabel_nodes": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "agx_restrict_flags": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_double, c_void_p, c_void_p],
    ),
    "agx_sort_edges": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p]),
    "agx_gather_edge_columns": (
        c_int,
        [c_int, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_void_p, c_int64, c_void_p],
    ),
    "agx_set_output_maps": (None, [c_void_p, c_void_p]),
    "agx_concat_edges": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, POINTER(c_int64), c_void_p],
    ),
    "agx_relabel_rows": (c_int, [POINTER(c_void_p), POINTER(c_int64), c_int, c_void_p, c_void_p]),
    "agx_node_tables": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "agx_edge_attrs": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int,
         c_void_p, c_void_p, c_int, c_void_p],
    ),  # fmt: skip
    "agx_edge_attrs_workspace": (c_int64, []),
    "agx_edge_attrs_stats": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
         c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p],
    ),  # fmt: skip
    "agx_edge_attrs_apply": (
        c_int,
        [c_int64, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p],
    ),
    "agx_edge_azimuth": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p],
    ),
    "agx_gaussian_weights": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_double, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "agx_gaussian_weights_scratch_bytes": (c_int64, [c_int64, c_int64]),
    "agx_icosphere": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "agx_multiscale_tri_count": (
        c_int,
        [c_int, c_void_p, POINTER(c_int32), c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "agx_multiscale_scratch_per_node": (c_int64, [c_int, c_int]),
    "agx_multiscale_tri_count_mapped": (
        c_int,
        [c_int, c_void_p, POINTER(c_int32), c_int, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "agx_multiscale_tri_fill": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "agx_voronoi_areas": (
        c_int,
        [c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p, c_int64, c_double, c_void_p, c_void_p, c_void_p],
    ),
    "agx_voronoi_areas_small": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_double, c_void_p, c_void_p, c_void_p]),
    "agx_healpix_nodes": (c_int, [c_int, c_void_p, c_void_p]),
    "agx_gaussian_latitudes": (c_int, [c_int, c_void_p, c_void_p]),
    "agx_octahedral_nodes": (c_int, [c_int, c_void_p, c_void_p, c_void_p]),
    "agx_hex_num_cells": (c_int64, [c_int]),
    "agx_hex_cells": (c_int, [c_int, c_void_p, c_void_p, c_void_p]),
    "agx_hex_adjacency": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "agx_multiscale_adj_count": (
        c_int,
        [c_int, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), c_int, c_int, c_int64,
         c_void_p, c_void_p, c_void_p],
    ),  # fmt: skip
}

_lib = None


class AgxError(RuntimeError):
    """A CUDA-side failure reported by libagx_b200."""


def load_library(path: Path | None = None) -> ctypes.CDLL:
    """Load (once) and type the shared library.  Raises if it has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path is not None else LIB_PATH
    if not p.exists():
        raise RuntimeError(
            f"{p} is missing: the CUDA extension has not been built. Run `python -m anemoi_graphs_b200._build` "
            "(needs nvcc). This package has no CPU fallback."
        )
    lib = ctypes.CDLL(str(p))
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.agx_abi_version() != ABI_VERSION:
        raise RuntimeError(f"{p}: ABI version {lib.agx_abi_version()} != {ABI_VERSION}; rebuild the library")
    if path is None:
        _lib = lib
    return lib


def require_cuda() -> None:
    if not torch.cuda.is_available():
        raise RuntimeError(
            "anemoi_graphs_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback for the "
            "edge-construction path."
        )


def check(rc: int) -> None:
    """Map a library return code onto the exception type the reference would raise."""
    if rc == AGX_OK:
        return
    msg = load_library().agx_last_error().decode(errors="replace")
    if rc == AGX_ERR_ARG:
        raise ValueError(msg)
    if rc == AGX_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise AgxError(f"libagx_b200 error {rc}: {msg}")


def ptr(t: torch.Tensor | None) -> int | None:
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "C-ABI buffers must be contiguous CUDA tensors"
    return t.data_ptr()


def current_stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
    return int(load_library().agx_launch_count())
