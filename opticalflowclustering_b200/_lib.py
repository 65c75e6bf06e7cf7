"""ctypes binding of libofc.so (C-ABI declared in include/ofc.h).

There is no CPU fallback: if the CUDA library is missing the import of any
operator fails loudly with instructions to build it.
"""
from __future__ import annotations

import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(PKG, "libofc.so")

OFC_OK, OFC_ERR_INVALID, OFC_ERR_UNSUPPORTED, OFC_ERR_CUDA, OFC_ERR_WORKSPACE = 0, -1, -2, -3, -4
#: OR-ed into the dtype of the stepwise k-means calls: every problem of the batch reads the same rows
OFC_KMEANS_SHARED_ROWS = 0x100

_vp, _i, _i64, _sz, _d = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_double

# name -> (restype, argtypes); mirrors include/ofc.h one to one
SIGNATURES = {
    "ofc_version": (_i, []),
    "ofc_last_error": (C.c_char_p, []),
    "ofc_profile_begin": (_i, []),
    "ofc_profile_end": (_i, [_vp, _vp, _i]),
    "ofc_flow_plan_create": (_i, [C.POINTER(_vp), _i, _i, _i, _d, _i, _i, _i, _i, _d, _i]),
    "ofc_flow_plan_destroy": (None, [_vp]),
    "ofc_flow_plan_workspace_bytes": (_sz, [_vp]),
    "ofc_flow_plan_keep_intermediates": (_i, [_vp, _i]),
    "ofc_flow_plan_num_levels": (_i, [_vp]),
    "ofc_flow_plan_level_size": (_i, [_vp, _i, C.POINTER(_i), C.POINTER(_i)]),
    "ofc_flow_plan_buffer": (_i, [_vp, _i, _i, C.POINTER(_sz), C.POINTER(_sz)]),
    "ofc_farneback_sequence": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _sz, _vp]),
    "ofc_farneback_pair": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_farneback_pair_init": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_farneback_stream_begin": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "ofc_farneback_stream_next": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_bgr2gray": (_i, [_vp, _vp, _i64, _vp]),
    "ofc_bgr2hsv": (_i, [_vp, _vp, _i64, _vp]),
    "ofc_flow_minmax": (_i, [_vp, _i, _i64, _vp, _vp]),
    "ofc_flow_to_bgr": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "ofc_flow_to_hsv": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "ofc_flow_to_bgr_grid": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "ofc_grid_cells": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ofc_draw_grid": (_i, [_vp, _i, _i, _i, _i, _i, _vp]),
    "ofc_kmeans_workspace_bytes": (_sz, [_i, _i64, _i, _i]),
    "ofc_kmeans_assign_workspace_bytes": (_sz, [_i, _i64, _i, _i]),
    "ofc_kmeans_assign": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_sums": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_step_supported": (_i, [_i, _i, _i]),
    "ofc_kmeans_step": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_centres": (_i, [_i, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_update": (_i, [_i, _i64, _i, _i, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                               _sz, _vp]),
    "ofc_minibatch_update": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "ofc_minibatch_update_weighted": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ofc_kmeans_relocate": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "ofc_kmeans_assign_weighted": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_sums_weighted": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_update_weighted": (_i, [_i, _i64, _i, _i, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp,
                                        _vp, _vp, _sz, _vp]),
    "ofc_kmeans_relocate_weighted": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "ofc_kmeans_far_points": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "ofc_kmeans_far_payload": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _i64, _vp, _vp, _vp, _vp]),
    "ofc_kmeans_relocate_merge": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ofc_peer_header_bytes": (_sz, []),
    "ofc_peer_alloc": (_i, [_sz, _vp, _vp]),
    "ofc_peer_open": (_i, [_vp, _vp]),
    "ofc_peer_close": (_i, [_vp]),
    "ofc_peer_free": (_i, [_vp]),
    "ofc_peer_exchange": (_i, [_vp, _i, _i, _sz, _i, _i64, _i64, _vp, _vp, _vp, _i, _d, _vp]),
    "ofc_peer_error": (_i, [_vp, _vp]),
    "ofc_kmeans_cells": (_i, [_vp, _i, _i64, _i, _i, _vp, C.c_uint64, _i, _d, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_grid_kmeans_cells_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i]),
    "ofc_grid_kmeans_cells": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, C.c_uint64, C.c_uint64, _i, _d, _vp, _vp, _vp, _vp,
                                   _vp, _vp, _sz, _vp]),
    "ofc_kmeans_tc_workspace_bytes": (_sz, [_i64, _i, _i]),
    "ofc_kmeans_tc_prepare": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    "ofc_kmeans_tc_assign": (_i, [_vp, _vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_tc_sums": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_tc_prepare_u8": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    "ofc_kmeans_tc_assign_u8": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_tc_sums_u8": (_i, [_vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_tc_assign_weighted": (_i, [_vp, _vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_tc_sums_weighted": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_tc_sums_u8_weighted": (_i, [_vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_distances": (_i, [_vp, _i, _i64, _i, _i, _vp, _vp, _i, _vp]),
    "ofc_kmeans_elkan_centres": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_elkan_init": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ofc_kmeans_elkan_step": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ofc_kmeans_elkan_bounds": (_i, [_i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_kmeans_elkan_inertia": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ofc_grid_extract_cells": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "ofc_sliding_cosine": (_i, [_vp, _i, _vp, _i64, _vp, _vp, _vp, _vp]),
    "ofc_row_cosine": (_i, [_vp, _i, _i64, _i, _vp, _vp, _vp]),
    "ofc_vector_distance": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, _vp]),
}

_lib = None


class OfcError(RuntimeError):
    pass


def lib():
    """The loaded libofc.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO):
            raise OfcError(
                f"{SO} not found: the CUDA extension is required (there is no CPU fallback). "
                "Build it with `python -c 'import __graft_entry__ as g; g.build()'` or "
                "`python -m opticalflowclustering_b200._build`.")
        handle = C.CDLL(SO)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)          # AttributeError if the .so is stale
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc == OFC_OK:
        return
    msg = lib().ofc_last_error().decode(errors="replace")
    if rc == OFC_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == OFC_ERR_INVALID:
        raise ValueError(msg)
    if rc == OFC_ERR_WORKSPACE:
        raise MemoryError(msg)
    raise OfcError(f"libofc error {rc}: {msg}")
