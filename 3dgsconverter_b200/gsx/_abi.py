"""ctypes binding of libgsx.so (include/gsx.h).  No torch types cross this boundary.

The library is built in-tree by ``__graft_entry__.build()`` (3dgsconverter_b200/lib/libgsx.so).
There is NO CPU fallback: if the shared object is missing this module raises at import.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent.parent
LIB_PATH = Path(os.environ.get("GSX_LIB", _PKG / "lib" / "libgsx.so"))


class GsxError(RuntimeError):
    """A libgsx entry point returned a non-zero status."""


if not LIB_PATH.exists():
    raise ImportError(
        f"libgsx.so not found at {LIB_PATH}: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(nvcc, sm_100a).  gsx has no CPU fallback.")

lib = C.CDLL(str(LIB_PATH))

_f32p = C.POINTER(C.c_float)
_vp = C.c_void_p
_i64 = C.c_int64
_i32 = C.c_int32

_SIGS = {
    "gsx_last_error": (C.c_char_p, []),
    "gsx_version": (C.c_int, []),
    "gsx_build_info": (C.c_char_p, []),
    "gsx_device_sm_count": (C.c_int, []),
    "gsx_kernel_launches": (C.c_longlong, []),
    "gsx_sor_workspace_bytes": (_i64, [_i64]),
    "gsx_sor_grid_workspace_bytes": (_i64, [_i64]),
    "gsx_sor_minmax": (C.c_int, [_vp, _i64, _vp, _vp, _i64, _vp]),
    "gsx_sor_cell_size": (C.c_float, [_f32p, _i64]),
    "gsx_sor_build": (C.c_int, [_vp, _i64, _f32p, C.c_float, _vp, _i64, _vp]),
    "gsx_sor_dist_local_run": (C.c_int, [_vp, _i64, _i64, _i64, _i32, _f32p, C.c_float, _vp, _vp, _vp, _i64, _vp]),
    "gsx_sor_dist_merge": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _f32p, C.c_float, _vp, _vp, _vp, _i64, _vp]),
    "gsx_sor_spos_offset": (_i64, [_i64]),
    "gsx_sor_build_from_sorted": (C.c_int, [_vp, _vp, _i64, _f32p, C.c_float, _vp, _i64, _vp]),
    "gsx_sor_mean_dists": (C.c_int, [_i64, _i32, _i32, _f32p, C.c_float, _vp, _i64, _vp, _vp, _vp]),
    "gsx_sor_mean_dists_range": (C.c_int, [_i64, _i64, _i64, _i32, _i32, _f32p, C.c_float, _vp, _i64, _vp, _vp, _vp]),
    "gsx_sor_mean_dists_strided": (C.c_int, [_i64, _i32, _i32, _i32, _i32, _f32p, C.c_float, _vp, _i64, _vp, _vp, _vp]),
    "gsx_sort_pairs_workspace_bytes": (_i64, [_i64]),
    "gsx_sort_pairs": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _i64, _vp]),
    "gsx_mean_std_workspace_bytes": (_i64, [_i64]),
    "gsx_mean_std_f32": (C.c_int, [_vp, _i64, _vp, _vp, _i64, _vp]),
    "gsx_pairwise_slots": (_i64, [_i64]),
    "gsx_pairwise_leaves_dist": (C.c_int, [_vp, _i64, _i64, _i64, _i32, _vp, _vp, _vp, _i32, _vp, _vp]),
    "gsx_pairwise_finish": (C.c_int, [_vp, _i64, _i32, _vp, _vp]),
    "gsx_threshold_mask": (C.c_int, [_vp, _i64, _vp, C.c_float, _vp, _vp]),
    "gsx_sor_filter_device": (C.c_int, [_vp, _i64, _i32, C.c_float, _i32, _vp, _vp, _vp, _i64, _vp]),
    "gsx_sor_filter_host": (C.c_int, [_vp, _i64, _i32, C.c_float, _i32, _vp, _vp]),
    "gsx_knn_exact_workspace_bytes": (_i64, [_i64]),
    "gsx_knn_exact_mean_dists": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _i64, _vp]),
    "gsx_sor_ckdtree_filter_host": (C.c_int, [_vp, _i64, _i32, C.c_float, _vp, _vp]),
    "gsx_bbox_mask": (C.c_int, [_vp, _i64, _f32p, _vp, _vp]),
    "gsx_alpha_mask": (C.c_int, [_vp, _i64, C.c_double, _vp, _vp]),
    "gsx_alpha_logit_threshold": (C.c_double, [C.c_double]),
    "gsx_compact_workspace_bytes": (_i64, [_i64]),
    "gsx_compact_points": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(_i64), _vp, _i64, _vp]),
    "gsx_density_workspace_bytes": (_i64, [_i64, _i64]),
    "gsx_density_voxel_count": (C.c_int, [_vp, _i64, C.c_float, _i64, _vp, _vp, _i64, C.POINTER(_i64),
                                          C.POINTER(_i64), _vp, _i64, _vp]),
    "gsx_density_member_mask": (C.c_int, [_vp, _i64, C.c_float, _vp, _i64, _vp, _vp, _i64, _vp]),
    "gsx_density_voxel_range": (None, [_f32p, C.c_float, C.POINTER(_i64), C.POINTER(_i64)]),
    "gsx_density_grid_count": (C.c_int, [_vp, _i64, C.c_float, C.POINTER(_i64), C.POINTER(_i64), _vp, _vp, _vp]),
    "gsx_density_grid_dense": (C.c_int, [_vp, C.POINTER(_i64), C.POINTER(_i64), _i64, _vp, _vp, _i64,
                                         C.POINTER(_i64), C.POINTER(_i64), _vp, _i64, _vp]),
    "gsx_lexsort_workspace_bytes": (_i64, [_i64]),
    "gsx_lexsort_zyx": (C.c_int, [_vp, _i64, _vp, _vp, _i64, _vp]),
    "gsx_quantize_to_codebook": (C.c_int, [_vp, _i64, _f32p, _i32, _vp, _vp, _i64, _vp]),
    "gsx_kmeans_workspace_bytes": (_i64, [_i64, _i32, _i32, _i32]),
    "gsx_kmeans_lloyd_device": (C.c_int, [_vp, C.POINTER(_i64), _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _i64,
                                          _i32, _vp, _vp]),
    "gsx_kmeans_tensor_core_supported": (_i32, [_i32, _i32]),
    "gsx_kmeans_tc_debug_scores": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _i32, _vp, _vp, _i64, _vp]),
    "gsx_kmeans_host": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _vp, _vp, _i32]),
    "gsx_kmeans_host_batched": (C.c_int, [_vp, C.POINTER(_i64), _i32, _i32, _i32, _i32, _vp, _vp, _i32]),
    "gsx_records_extract_xyz_opacity": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "gsx_records_gather_rows": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "gsx_records_color_rgba8": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _i32, _i32, C.c_float, _vp, _vp]),
    "gsx_records_scale_exp": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp]),
    "gsx_morton_workspace_bytes": (_i64, [_i64]),
    "gsx_morton_order": (C.c_int, [_vp, _i64, _vp, _i32, C.POINTER(_i32), _vp, _i64, _vp]),
    "gsx_chunk_minmax": (C.c_int, [_vp, _i64, _i32, _vp, _i32, C.POINTER(_i32), _i32, C.c_float, C.c_float, _vp, _vp, _vp,
                                   _i64, _vp]),
    "gsx_copy_h2d": (C.c_int, [_vp, _vp, _i64, _vp]),
    "gsx_copy_d2h": (C.c_int, [_vp, _vp, _i64, _vp]),
    "gsx_host_gather_rows": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp]),
    "gsx_host_extract_xyz_opacity": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp]),
    "gsx_device_memory": (C.c_int, [C.POINTER(_i64), C.POINTER(_i64)]),
}

for _name, (_res, _args) in _SIGS.items():
    _fn = getattr(lib, _name)  # AttributeError here == a symbol declared in gsx.h is missing
    _fn.restype = _res
    _fn.argtypes = _args

HASH_MODES = {"i32wrap": 0, "i64": 1}
KM_ASSIGN = {"auto": 0, "strict": 1, "fma": 2, "tensor": 3, "tensor_bf16": 4}


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib.gsx_last_error().decode("utf-8", "replace")
        raise GsxError(f"{what or 'gsx'} failed (status {rc}): {msg}")


def workspace_size(name: str, *args) -> int:
    """Byte size from a *_workspace_bytes entry point; a negative result (n out of range) raises GsxError."""
    nbytes = getattr(lib, name)(*args)
    check(nbytes if nbytes < 0 else 0, name)
    return nbytes


def f32x(*vals):
    return (C.c_float * len(vals))(*[float(v) for v in vals])
