"""SOR (Taichi semantics) on device buffers: host plumbing over the gsx_sor_* C ABI.

Mirrors the staging of ``filter_sor_gpu`` (/root/reference/gsconverter/processing/gpu_ops.py:193-263):
min/max -> cell size -> hash grid build -> K-nearest mean distance -> global mean/std -> mask.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _abi
from ._abi import lib, check, HASH_MODES


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def default_hash_mode() -> str:
    import os
    return os.environ.get("GSX_SOR_HASH", "i32wrap")


def _check_xyz(xyz: torch.Tensor):
    if xyz.dim() != 2 or xyz.shape[1] != 3:
        raise ValueError("Requires 3D data")
    if not xyz.is_cuda or xyz.dtype != torch.float32 or not xyz.is_contiguous():
        raise ValueError("xyz must be a contiguous float32 CUDA tensor [N,3]")


@dataclass
class SorGrid:
    """A built hash grid living in `ws` (valid until `ws` is reused)."""
    n: int
    ws: torch.Tensor
    bmin: np.ndarray
    cell: float


def workspace(n: int, device) -> torch.Tensor:
    return torch.empty(_abi.workspace_size("gsx_sor_workspace_bytes", n), dtype=torch.uint8, device=device)


def build_grid(xyz: torch.Tensor, ws: torch.Tensor | None = None, cell_scale: float = 1.0) -> SorGrid:
    """gpu_ops.py:203-237 on device (one 24-byte D2H for the cell size).  `cell_scale` != 1 is a test hook (a finer
    grid than the reference's, to reach the many-tiny-buckets paths of the build)."""
    _check_xyz(xyz)
    n = xyz.shape[0]
    if ws is None:
        ws = workspace(n, xyz.device)
    mm_dev = torch.empty(8, dtype=torch.float32, device=xyz.device)
    check(lib.gsx_sor_minmax(_ptr(xyz), n, _ptr(mm_dev), _ptr(ws), ws.numel(), _stream()), "gsx_sor_minmax")
    mm = mm_dev[:6].cpu().numpy()
    cell = float(lib.gsx_sor_cell_size(mm.ctypes.data_as(C.POINTER(C.c_float)), n))
    if cell != cell:
        raise _abi.GsxError("sor: non-finite coordinates")
    if cell_scale != 1.0:
        cell = float(np.float32(cell * cell_scale))
    bmin = mm[:3].copy()
    check(lib.gsx_sor_build(_ptr(xyz), n, bmin.ctypes.data_as(C.POINTER(C.c_float)), cell, _ptr(ws), ws.numel(),
                            _stream()), "gsx_sor_build")
    return SorGrid(n, ws, bmin, cell)


def _stats_dict(v) -> dict:
    """The 16 counters of gsx_sor_mean_dists (gsx.h); class_cycles / class_queries are zero unless the library was
    built with -DGSX_KNN_PROFILE=1."""
    return dict(visits=int(v[0]), scanned=int(v[1]), box_tests=int(v[2]), queries=int(v[3]), group_queries=int(v[4]),
                class_cycles=[int(x) for x in v[8:12]], class_queries=[int(x) for x in v[12:16]])


def mean_dists(grid: SorGrid, k: int, hash_mode: str | None = None, out: torch.Tensor | None = None,
               want_stats: bool = False, q_range: tuple[int, int] | None = None):
    """gpu_ops.py:98-176 + unsort (:255-256).  Returns final_means (and the counters if asked)."""
    mode = HASH_MODES[hash_mode or default_hash_mode()]
    dev = grid.ws.device
    if out is None:
        out = torch.empty(grid.n, dtype=torch.float32, device=dev)
    stats = torch.zeros(16, dtype=torch.int64, device=dev) if want_stats else None
    qb, qe = q_range if q_range is not None else (0, grid.n)
    check(lib.gsx_sor_mean_dists_range(grid.n, qb, qe, int(k), mode, grid.bmin.ctypes.data_as(C.POINTER(C.c_float)),
                                       grid.cell, _ptr(grid.ws), grid.ws.numel(), _ptr(out), _ptr(stats), _stream()),
          "gsx_sor_mean_dists")
    if want_stats:
        return out, _stats_dict(stats.cpu().numpy())
    return out


def mean_dists_strided(grid: SorGrid, k: int, hash_mode: str | None, out: torch.Tensor, stride: int, phase: int,
                       want_stats: bool = False):
    """Queries the 16-position batches b with b % stride == phase (cost-balanced multi-GPU sharding)."""
    mode = HASH_MODES[hash_mode or default_hash_mode()]
    stats = torch.zeros(16, dtype=torch.int64, device=out.device) if want_stats else None
    check(lib.gsx_sor_mean_dists_strided(grid.n, int(stride), int(phase), int(k), mode,
                                         grid.bmin.ctypes.data_as(C.POINTER(C.c_float)), grid.cell, _ptr(grid.ws),
                                         grid.ws.numel(), _ptr(out), _ptr(stats), _stream()), "gsx_sor_mean_dists_strided")
    if want_stats:
        return out, _stats_dict(stats.cpu().numpy())
    return out


def mean_std(a: torch.Tensor) -> torch.Tensor:
    """np.mean / np.std (float32 pairwise) of a float32 CUDA vector -> tensor [mean, std] on device."""
    n = a.numel()
    ws = torch.empty(lib.gsx_mean_std_workspace_bytes(n), dtype=torch.uint8, device=a.device)
    out = torch.empty(2, dtype=torch.float32, device=a.device)
    check(lib.gsx_mean_std_f32(_ptr(a), n, _ptr(out), _ptr(ws), ws.numel(), _stream()), "gsx_mean_std_f32")
    return out


def threshold_mask(a: torch.Tensor, meanstd: torch.Tensor, threshold_factor: float) -> torch.Tensor:
    mask = torch.empty(a.numel(), dtype=torch.uint8, device=a.device)
    check(lib.gsx_threshold_mask(_ptr(a), a.numel(), _ptr(meanstd), float(np.float32(threshold_factor)), _ptr(mask),
                                 _stream()), "gsx_threshold_mask")
    return mask.view(torch.bool)


def sor_filter(xyz: torch.Tensor, k: int = 25, threshold_factor: float = 1.0, hash_mode: str | None = None,
               ws: torch.Tensor | None = None, return_means: bool = False):
    """Whole filter on a device tensor: bool mask [N] (and final_means if asked)."""
    _check_xyz(xyz)
    n = xyz.shape[0]
    mode = HASH_MODES[hash_mode or default_hash_mode()]
    if ws is None:
        ws = workspace(n, xyz.device)
    mask = torch.empty(n, dtype=torch.uint8, device=xyz.device)
    means = torch.empty(n, dtype=torch.float32, device=xyz.device) if return_means else None
    check(lib.gsx_sor_filter_device(_ptr(xyz), n, int(k), float(np.float32(threshold_factor)), mode, _ptr(mask),
                                    _ptr(means), _ptr(ws), ws.numel(), _stream()), "gsx_sor_filter_device")
    mask = mask.view(torch.bool)
    return (mask, means) if return_means else mask


def sor_filter_host(data_np: np.ndarray, k: int = 25, threshold_factor: float = 1.0, hash_mode: str | None = None,
                    return_means: bool = False):
    """Host-buffer entry (H2D + compute + D2H inside libgsx): what gpu_ops.filter_sor_gpu binds."""
    if data_np.ndim != 2 or data_np.shape[1] != 3:
        raise ValueError("Requires 3D data")
    pos = np.ascontiguousarray(data_np, dtype=np.float32)
    n = pos.shape[0]
    mode = HASH_MODES[hash_mode or default_hash_mode()]
    mask = np.empty(n, dtype=np.bool_)
    means = np.empty(n, dtype=np.float32) if return_means else None
    check(lib.gsx_sor_filter_host(pos.ctypes.data_as(C.c_void_p), n, int(k), float(np.float32(threshold_factor)), mode,
                                  mask.ctypes.data_as(C.c_void_p),
                                  means.ctypes.data_as(C.c_void_p) if return_means else None), "gsx_sor_filter_host")
    return (mask, means) if return_means else mask


# ------------------------------------------------------------------ cKDTree semantics (the reference's CPU path)
def ckdtree_mean_dists(xyz: torch.Tensor, k: int) -> torch.Tensor:
    """data_processor.py:160-173 on device: exact (k+1)-NN in float64, mean of neighbours 1..k -> float32."""
    _check_xyz(xyz)
    n = xyz.shape[0]
    ws = torch.empty(_abi.workspace_size("gsx_knn_exact_workspace_bytes", n), dtype=torch.uint8, device=xyz.device)
    out = torch.empty(n, dtype=torch.float32, device=xyz.device)
    check(lib.gsx_knn_exact_mean_dists(_ptr(xyz), n, int(k), _ptr(out), _ptr(ws), ws.numel(), _stream()),
          "gsx_knn_exact_mean_dists")
    return out


def ckdtree_filter(xyz: torch.Tensor, k: int = 25, threshold_factor: float = 10.5, return_means: bool = False):
    """data_processor.py:155-180 on device: the mask the reference computes (and then discards, SURVEY F5)."""
    means = ckdtree_mean_dists(xyz, k)
    mask = threshold_mask(means, mean_std(means), threshold_factor)
    return (mask, means) if return_means else mask


def ckdtree_filter_host(data_np: np.ndarray, k: int = 25, threshold_factor: float = 10.5, return_means: bool = False):
    if data_np.ndim != 2 or data_np.shape[1] != 3:
        raise ValueError("Requires 3D data")
    pos = np.ascontiguousarray(data_np, dtype=np.float32)
    n = pos.shape[0]
    mask = np.empty(n, dtype=np.bool_)
    means = np.empty(n, dtype=np.float32) if return_means else None
    check(lib.gsx_sor_ckdtree_filter_host(pos.ctypes.data_as(C.c_void_p), n, int(k), float(np.float32(threshold_factor)),
                                          mask.ctypes.data_as(C.c_void_p),
                                          means.ctypes.data_as(C.c_void_p) if return_means else None),
          "gsx_sor_ckdtree_filter_host")
    return (mask, means) if return_means else mask


def sort_pairs(keys: torch.Tensor, vals: torch.Tensor | None, begin_bit: int = 0, end_bit: int = 64):
    """In-place stable radix sort of (int64-viewed-as-uint64 keys, int32 vals) on key bits [begin,end).
    vals=None sorts bare 64-bit words (payload packed below begin_bit), the form the grid build uses."""
    n = keys.numel()
    ws = torch.empty(_abi.workspace_size("gsx_sort_pairs_workspace_bytes", n), dtype=torch.uint8, device=keys.device)
    check(lib.gsx_sort_pairs(_ptr(keys), _ptr(vals), n, begin_bit, end_bit, _ptr(ws), ws.numel(), _stream()),
          "gsx_sort_pairs")
    return keys, vals
