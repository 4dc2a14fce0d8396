"""Device-resident filter chain: the columns the filters read (xyz, opacity) and the surviving ORIGINAL
row indices live in HBM across bbox -> alpha -> density -> SOR (converter.py:194-236 order); the 248-byte
records stay on the host and are gathered once with `indices()`.

Every step computes its keep-mask with the same kernels as the one-shot entry points (bit-identical
masks) and compacts the working set with gsx_compact_points (stable, like NumPy boolean indexing).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import density as _density, masks as _masks, sor as _sor
from ._abi import lib, check, workspace_size
from .sor import _ptr, _stream


def compact(mask: torch.Tensor, xyz: torch.Tensor, opacity: torch.Tensor | None, idx: torch.Tensor | None):
    """Stable compaction of (xyz, opacity, idx) by a bool/uint8 mask.  Returns (xyz, opacity, idx, count)."""
    n = xyz.shape[0]
    dev = xyz.device
    m8 = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
    ws = torch.empty(workspace_size("gsx_compact_workspace_bytes", n), dtype=torch.uint8, device=dev)
    xyz_o = torch.empty_like(xyz)
    op_o = torch.empty_like(opacity) if opacity is not None else None
    idx_o = torch.empty(n, dtype=torch.int32, device=dev)
    cnt = C.c_int64(0)
    check(lib.gsx_compact_points(_ptr(m8), n, _ptr(xyz), _ptr(opacity), _ptr(idx), _ptr(xyz_o), _ptr(op_o),
                                 _ptr(idx_o), C.byref(cnt), _ptr(ws), ws.numel(), _stream()), "gsx_compact_points")
    m = cnt.value
    return xyz_o[:m], (op_o[:m] if op_o is not None else None), idx_o[:m], m


class FilterChain:
    def __init__(self, xyz, opacity=None, device="cuda"):
        from .hostcopy import to_device
        to_dev = lambda a: (a.to(device) if isinstance(a, torch.Tensor) else  # noqa: E731
                            to_device(np.ascontiguousarray(a, dtype=np.float32), device))
        self.xyz = to_dev(xyz).contiguous()
        self.opacity = to_dev(opacity).contiguous() if opacity is not None else None
        self.idx = None            # None == identity (nothing removed yet)
        self.n0 = self.xyz.shape[0]

    @property
    def count(self) -> int:
        return self.xyz.shape[0]

    def _apply(self, mask: torch.Tensor) -> int:
        if self.count == 0:
            return 0
        self.xyz, self.opacity, self.idx, m = compact(mask, self.xyz, self.opacity, self.idx)
        return m

    def clear(self):
        self.xyz = self.xyz[:0]
        self.opacity = self.opacity[:0] if self.opacity is not None else None
        self.idx = torch.empty(0, dtype=torch.int32, device=self.xyz.device)

    # -- the four filters (same arithmetic as gsx.masks / gsx.density / gsx.sor) ---------------------
    def crop_by_bbox(self, min_x, min_y, min_z, max_x, max_y, max_z) -> int:
        if self.count:
            self._apply(_masks.bbox_mask(self.xyz, min_x, min_y, min_z, max_x, max_y, max_z))
        return self.count

    def alpha(self, min_opacity_u8) -> int:
        if self.opacity is None:
            raise ValueError("no opacity column")
        if self.count:
            self._apply(_masks.alpha_mask(self.opacity, min_opacity_u8))
        return self.count

    def density(self, voxel_size=1.0, threshold_percentage=0.32, sensitivity=None, keep_multicluster=False):
        if self.count == 0:
            return 0, dict(clusters=0, max_len=0, dense=0, voxels=0)
        mask, info = _density.density_filter(self.xyz, voxel_size, threshold_percentage, sensitivity,
                                             keep_multicluster)
        if info["dense"] == 0 or info["clusters"] == 0:
            self.clear()
        else:
            self._apply(mask)
        return self.count, info

    def sor(self, k=25, threshold_factor=1.0, hash_mode=None, semantics="taichi") -> int:
        if self.count:
            if semantics == "ckdtree":
                mask = _sor.ckdtree_filter(self.xyz, k, threshold_factor)
            else:
                mask = _sor.sor_filter(self.xyz, k, threshold_factor, hash_mode=hash_mode)
            self._apply(mask)
        return self.count

    def indices(self) -> np.ndarray:
        """Surviving original row indices (ascending), on the host."""
        if self.idx is None:
            return np.arange(self.n0, dtype=np.int64)
        from .hostcopy import to_host
        return to_host(self.idx).astype(np.int64)

    def rebase(self):
        """Declare the current survivors to be rows 0..count-1 of a freshly compacted host array."""
        self.idx = None
        self.n0 = self.count
