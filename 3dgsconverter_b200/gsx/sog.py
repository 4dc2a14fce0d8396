"""Device helpers for the SOG writer steps either side of K-Means (formats/sog.py:262-552, SURVEY §8(f) item 1).

    lexsort_zyx(xyz)                     == np.lexsort((z, y, x))                       sog.py:264
    quantize_to_codebook(vals, codebook) == the writer's sorted-codebook nearest lookup  sog.py:408-419
    codebook_1d(values, k, max_iter)     == gpu_ops.kmeans(values.reshape(-1,1), k, max_iter) + sorted(c.flatten())
                                            (sog.py:402-403, 443-444) on the 1-D Lloyd kernel
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from ._abi import lib, check, workspace_size
from .sor import _ptr, _stream, _check_xyz


def lexsort_zyx(xyz: torch.Tensor) -> torch.Tensor:
    """int32 [N]: indices that order the splats by x, then y, then z (stable), like np.lexsort((z, y, x))."""
    _check_xyz(xyz)
    n = xyz.shape[0]
    order = torch.empty(n, dtype=torch.int32, device=xyz.device)
    ws = torch.empty(workspace_size("gsx_lexsort_workspace_bytes", n), dtype=torch.uint8, device=xyz.device)
    check(lib.gsx_lexsort_zyx(_ptr(xyz), n, _ptr(order), _ptr(ws), ws.numel(), _stream()), "gsx_lexsort_zyx")
    return order


def quantize_to_codebook(vals: torch.Tensor, codebook) -> torch.Tensor:
    """uint8 [N]: nearest entry of the ascending float32 codebook (reference semantics incl. the left-neighbour rule)."""
    if not vals.is_cuda or vals.dtype != torch.float32 or not vals.is_contiguous():
        raise ValueError("vals must be a contiguous float32 CUDA tensor")
    cb = np.ascontiguousarray(codebook, dtype=np.float32)
    n = vals.numel()
    out = torch.empty(n, dtype=torch.uint8, device=vals.device)
    ws = torch.empty(max(4 * len(cb), 256), dtype=torch.uint8, device=vals.device)
    check(lib.gsx_quantize_to_codebook(_ptr(vals), n, cb.ctypes.data_as(C.POINTER(C.c_float)), len(cb), _ptr(out),
                                       _ptr(ws), ws.numel(), _stream()), "gsx_quantize_to_codebook")
    return out


def codebook_1d(values: np.ndarray, k: int = 256, max_iter: int = 20) -> np.ndarray:
    """The scalar codebook of sog.py:392-403 / 435-444: subsample <= 50 000 values with the reference's
    np.random.choice draw, Lloyd K-Means (D=1) on the GPU, return the sorted centroids (float32[k])."""
    from gsconverter.processing import gpu_ops
    fit = values
    if len(values) > 50000:
        fit = values[np.random.choice(len(values), 50000, replace=False)]
    c, _ = gpu_ops.kmeans(fit.reshape(-1, 1), k, max_iter=max_iter)
    return np.array(sorted(c.flatten()), dtype=np.float32)
