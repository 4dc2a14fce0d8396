"""Morton ordering and chunk bounds as shared primitives (SURVEY 8(f) item 3): host plumbing over gsx_morton_order /
gsx_chunk_minmax (formats/compressed_ply.py:252-297, :206-246; formats/ksplat.py:426-441)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from ._abi import lib, check, workspace_size
from .sor import _ptr, _stream, _check_xyz


def morton_order(xyz: torch.Tensor, run_limit: int = 256, return_levels: bool = False):
    """order int32[N]: the recursive 3 x 10-bit Morton order of compressed_ply.py:252-297 (stable inside equal codes)."""
    _check_xyz(xyz)
    n = xyz.shape[0]
    order = torch.empty(n, dtype=torch.int32, device=xyz.device)
    ws = torch.empty(workspace_size("gsx_morton_workspace_bytes", n), dtype=torch.uint8, device=xyz.device)
    lv = C.c_int32(0)
    check(lib.gsx_morton_order(_ptr(xyz), n, _ptr(order), int(run_limit), C.byref(lv), _ptr(ws), ws.numel(), _stream()),
          "gsx_morton_order")
    return (order, int(lv.value)) if return_levels else order


def chunk_minmax(rows: torch.Tensor, cols, order: torch.Tensor | None = None, chunk: int = 256,
                 clip: tuple[float, float] | None = None):
    """(lo, hi) float32 [ceil(N/chunk), len(cols)]: per-chunk min / max of the given columns of the row-major matrix
    `rows` [N,F], rows taken in `order` (None = as stored), values optionally clipped first."""
    if rows.dim() != 2 or rows.dtype != torch.float32 or not rows.is_contiguous() or not rows.is_cuda:
        raise ValueError("rows must be a contiguous float32 CUDA matrix [N,F]")
    n, F = rows.shape
    cols = [int(c) for c in cols]
    nchunk = (n + chunk - 1) // chunk
    lo = torch.empty((nchunk, len(cols)), dtype=torch.float32, device=rows.device)
    hi = torch.empty_like(lo)
    ws = torch.empty(256, dtype=torch.uint8, device=rows.device)
    cl, ch = clip if clip is not None else (float("-inf"), float("inf"))
    carr = (C.c_int32 * len(cols))(*cols)
    check(lib.gsx_chunk_minmax(_ptr(rows), n, F, _ptr(order), int(chunk), carr, len(cols), float(cl), float(ch), _ptr(lo),
                               _ptr(hi), _ptr(ws), ws.numel(), _stream()), "gsx_chunk_minmax")
    return lo, hi
