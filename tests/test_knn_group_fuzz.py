"""CPU: the group path of the query kernel (GSX_KNN_GROUP; tests/knn_group_emulator.py) equals the brute-force
oracle bit for bit -- the box-to-box bound against the largest seed tau of a batch never drops a chunk that one of its
queries needs.  Small fan-outs and small batches put many batches on the group path on clouds of a few hundred points;
a 2-entry list makes most of them overflow and fall back to the per-query path."""
import numpy as np
import pytest

import oracle
from knn_group_emulator import emulate_group
from test_knn_algorithm_fuzz import _clouds


def _group_clouds():
    rng = np.random.default_rng(7)
    yield from _clouds()
    yield "lattice_dense", np.stack(np.meshgrid(*[np.arange(9)] * 3), -1).reshape(-1, 3) * 0.125   # ties at tau
    yield "duplicate_blob", np.repeat(rng.normal(0, 0.01, (120, 3)), 4, axis=0)
    # a dense blob cut by cell faces: batches that straddle a cell boundary take the per-query path
    yield "blob_on_cell_faces", np.r_[rng.normal(0, 0.02, (600, 3)), rng.uniform(-1, 1, (100, 3))]


@pytest.mark.parametrize("mode", ["i32wrap", "i64"])
@pytest.mark.parametrize("k", [1, 7, 16, 27])
def test_group_path_is_exact(mode, k):
    ran = 0
    for name, pts in _group_clouds():
        xyz = pts.astype(np.float32)
        want = oracle.sor_taichi_mean_dists(xyz, k, mode)
        chunk = 4 if k < 4 else 32   # a seed list is full only if the chunk holds K other points
        for batch, glist, flat in ((chunk, 64, 0), (chunk // 2 + 1, 2, 1000)):
            got, st = emulate_group(xyz, k, mode, chunk=chunk, fan=4, small_bucket=6, flat_supers=flat, batch=batch,
                              group_list=glist)
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (name, mode, k, batch, glist, flat)
            ran += st["group_queries"]
    assert ran > 0


def test_group_path_runs_and_overflows():
    rng = np.random.default_rng(3)
    xyz = np.r_[rng.normal(0, 0.01, (800, 3)), rng.uniform(-2, 2, (200, 3))].astype(np.float32)
    want = oracle.sor_taichi_mean_dists(xyz, 8, "i64")
    big, st_big = emulate_group(xyz, 8, "i64", chunk=16, fan=4, small_bucket=6, batch=8, group_list=64)
    tiny, st_tiny = emulate_group(xyz, 8, "i64", chunk=16, fan=4, small_bucket=6, batch=8, group_list=2)
    assert st_big["group_queries"] > 0.3 * len(xyz), st_big
    assert st_tiny["group_fallbacks"] > 0 and st_tiny["group_queries"] < st_big["group_queries"], st_tiny
    assert np.array_equal(big.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(tiny.view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("mode", ["i32wrap", "i64"])
def test_group_path_with_colliding_cells(mode):
    """Two-point small buckets and a 1-bit Morton order: more long buckets, shared by several cells (the hash is
    modulo the point count), where the centre probe's bucket need not hold the whole batch."""
    rng = np.random.default_rng(11)
    xyz = np.r_[rng.normal(0, 0.05, (500, 3)), rng.uniform(-1, 1, (200, 3))].astype(np.float32)
    for k in (1, 16):
        want = oracle.sor_taichi_mean_dists(xyz, k, mode)
        got, st = emulate_group(xyz, k, mode, chunk=4, fan=4, small_bucket=2, morton_bits=1, batch=4, group_list=64)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (mode, k)
