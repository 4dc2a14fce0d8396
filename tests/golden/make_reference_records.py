"""Record what the reference 3dgsconverter computes for the two checks that used to import it at test time.

    python tests/golden/make_reference_records.py <path of a 3dgsconverter source tree>

Writes (the tests read only these files; the reference is never needed to run the suite):
  * g9_reference_small_run.npz -- the reference's own `gsconverter/processing/gpu_ops.py`, loaded unmodified under
    the serial `taichi` stand-in (ti_serial.py): `filter_sor_gpu` on a 400-point cloud (k=12, sigma=1.5) and
    `_kmeans_taichi` on 300 x 5 (K=7, 3 iterations, NumPy seed 11).  Read by tests/test_reference_kernels_pin.py.
  * g10_reference_dropin.npz -- on the 100 k `mixed` record array (gsx.synth.structured): SHA-256 digests and row
    counts of the unpatched reference DataProcessor's crop_by_bbox -> apply_alpha_filter -> apply_density_filter
    outputs, and the sequence of `gpu_ops.kmeans` calls the reference's SogFormat.write makes on the survivors of
    SOR k=16 / sigma=2 (shape, K, max_iter, row-range view of a larger array or not, global RNG used since the
    previous call).  Read by tests/test_dropin_reference_cpu.py.
The script asserts the oracle equal to every reference output it records.
"""
import hashlib
import sys
import tempfile
import types
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "3dgsconverter_b200"), str(HERE)]

import oracle  # noqa: E402
from gsx import synth  # noqa: E402


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def chunk_view(data):
    """(start row, rows of the base array) when `data` is a row range of a larger 2-D array, else (-1, -1)."""
    base = data.base
    if not isinstance(base, np.ndarray) or base.ndim != 2 or data.ndim != 2 or base.shape[1] != data.shape[1]:
        return -1, -1
    off = data.ctypes.data - base.ctypes.data
    return off // (base.shape[1] * base.itemsize), base.shape[0]


def dropin_records(ref_root: str) -> dict:
    sys.path.insert(0, ref_root)
    ply = types.ModuleType("plyfile")
    ply.PlyData = ply.PlyElement = object
    sys.modules["plyfile"] = ply
    import gsconverter
    assert gsconverter.__file__.startswith(ref_root), gsconverter.__file__
    from gsconverter.processing.data_processor import DataProcessor
    from gsconverter.processing import gpu_ops
    from gsconverter.formats.sog import SogFormat

    data = synth.structured(100_000, "mixed")
    dp = DataProcessor(data.copy())
    r_bbox = dp.crop_by_bbox(-11, -11, -11, 11, 11, 11).copy()
    r_alpha = dp.apply_alpha_filter(5).copy()
    r_dens = dp.apply_density_filter(1.0, 0.32, sensitivity=0.5, keep_multicluster=True).copy()
    xyz = np.column_stack((r_dens["x"], r_dens["y"], r_dens["z"]))
    survivors = r_dens[oracle.sor_taichi_mask(xyz, 16, 2.0, "i32wrap")]

    calls, last = [], [np.random.get_state()]

    def kmeans(d, k, max_iter=10, tolerance=1e-4, use_gpu=True, verbose=False):
        """The reference's call contract (passthrough for k >= n, init drawn from the global NumPy RNG), oracle
        arithmetic; records the call."""
        st = np.random.get_state()
        moved = not (st[0] == last[0][0] and np.array_equal(st[1], last[0][1]) and st[2:] == last[0][2:])
        start, base_rows = chunk_view(d)
        calls.append((d.shape[0], d.shape[1], int(k), int(max_iter), start, base_rows, int(moved)))
        n = d.shape[0]
        if k >= n:
            res = d.copy(), np.arange(n, dtype=np.int32)
        else:
            x = d.astype(np.float32)
            C, L, _ = oracle.kmeans_lloyd(x, int(k), int(max_iter), init=x[np.random.choice(n, k, replace=False)])
            res = C, L
        last[0] = np.random.get_state()
        return res

    gpu_ops.kmeans = kmeans
    np.random.seed(4242)
    last[0] = np.random.get_state()
    with tempfile.TemporaryDirectory() as tmp:
        SogFormat().write(survivors.copy(), str(Path(tmp) / "out.sog"), compression_level=5)
    return {"bbox_sha": sha(r_bbox), "alpha_sha": sha(r_alpha), "density_sha": sha(r_dens),
            "counts": np.array([len(r_bbox), len(r_alpha), len(r_dens), len(survivors)], np.int64),
            "sog_kmeans_calls": np.array(calls, np.int64)}


def small_run_records(ref_root: str) -> dict:
    import ti_serial
    ref = ti_serial.import_reference_gpu_ops(ref_root)
    src = ref.sor_compute_mean_dists.__ti_serial_source__
    for fragment in ("h = (nx * p1 ^ ny * p2 ^ nz * p3) % hash_size", "while ins_pos >", "d = ti.sqrt(d2)",
                     "mean_dists[i] = sum_d / _ti_f32cast(valid_k)"):
        assert fragment in src, fragment
    assert "centroids[l, dim] += data[i, dim]" in ref.k_means_update.__ti_serial_source__
    rng = np.random.default_rng(3)
    xyz = np.concatenate([rng.normal(0, 0.05, (250, 3)), rng.uniform(-2, 2, (150, 3))]).astype(np.float32)
    mask = ref.filter_sor_gpu(xyz, k=12, threshold_factor=1.5)
    assert np.array_equal(mask, oracle.sor_taichi_mask(xyz, 12, 1.5, "i32wrap"))
    X = rng.normal(size=(300, 5)).astype(np.float32)
    np.random.seed(11)
    C, L = ref._kmeans_taichi(X, 7, max_iter=3)
    np.random.seed(11)
    Co, Lo, _ = oracle.kmeans_lloyd(X, 7, 3, init=X[np.random.choice(300, 7, replace=False)])
    assert np.array_equal(L, Lo) and np.array_equal(C.view(np.uint32), Co.view(np.uint32))
    return {"sor_mask": mask, "km_centroids": C, "km_labels": L}


def main():
    ref_root = str(Path(sys.argv[1]).resolve())
    # the package import first: the stand-in `taichi` installed by small_run_records would change what it imports
    np.savez_compressed(HERE / "g10_reference_dropin.npz", **dropin_records(ref_root))
    np.savez_compressed(HERE / "g9_reference_small_run.npz", **small_run_records(ref_root))
    print("wrote g9_reference_small_run.npz, g10_reference_dropin.npz")


if __name__ == "__main__":
    main()
