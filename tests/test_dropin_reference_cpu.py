"""CPU: gsx.dropin.patch() on a `gsconverter` package, checked against what the reference 3dgsconverter computes on
the same records (tests/golden/g10_reference_dropin.npz, recorded by tests/golden/make_reference_records.py).
The patch is applied to this repository's own `gsconverter` package, and the device layer (gsx.pipeline.FilterChain,
the gsx.kmeans host entry points) is replaced by oracle-backed stand-ins so that the test needs no GPU; everything
between the package's call sites and that layer is the shipped code: the patched gsconverter.processing.
{DataProcessor, gpu_ops}, the converter.py:194-236 filter chain, and the batch-ahead of the SOG shN chunk loop with its
RNG transparency.  Checks:
  * bbox / alpha / density outputs of the patched chain == the UNPATCHED reference's outputs (SHA-256 of the records);
  * SOR through the patch == the oracle's Taichi-semantics mask (the reference's own CPU path discards its mask, F5);
  * the reference SogFormat.write's sequence of gpu_ops.kmeans calls, replayed through the patched gpu_ops: the
    shN chunk loop reaches the backend as ONE batched launch, the call shapes follow sog.py:392-552, and every result
    and the global RNG stream are bit-identical with batch-ahead on and off (same seed).
"""
import json
import os
import subprocess
import sys
import textwrap
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
GOLD = ROOT / "tests" / "golden" / "g10_reference_dropin.npz"

DRIVER = textwrap.dedent(r'''
    import hashlib, json, sys
    import numpy as np
    ROOT, GOLD = sys.argv[1], sys.argv[2]
    sys.path[:0] = [ROOT, ROOT + "/3dgsconverter_b200"]
    import gsconverter                                                 # this repository's package
    assert gsconverter.__file__.startswith(ROOT + "/3dgsconverter_b200/"), gsconverter.__file__
    from gsconverter.processing.data_processor import DataProcessor as UnpatchedDP
    import oracle
    import gsx, gsx.pipeline, gsx.kmeans, gsx.dropin
    from gsx import synth
    ref = np.load(GOLD)
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()

    # ---------------- oracle-backed stand-ins for the device layer (no GPU needed)
    calls = {"kmeans_host": [], "kmeans_host_batched": []}

    class OracleChain:
        def __init__(self, xyz, opacity=None, device=None):
            self.xyz = np.ascontiguousarray(xyz, dtype=np.float32)
            self.opacity = None if opacity is None else np.ascontiguousarray(opacity, dtype=np.float32)
            self.idx, self.n0 = None, len(self.xyz)
        @property
        def count(self): return len(self.xyz)
        def _apply(self, m):
            cur = np.arange(self.n0) if self.idx is None else self.idx
            self.idx = cur[m]; self.xyz = self.xyz[m]
            if self.opacity is not None: self.opacity = self.opacity[m]
            return len(self.xyz)
        def clear(self): self._apply(np.zeros(self.count, bool))
        def crop_by_bbox(self, *b):
            return self._apply(oracle.bbox_mask(self.xyz[:, 0], self.xyz[:, 1], self.xyz[:, 2], *b))
        def alpha(self, a): return self._apply(oracle.alpha_mask(self.opacity, a))
        def density(self, voxel_size=1.0, threshold_percentage=0.32, sensitivity=None, keep_multicluster=False):
            m, info = oracle.density_mask(self.xyz, voxel_size, threshold_percentage, sensitivity, keep_multicluster)
            info = dict(info, voxels=-1)
            if info["dense"] == 0 or info["clusters"] == 0: self.clear()
            else: self._apply(m)
            return self.count, info
        def sor(self, k=25, threshold_factor=1.0, hash_mode=None, semantics="taichi"):
            return self._apply(oracle.sor_taichi_mask(self.xyz, k, threshold_factor, hash_mode or "i32wrap"))
        def indices(self): return np.arange(self.n0) if self.idx is None else self.idx
        def rebase(self): self.idx, self.n0 = None, self.count

    def kmeans_host(data, K, max_iter, init, assign=None):
        calls["kmeans_host"].append((tuple(data.shape), int(K), int(max_iter)))
        C, L, _ = oracle.kmeans_lloyd(np.asarray(data), K, max_iter, init=np.asarray(init))
        return C, L

    def kmeans_host_batched(base, row_off, K, max_iter, init, assign=None):
        calls["kmeans_host_batched"].append((tuple(base.shape), len(row_off) - 1, int(K), int(max_iter)))
        Cs, Ls = [], []
        for p in range(len(row_off) - 1):
            C, L, _ = oracle.kmeans_lloyd(np.asarray(base[row_off[p]:row_off[p + 1]]), K, max_iter, init=np.asarray(init[p]))
            Cs.append(C); Ls.append(L)
        return np.stack(Cs), np.concatenate(Ls)

    gsx.pipeline.FilterChain = OracleChain
    gsx.kmeans.kmeans_host = kmeans_host
    gsx.kmeans.kmeans_host_batched = kmeans_host_batched
    gsx.kmeans.device_free_bytes = lambda: 1 << 40
    gsx.backend_available = lambda: True
    gsx.dropin.backend_available = gsx.backend_available if hasattr(gsx.dropin, "backend_available") else None

    data = synth.structured(100_000, "mixed")
    out = {}

    # ---------------- 1. patch and run the converter.py:194-236 chain through gsconverter.processing
    assert gsx.dropin.patch(defer=True) is True
    import gsconverter.processing as proc
    from gsconverter.processing import gpu_ops
    assert gpu_ops._GSX_PATCHED and gpu_ops.HAS_TAICHI is True
    P = proc.DataProcessor
    assert P is not UnpatchedDP and P.__module__.endswith("_gsx_data_processor")
    dp = P(data.copy())
    dp.crop_by_bbox(-11, -11, -11, 11, 11, 11); p_bbox = dp.data.copy()
    dp.apply_alpha_filter(5); p_alpha = dp.data.copy()
    dp.apply_density_filter(1.0, 0.32, sensitivity=0.5, keep_multicluster=True); p_dens = dp.data.copy()
    dp.remove_flyers(16, 2.0); p_sor = dp.data.copy()
    # ---------------- 2. against the UNPATCHED reference on the same records (its own NumPy paths)
    out["bbox_equal"] = sha(p_bbox) == str(ref["bbox_sha"])
    out["alpha_equal"] = sha(p_alpha) == str(ref["alpha_sha"])
    out["density_equal"] = sha(p_dens) == str(ref["density_sha"])
    xyz_d = np.column_stack((p_dens["x"], p_dens["y"], p_dens["z"]))
    want = oracle.sor_taichi_mask(xyz_d, 16, 2.0, "i32wrap")
    out["sor_equal_oracle"] = bool(np.array_equal(p_dens[want], p_sor))
    out["counts"] = [len(p_bbox), len(p_alpha), len(p_dens), len(p_sor)]
    out["ref_counts"] = ref["counts"].tolist()

    # ---------------- 3. the reference SogFormat.write's gpu_ops.kmeans calls through the patch: call shapes, one
    # batched launch, RNG transparency.  The shN chunks are row ranges of one block of the survivors' SH rows, as in
    # the writer; the other inputs come from a generator of their own, outside the global RNG.
    block = np.ascontiguousarray(np.column_stack([p_sor[f"f_rest_{i}"] for i in range(45)]), dtype=np.float32)
    def write(batch_ahead):
        g = gpu_ops._gsx_module
        g.BATCH_AHEAD = batch_ahead
        g._BATCH = None
        for k in g.batch_stats: g.batch_stats[k] = 0
        calls["kmeans_host"].clear(); calls["kmeans_host_batched"].clear()
        np.random.seed(4242)
        digests = []
        for i, (rows, cols, k, max_iter, start, base_rows, rng_moved) in enumerate(ref["sog_kmeans_calls"].tolist()):
            if rng_moved:
                np.random.random()            # the writer drew from the global RNG since the previous call
            if start >= 0:
                assert base_rows == len(block) and cols == 45, (base_rows, len(block))
                d = block[start:start + rows]
            else:
                d = np.random.default_rng(i).standard_normal((rows, cols), dtype=np.float32)
            C, L = gpu_ops.kmeans(d, k, max_iter=max_iter)
            digests.append((sha(C), sha(L)))
        return digests, dict(g.batch_stats), list(calls["kmeans_host"]), list(calls["kmeans_host_batched"]), np.random.get_state()[1].tolist()
    d_on, st_on, single_on, batched_on, rng_on = write(True)
    d_off, st_off, single_off, batched_off, rng_off = write(False)
    n_s = len(p_sor)
    num_chunks = max(1, min(64, n_s // 1024)); chunk = int(np.ceil(n_s / num_chunks))
    out["sog"] = {"results_equal_batch_on_off": d_on == d_off,
                  "stats_on": st_on, "stats_off": st_off, "batched_calls_on": batched_on, "single_calls_on": single_on[:4],
                  "single_calls_off_shN": [c for c in single_off if c[0][1] == 45][:2], "n_single_off_shN": len([c for c in single_off if c[0][1] == 45]),
                  "num_chunks": num_chunks, "chunk": chunk, "n": n_s,
                  "rng_after_equal": rng_on == rng_off}
    print("RESULT " + json.dumps(out))
''')


def test_patch_against_the_real_reference(tmp_path, gsx_lib):
    drv = tmp_path / "driver.py"
    drv.write_text(DRIVER)
    env = dict(os.environ, OMP_NUM_THREADS="8", PYTHONWARNINGS="ignore")
    r = subprocess.run([sys.executable, str(drv), str(ROOT), str(GOLD)], capture_output=True, text=True,
                       timeout=1500, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1]
    out = json.loads(line[7:])
    assert out["bbox_equal"] and out["alpha_equal"] and out["density_equal"], out
    assert out["sor_equal_oracle"] and out["counts"] == out["ref_counts"], out
    sog = out["sog"]
    # sog.py:392-445: two 1-D fits on <= 50 000 scalars, K=256, max_iter=20 -- single calls in both modes
    assert sog["single_calls_on"][:2] == [[[50000, 1], 256, 20], [[50000, 1], 256, 20]], sog
    # sog.py:513-552: the shN loop = num_chunks calls of (chunk x 45, k_per_chunk, 10) ...
    assert sog["n_single_off_shN"] == sog["num_chunks"] and sog["single_calls_off_shN"][0][0] == [sog["chunk"], 45], sog
    # ... which the patch turns into ONE batched launch over the whole SH block (uploaded once)
    assert sog["stats_on"]["batched_launches"] == 1 and sog["stats_on"]["served_from_batch"] == sog["num_chunks"], sog
    assert len(sog["batched_calls_on"]) == 1 and sog["batched_calls_on"][0][1] == sog["num_chunks"], sog
    assert sog["batched_calls_on"][0][0] == [sog["n"], 45], sog
    # identical results and identical global RNG stream either way
    assert sog["results_equal_batch_on_off"] and sog["rng_after_equal"], sog
