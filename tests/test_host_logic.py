"""CPU: host-side logic of the product (no GPU): cluster selection, slider maps, owner partition, bench
reference arm.  Anything numeric is checked against the oracle / the reference's formulas."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import oracle

ROOT = Path(__file__).resolve().parent.parent


def _cloud_for_voxels(vox, counts, voxel):
    pts = []
    for v, c in zip(vox, counts):
        pts.append(np.tile((np.asarray(v) + 0.5) * voxel, (c, 1)))
    return np.concatenate(pts).astype(np.float32)


@pytest.mark.parametrize("seed", range(8))
@pytest.mark.parametrize("multi", [False, True])
def test_select_clusters_matches_reference_order(gsx_lib, seed, multi):
    """6-connected components + 'largest / >= 5 % of largest' incl. ties between equally large clusters
    (decided by Python set iteration order, SURVEY A.3): gsx.density.select_clusters vs the oracle's BFS."""
    from gsx import density
    rng = np.random.default_rng(seed)
    # a few blobs of voxels, several with the same size so that ties occur
    vox = set()
    for _ in range(6):
        c = rng.integers(-6, 6, 3)
        for _ in range(int(rng.integers(1, 4))):
            c = c + rng.integers(-1, 2, 3) * (rng.random(3) < 0.5)
            vox.add(tuple(int(x) for x in c))
    vox = np.array(sorted(vox), dtype=np.int64)
    counts = np.full(len(vox), 5)
    voxel = 1.0
    pts = _cloud_for_voxels(vox, counts, voxel)
    thr_pct = 100.0 * 5 / len(pts) * 0.999          # min_points = int(n * thr/100) = 4 -> every voxel dense
    want_mask, info = oracle.density_mask(pts, voxel, thr_pct, None, multi)
    kept, n_kept, max_len = density.select_clusters(vox, multi)      # vox is already lexicographically sorted
    kept_set = set(map(tuple, kept))
    q = np.floor(pts / np.float32(voxel)).astype(np.int64)
    got_mask = np.array([tuple(v) in kept_set for v in q])
    assert n_kept == info["clusters"] and max_len == info["max_len"]
    assert np.array_equal(got_mask, want_mask)


def test_sliders_match_reference_formulas(gsx_lib):
    from gsx import density
    for s in (0.0, 0.1, 0.5, 0.9, 1.0, 1.5):
        assert density.slider(s) == oracle.density_slider(s) == (max(0.1, 2.0 - s * 1.8), 0.1 + s * 0.9)


def test_owner_partition_formula(gsx_lib):
    """Bucket-range ownership of the distributed build: floor(h*G/N) is the owner whose range
    [ceil(o*N/G), ceil((o+1)*N/G)) contains h, the ranges tile [0,N) and are balanced."""
    from gsx.dist import _owner_bounds
    rng = np.random.default_rng(0)
    for n in (1, 7, 1000, 10_000_019, 2_000_000_000):
        for g in (1, 2, 3, 4, 8):
            b = _owner_bounds(n, g)
            assert b[0] == 0 and b[-1] == n and all(b[i] <= b[i + 1] for i in range(g))
            assert max(b[i + 1] - b[i] for i in range(g)) - min(b[i + 1] - b[i] for i in range(g)) <= 1
            hs = np.unique(np.r_[rng.integers(0, n, 200), [0, n - 1], np.array(b[:-1]), np.maximum(np.array(b[1:]) - 1, 0)])
            for h in hs[hs < n]:
                o = int(h) * g // n
                assert b[o] <= h < b[o + 1], (n, g, h, o)


def test_bench_reference_arm_line():
    """`bench.py --impl reference` prints one JSON line with the contract's keys (tiny sample, CPU only)."""
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--splats-per-gpu", "20000"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Msplats/s" and line["value"] > 0
    # same `config` object as the gsx arm prints for this workload (the driver compares them)
    assert line["config"] == {"workload": "0M-splat mixed cloud per GPU (SURVEY 8d generator), SOR k=16 sigma=2.0; global "
                                          "filter over the union cloud of 20000 splats", "splats_per_gpu": 20000, "k": 16,
                              "sigma": 2.0, "cloud": "mixed"}
    assert line["cpu_baseline"]["sample_points"] == 20000
    for key in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "config", "e2e",
                "cpu_baseline"):
        assert key in line
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0


def test_bench_reference_arm_does_not_load_libgsx():
    """VERDICT r1: the reference arm's process must not map libgsx.so (the generator is loaded as a file)."""
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0', "
            "'--splats-per-gpu', '5000']; runpy.run_path(r'%s', run_name='__main__'); "
            "maps = open('/proc/self/maps').read(); assert 'libgsx' not in maps, 'libgsx.so mapped'; "
            "assert 'gsx' not in sys.modules and 'torch' not in sys.modules") % str(ROOT / "bench.py")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "d"],
                                  ["--config", "c3", "--dump-outputs", "d"]])
def test_bench_rejects_arguments_it_cannot_honour(argv, tmp_path):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), *argv], capture_output=True, text=True, timeout=120,
                         cwd=tmp_path)
    assert out.returncode == 2 and "error:" in out.stderr, out.stderr[-2000:]
    assert not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_timed_step_results(cuda, gsx_lib, tmp_path):
    """`bench.py --dump-outputs DIR`: the last timed step's keep-mask and mean distances, equal to the oracle's."""
    from gsx import synth
    n = 200_000
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                          "--no-extras", "--splats-per-gpu", str(n), "--dump-outputs", str(tmp_path / "d")],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["warmup"] == 1
    d = {p.stem: np.load(p) for p in (tmp_path / "d").glob("*.npy")}
    assert set(d) == {"sample_index", "keep_mask", "keep_count", "mean_dists", "mean_std"}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert sum(p.stat().st_size for p in (tmp_path / "d").glob("*.npy")) <= 64 << 20
    assert np.array_equal(d["sample_index"], np.arange(n))        # below the sample size: every point
    want = oracle.sor_taichi_mean_dists(synth.xyz(n, "mixed"), 16, "i32wrap")
    assert np.array_equal(d["mean_dists"].view(np.uint32), want.view(np.uint32))
    mask = oracle.threshold_mask(want, 2.0)
    assert np.array_equal(d["keep_mask"], mask.astype(np.float32)) and d["keep_count"][0] == mask.sum() == line["run"]["kept"]


def test_dropin_mirror_has_reference_surface():
    """Names and signatures of the plugin surface (SURVEY §8b) -- importable without a GPU."""
    import inspect
    from gsconverter.processing import DataProcessor, gpu_ops
    sig = lambda f: list(inspect.signature(f).parameters)  # noqa: E731
    assert sig(gpu_ops.kmeans) == ["data", "k", "max_iter", "tolerance", "use_gpu", "verbose"]
    assert sig(gpu_ops.filter_sor_gpu) == ["data_np", "k", "threshold_factor", "verbose"]
    assert sig(DataProcessor.apply_density_filter) == ["self", "voxel_size", "threshold_percentage", "sensitivity",
                                                       "keep_multicluster"]
    assert sig(DataProcessor.remove_flyers) == ["self", "k", "threshold_factor", "chunk_size", "intensity"]
    assert sig(DataProcessor.crop_by_bbox) == ["self", "min_x", "min_y", "min_z", "max_x", "max_y", "max_z"]
    assert sig(DataProcessor.apply_alpha_filter) == ["self", "min_opacity_u8"]
    assert isinstance(gpu_ops.HAS_TAICHI, bool)
    d = inspect.signature(gpu_ops.kmeans).parameters
    assert d["max_iter"].default == 10 and d["tolerance"].default == 1e-4 and d["use_gpu"].default is True
    d = inspect.signature(DataProcessor.remove_flyers).parameters
    assert d["k"].default == 25 and d["threshold_factor"].default == 10.5 and d["chunk_size"].default == 50000
    # k >= N passthrough and the explicit CPU request work without a GPU (gpu_ops.py:30-38)
    X = np.arange(12, dtype=np.float32).reshape(4, 3)
    C, L = gpu_ops.kmeans(X, 9)
    assert np.array_equal(C, X) and np.array_equal(L, np.arange(4, dtype=np.int32))
    C, L = gpu_ops.kmeans(np.random.default_rng(0).random((200, 3)).astype(np.float32), 4, use_gpu=False)
    assert C.shape == (4, 3) and L.shape == (200,)


def test_build_ops_glue_reaches_the_library(gsx_lib, monkeypatch):
    """CPU: the ctypes glue of gsx.dist._GsxBuildOps is well-formed -- without a GPU every stage gets as far as the
    CUDA launch inside libgsx and fails there with GsxError (not with a Python-level error)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("meant for the CPU box")
    import ctypes
    from gsx import GsxError, sor
    from gsx.dist import _GsxBuildOps
    monkeypatch.setattr(sor, "_stream", lambda: ctypes.c_void_p(0))   # torch has no CUDA stream on this box
    ops = _GsxBuildOps()
    mm = np.array([0, 0, 0, 1, 2, 3], np.float32)
    cell = ops.cell_size(mm, 1000)
    assert cell == pytest.approx(float((np.float32(6.0) / 1000 * 32) ** (1.0 / 3.0)), rel=1e-6)
    xyz = torch.rand((1000, 3))
    bmin = mm[:3].copy()
    with pytest.raises(GsxError):
        ops.local_run(xyz, 0, 1000, 2, bmin, cell)
    with pytest.raises(GsxError):
        ops.merge_into(torch.rand((1000, 4)), 1000, bmin, cell, torch.empty((1000, 4)))
    ws, spos = ops.new_grid_storage(1000, torch.device("cpu"))
    assert spos.shape == (1000, 4) and spos.data_ptr() >= ws.data_ptr()
    with pytest.raises(GsxError):
        ops.finish(ws, spos, 1000, bmin, cell)


def _load_bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bench_mod", ROOT / "bench.py")
    mod = importlib.util.module_from_spec(spec)
    old = sys.argv
    sys.argv = ["bench.py"]
    try:
        spec.loader.exec_module(mod)
    finally:
        sys.argv = old
    return mod


def test_bench_clock_sampler_reports_clocks_under_load(tmp_path, monkeypatch):
    """The bench contract needs `clocks` sampled DURING the timed region.  With a fake nvidia-smi whose first row takes
    150 ms: (a) rows inside the window are used; (b) a timed region shorter than the sampler's start-up makes the caller
    run extra busy steps until a row arrives -- never an idle-clock row from after the run."""
    import os
    import time
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/bash\nsleep 0.15\nwhile true; do echo '0, 1965, 1965, 400.0, 0x0, Not Active, Not Active, "
                    "Not Active, Active'; sleep 0.025; done\n")
    fake.chmod(0o755)
    monkeypatch.setenv("PATH", f"{tmp_path}:{os.environ['PATH']}")
    bench = _load_bench()
    c = bench.ClockSampler(0)
    c.start()
    time.sleep(0.6)              # (generous margins: the CPU suite may share the machine)
    c.window_begin()
    time.sleep(0.4)
    c.window_end()
    r = c.stop()
    assert r["window"] == "timed region" and r["samples"] >= 1 and r["sm_mhz"] == 1965.0
    assert r["reasons"] == ["sw_power_cap"]
    c = bench.ClockSampler(0)
    c.start()
    c.window_begin()
    time.sleep(0.03)
    c.window_end()
    busy = []
    r = c.stop(keep_busy=lambda: (busy.append(1), time.sleep(0.01)))
    assert r is not None and len(busy) >= 1 and r["window"].startswith("extra untimed steps")
    import torch
    r = bench.finish_clocks(bench.ClockSampler(0), 1, 0, torch.device("cpu"), lambda: None)   # never started: no clocks
    assert r is None


def _clock_rank(rank, world, fakedir, port, q):
    import importlib.util
    import time
    import torch
    import torch.distributed as dist
    os.environ["PATH"] = f"{fakedir}:{os.environ['PATH']}"
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    spec = importlib.util.spec_from_file_location("_bench_mod", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    sys.argv = ["bench.py"]
    spec.loader.exec_module(bench)
    c = bench.ClockSampler(0)
    if rank == 0:
        c.start()
    c.window_begin()
    time.sleep(0.02)                      # a timed region shorter than the sampler's start-up
    c.window_end()
    steps = [0]

    def busy():                           # the extra step contains a collective, like the sharded filter
        t = torch.ones(1)
        dist.all_reduce(t)
        steps[0] += 1
        time.sleep(0.01)
    r = bench.finish_clocks(c, world, rank, torch.device("cpu"), busy)
    q.put((rank, steps[0], r))
    dist.destroy_process_group()


def test_bench_finish_clocks_is_collective_at_n_gt_1(tmp_path):
    """N > 1: while rank 0's sampler still needs a row under load, EVERY rank must run the same number of extra
    steps (they contain collectives) -- the decision is broadcast from rank 0; no rank may hang or diverge."""
    import torch.multiprocessing as mp
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/bash\nsleep 0.2\nwhile true; do echo '0, 1965, 1965, 400.0, 0x0, Not Active, Not Active, "
                    "Not Active, Not Active'; sleep 0.025; done\n")
    fake.chmod(0o755)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 400)
    procs = [ctx.Process(target=_clock_rank, args=(r, 2, str(tmp_path), port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    (r0, n0, clk0), (r1, n1, clk1) = res
    assert n0 == n1 >= 1                                   # same number of collective busy steps on both ranks
    assert clk1 is None and clk0 is not None and clk0["sm_mhz"] == 1965.0 and clk0["window"].startswith("extra untimed")
