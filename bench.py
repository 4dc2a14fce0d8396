#!/usr/bin/env python
"""bench.py -- headline benchmark of the gsx hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl gsx|reference] [--config c2|c3|c4|c5] [--splats-per-gpu N]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Default (`--config c2`, the driver's contract line).  Metric: Msplats/s of Statistical Outlier Removal, k=16,
sigma=2.0, on BASELINE configs[1]: a 10 M-splat synthetic `mixed` cloud per GPU (SURVEY 8d generator), Taichi
semantics with the faithful int32-wrapping probe hash (SURVEY F8).  A step = one full pass of the filter (min/max ->
hash grid build -> K-nearest mean distances -> NumPy-order mean/std -> keep-mask) over the batch, inputs resident in
HBM.  N>1: weak scaling -- every rank holds a 10 M slab, the filter is the GLOBAL one over the union cloud
(gsx/dist.py), and the line carries `parity`: the N-rank mask digest against the single-GPU filter on the union cloud.

Other configs (one JSON line each, same contract keys):
    c3  50 M-splat SOG level-5 K-Means schedule (64 chunks x 781 250 x 45, K=256, 10 Lloyd iterations), 1 GPU
    c4  200 M splats on 4 GPUs (50 M per rank): SOR + density --keep_multicluster, N-GPU == 1-GPU digests
    c5  1 B splats on 8 GPUs (125 M per rank): bbox -> alpha -> density -> SOR -> K-Means, device-generated cloud

Extra objects of the c2 line: roofline (dominant kernel k_sor_knn), cpu_baseline, e2e (through
gsconverter.processing.gpu_ops.filter_sor_gpu with host buffers, pinned and pageable), clocks, like_for_like (the
cKDTree-semantics GPU path against the reference's cKDTree CPU path), pipeline, kmeans (secondary metric).

`--impl reference`: the reference's own CPU implementation of the path (SciPy cKDTree, data_processor.py:155-180 --
a port: the reference is pure Python and is not present on the GPU box) on the SAME config; no gsx import, no
libgsx.so in that process.
"""
from __future__ import annotations

import argparse
import hashlib
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
PKG = ROOT / "3dgsconverter_b200"

import numpy as np  # noqa: E402

K_SOR = 16
SIGMA = 2.0
L2_FLUSH_BYTES = 256 << 20
REFERENCE_BUDGET_S = 360.0   # the reference arm sizes its per-step sample so that the whole run fits this


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gsx", choices=["gsx", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--splats-per-gpu", "--points", dest="n", type=int, default=None,
                    help="splats per GPU (default: the config's); not `--n`: torchrun would swallow it")
    ap.add_argument("--kind", default="mixed", choices=["mixed", "uniform", "clustered"])
    ap.add_argument("--hash", default="i32wrap", choices=["i32wrap", "i64"])
    ap.add_argument("--cpu-sample", type=int, default=1_000_000, help="points of the in-line CPU-baseline sample")
    ap.add_argument("--no-extras", action="store_true", help="skip cpu_baseline / e2e / kmeans / parity extras")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy "
                         "(--config c2, --impl gsx; see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and (a.impl != "gsx" or a.config != "c2"):
        ap.error("--dump-outputs is defined for --impl gsx --config c2")
    if a.n is None:
        a.n = {"c2": 10_000_000, "c3": 50_000_000, "c4": 50_000_000, "c5": 125_000_000}[a.config]
    return a


def load_synth():
    """The SURVEY 8(d) generator (3dgsconverter_b200/gsx/synth.py, pure NumPy) loaded as a FILE, so that the
    reference arm never imports the gsx package (which dlopens libgsx.so)."""
    spec = importlib.util.spec_from_file_location("gsx_synth_standalone", PKG / "gsx" / "synth.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def c2_config(args, world):
    """`config` of the c2 line -- identical in both arms (same workload, named once)."""
    n = args.n
    return {"workload": f"{n // 1_000_000}M-splat {args.kind} cloud per GPU (SURVEY 8d generator), SOR k=16 sigma=2.0; "
                        f"global filter over the union cloud of {n * world} splats",
            "splats_per_gpu": n, "k": K_SOR, "sigma": SIGMA, "cloud": args.kind}


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  nvidia-smi needs ~0.1 s to produce its
    first row and the default timed region is shorter than that, so the sampler is started BEFORE the warm-up steps
    (25 ms period), every row is stamped with the host clock, and `stop()` keeps the rows that fall inside
    [window_begin(), window_end()] -- the timed steps.  If the timed region was too short to catch a row, the rows
    of the warm-up steps (the same kernels on the same data) are reported instead and `window` says so."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index
        self.t0 = self.t1 = self.extra_from = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), [c.strip() for c in line.split(",")]))

    def window_begin(self):
        self.t0 = time.monotonic()

    def window_end(self):
        self.t1 = time.monotonic()

    def need_more(self) -> bool:
        """True while no row fell into the timed window AND no row has arrived yet from the extra busy steps the caller
        runs in the meantime (so the reported clocks are clocks UNDER LOAD, never idle clocks).  Gives up after 3 s."""
        if not self.proc:
            return False
        if self.t0 is not None and self.t1 is None:
            self.window_end()
        if [1 for t, _ in self.rows if self.t0 is not None and self.t0 <= t <= self.t1]:
            return False
        if self.extra_from is None:
            self.extra_from = time.monotonic()
        if time.monotonic() > self.extra_from + 3.0:
            return False
        return not [1 for t, _ in self.rows if t > self.extra_from + 0.03]

    def stop(self, keep_busy=None):
        """keep_busy: callable that runs one more (untimed) step while need_more()."""
        if not self.proc:
            return None
        while self.need_more():
            if keep_busy is not None:
                keep_busy()
            else:
                time.sleep(0.02)
        self.t_stop = time.monotonic()
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        ok = [(t, r) for t, r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        if not ok:
            return None
        window = "timed region"
        sel = [r for t, r in ok if self.t0 is not None and self.t0 <= t <= self.t1]
        if not sel and self.extra_from is not None:
            sel = [r for t, r in ok if self.extra_from + 0.03 < t <= self.t_stop]
            window = "extra untimed steps right after the timed region (it was shorter than nvidia-smi's sampling period)"
        if not sel:
            sel = [r for _, r in ok]
            window = "whole run (no row inside the timed region)"
        sm = [float(r[1]) for r in sel]
        mx = [float(r[2]) for r in sel if r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in sel:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


def finish_clocks(clocks, world, rank, dev, busy_step):
    """Stop the sampler on rank 0; while it still needs a row under load, EVERY rank runs extra untimed steps
    (the step may contain collectives, so the decision is broadcast from rank 0)."""
    import torch
    sync = torch.cuda.synchronize if torch.device(dev).type == "cuda" else (lambda: None)
    if world == 1:
        return clocks.stop(keep_busy=lambda: (busy_step(), sync()))
    import torch.distributed as dist
    for _ in range(64):
        need = torch.tensor([1 if (rank == 0 and clocks.need_more()) else 0], dtype=torch.int32, device=dev)
        dist.broadcast(need, 0)
        if int(need.item()) == 0:
            break
        busy_step()
        sync()
    return clocks.stop() if rank == 0 else None


def peaks():
    try:
        return json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        return {}


# ----------------------------------------------------------------------------- CPU reference arm
def cpu_reference_sor(xyz_sample: np.ndarray, k: int, sigma: float):
    """The reference's CPU implementation of the path (data_processor.py:155-180): SciPy cKDTree, exact
    (k+1)-NN on cpu_count()-1 workers, mean/std threshold.  (Port: oracle/sor.py restates those lines with the
    same SciPy calls.)"""
    sys.path.insert(0, str(ROOT))
    import oracle
    t0 = time.perf_counter()
    md = oracle.sor_ckdtree_mean_dists(xyz_sample, k, workers=max(1, (os.cpu_count() or 2) - 1))
    mask = oracle.threshold_mask(md, sigma)
    return time.perf_counter() - t0, int(mask.sum())


def cpu_taichi_port_sor(xyz_sample: np.ndarray, k: int, sigma: float, mode: str):
    """Same algorithm as the GPU path (Taichi semantics) on all host cores: the C oracle."""
    sys.path.insert(0, str(ROOT))
    import oracle
    t0 = time.perf_counter()
    md = oracle.sor_taichi_mean_dists(xyz_sample, k, mode)
    mask = oracle.threshold_mask(md, sigma)
    return time.perf_counter() - t0, int(mask.sum())


def run_reference(args):
    """`--impl reference`: rank 0 alone times the reference's cKDTree SOR on the c2 cloud.  A step = the whole filter
    on the FULL per-GPU cloud when the run fits REFERENCE_BUDGET_S, else on the largest prefix that does (stated)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.config != "c2":
        print(json.dumps({"impl": "reference", "unavailable": f"the reference arm is defined for --config c2 only "
                                                               f"(got {args.config})"}), flush=True)
        return
    synth = load_synth()
    n = args.n
    xyz = synth.xyz(n, args.kind)
    total_steps = args.warmup + args.steps
    ns = n
    # one probe step on a 1 M prefix sizes the sample (tree build + queries are ~n log n)
    probe_n = min(n, 1_000_000)
    dt_probe, _ = cpu_reference_sor(np.ascontiguousarray(xyz[:probe_n]), K_SOR, SIGMA)
    est_full = dt_probe * (n / probe_n) * 1.35
    if est_full * total_steps > REFERENCE_BUDGET_S:
        ns = int(max(probe_n, min(n, probe_n * REFERENCE_BUDGET_S / (dt_probe * 1.35 * total_steps))))
        ns -= ns % 1000
    sample = np.ascontiguousarray(xyz[:ns])
    times = []
    for i in range(total_steps):
        dt, kept = cpu_reference_sor(sample, K_SOR, SIGMA)
        if i >= args.warmup:
            times.append(dt)
    t = float(np.mean(times))
    val = ns / t / 1e6
    cores = os.cpu_count() or 1
    what = "the full per-GPU cloud" if ns == n else f"the first {ns} points of the cloud (the full cloud would not fit " \
                                                     f"{REFERENCE_BUDGET_S:.0f} s for {total_steps} steps)"
    line = {
        "impl": "reference", "metric": "Msplats/s SOR k=16", "value": round(val, 4), "unit": "Msplats/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(t * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": c2_config(args, args.gpus),
        "cpu_baseline": {"value": round(val, 4), "unit": "Msplats/s", "cores": cores, "kind": "port",
                         "sample": f"every step = the whole filter on {what}; reference CPU path = SciPy cKDTree "
                                   f"(k+1)-NN (data_processor.py:155-180) with workers=cpu_count()-1={max(1, cores - 1)}; "
                                   f"semantics: exact float64 KNN (the GPU arm's default is the Taichi hash-grid semantics; "
                                   f"its like_for_like object times the cKDTree-semantics GPU path)",
                         "sample_points": ns, "kept": kept},
        "e2e": {"value": round(val, 4), "unit": "Msplats/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- gsx arm plumbing
def setup_dist():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    return world, rank, local_rank, dev


def barrier(world):
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, dev, world):
    import torch
    import torch.distributed as dist
    if world == 1:
        return float(x)
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sha(t):
    """Digest of a device tensor's bytes (host side)."""
    return hashlib.sha256(t.contiguous().cpu().numpy().tobytes()).hexdigest()[:16]


def gather_to_rank0(t, world, rank):
    """Concatenation of every rank's 1-D / 2-D tensor on rank 0 (ragged allowed); None elsewhere."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return t
    n = torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device)
    sizes = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(sizes, n)
    sizes = [int(s.item()) for s in sizes]
    if rank == 0:
        out = torch.empty((sum(sizes),) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        off = sizes[0]
        out[:off] = t
        for r in range(1, world):
            if sizes[r]:
                dist.recv(out[off: off + sizes[r]], src=r)
            off += sizes[r]
        return out
    if t.shape[0]:
        dist.send(t.contiguous(), dst=0)
    return None


def device_cloud(n, dev, seed, synth, want_opacity=False, chunk=1 << 24):
    """The SURVEY 8(d) `mixed` distribution generated on the device (torch RNG; configs too large for the host
    generator, SURVEY 8d last bullet).  Inputs only -- nothing here is timed."""
    import torch
    g = torch.Generator(device=dev).manual_seed(int(seed))
    c_np, s_np = synth._cluster_params()
    c = torch.from_numpy(c_np.astype(np.float32)).to(dev)
    s = torch.from_numpy(s_np.astype(np.float32)).to(dev)
    xyz = torch.empty((n, 3), dtype=torch.float32, device=dev)
    op = torch.empty(n, dtype=torch.float32, device=dev) if want_opacity else None
    for a in range(0, n, chunk):
        m = min(chunk, n - a)
        u = torch.rand(m, device=dev, generator=g)
        uni = torch.rand((m, 3), device=dev, generator=g) * 20.0 - 10.0
        j = torch.randint(0, 16, (m,), device=dev, generator=g)
        gau = c[j] + s[j, None] * torch.randn((m, 3), device=dev, generator=g)
        fly = torch.rand((m, 3), device=dev, generator=g) * 24.0 - 12.0
        xyz[a:a + m] = torch.where((u < 0.4975)[:, None], uni, torch.where((u < 0.995)[:, None], gau, fly))
        if want_opacity:
            op[a:a + m] = torch.randn(m, device=dev, generator=g) * 2.0
        del u, uni, j, gau, fly
    return xyz, op


def device_sh_rows(n, dev, seed, D=45, chunk=1 << 22):
    """SH block of SURVEY 8(d): 1024 prototypes N(0,0.15^2) + N(0,0.03^2) noise, float32 [n, D] on the device."""
    import torch
    g = torch.Generator(device=dev).manual_seed(int(seed))
    proto = torch.randn(1024, D, device=dev, generator=g) * 0.15
    X = torch.empty((n, D), dtype=torch.float32, device=dev)
    for a in range(0, n, chunk):
        m = min(chunk, n - a)
        idx = torch.randint(0, 1024, (m,), device=dev, generator=g)
        X[a:a + m] = proto[idx] + 0.03 * torch.randn(m, D, device=dev, generator=g)
    return X


def sog_schedule(n_rows, level=5):
    """formats/sog.py:513-532: (num_chunks, chunk_size, k_per_chunk) of the shN clustering."""
    official = min(64, 2 ** int(np.floor(np.log2(max(n_rows, 1024) / 1024)))) * 1024
    target_k = min(65536, official) if level <= 3 else (min(16384, official) if level <= 6 else min(4096, official))
    target_k = max(256, target_k)
    num_chunks = max(1, min(64, n_rows // 1024))
    chunk = int(np.ceil(n_rows / num_chunks))
    return num_chunks, chunk, max(16, int(np.ceil(target_k / num_chunks)))


DUMP_SAMPLE = 1 << 21   # points of the dumped sample: 32 MiB of .npy files at most


def dump_outputs(out_dir: Path, mask, means=None):
    """What a caller of the c2 path receives from one step -- the keep-mask and (one GPU) the SOR mean distances --
    as .npy files, so that two builds can be compared output for output.  Above DUMP_SAMPLE points, the same seeded
    sample of point indices is written every run (`sample_index`).  `keep_count` (masked points of the whole cloud)
    and `mean_std` (the threshold statistics over all mean distances) cover every point."""
    import torch
    from gsx import sor
    n = mask.numel()
    if n > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))
    else:
        idx = np.arange(n)
    idx_d = torch.from_numpy(idx).to(mask.device)
    out = {"sample_index": idx.astype(np.float64),
           "keep_mask": mask[idx_d].cpu().numpy().astype(np.float32),
           "keep_count": np.array([int(mask.sum())], dtype=np.float64)}
    if means is not None:
        out["mean_dists"] = means[idx_d].cpu().numpy()
        out["mean_std"] = sor.mean_std(means).cpu().numpy()
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in out.items():
        np.save(out_dir / f"{name}.npy", a)


# ----------------------------------------------------------------------------- c2: the contract line
def run_c2(args):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(PKG))
    world, rank, local_rank, dev = setup_dist()
    from gsx import sor, synth, _abi
    from gsx import dist as gd
    n = args.n
    blocks_per_rank = (n + synth.BLOCK - 1) // synth.BLOCK
    xyz_np = synth.xyz(n, args.kind, start_block=rank * blocks_per_rank)
    xyz = torch.from_numpy(xyz_np).to(dev)
    n_total = n * world
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    ws = sor.workspace(n, dev) if world == 1 else None
    means = torch.empty(n, dtype=torch.float32, device=dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    knn_ms, build_ms = [], []
    use_dist_build = os.environ.get("GSX_DIST_BUILD", "1") != "0"

    def step(timed: bool):
        """One pass of the hot path; returns the keep-mask of this rank's slab (device)."""
        flush.fill_(1)  # L2 flush between iterations (a 256 MiB write; < 0.3 % of a step)
        if world == 1:
            e0, e1, e2 = ev(), ev(), ev()
            e0.record()
            grid = sor.build_grid(xyz, ws)
            e1.record()
            sor.mean_dists(grid, K_SOR, args.hash, out=means)
            e2.record()
            mask = sor.threshold_mask(means, sor.mean_std(means), SIGMA)
            if timed:
                step.events.append((e0, e1, e2))
            return mask
        return gd.sor_filter_auto(xyz, K_SOR, SIGMA, args.hash)

    step.events = []
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()          # before the warm-up: nvidia-smi's first row takes longer than a short timed region
    for _ in range(args.warmup):
        mask = step(False)
    barrier(world)
    launches0 = _abi.lib.gsx_kernel_launches()
    t_start, t_end = ev(), ev()
    barrier(world)
    clocks.window_begin()
    t_start.record()
    for _ in range(args.steps):
        mask = step(True)
    t_end.record()
    barrier(world)
    clocks.window_end()
    launches = _abi.lib.gsx_kernel_launches() - launches0
    if args.dump_outputs and rank == 0:       # before the busy steps below reuse `means`
        dump_outputs(Path(args.dump_outputs), mask, means if world == 1 else None)
    clk = finish_clocks(clocks, world, rank, dev, lambda: step(False))
    elapsed_ms = max_over_ranks(t_start.elapsed_time(t_end), dev, world)
    ms_per_step = elapsed_ms / args.steps
    value = n_total / (ms_per_step * 1e-3) / 1e6
    kept_t = mask.sum().to(torch.int64)
    if world > 1:
        dist.all_reduce(kept_t)
    kept = int(kept_t.item())

    # ---- per-stage times (N=1: events inside the timed steps; N>1: two extra untimed steps with stage stamps)
    stage = {}
    if world == 1:
        for e0, e1, e2 in step.events:
            build_ms.append(e0.elapsed_time(e1))
            knn_ms.append(e1.elapsed_time(e2))
        stage = {"build": round(float(np.mean(build_ms)), 3), "knn": round(float(np.mean(knn_ms)), 3)}
        knn_avg_ms = float(np.mean(knn_ms))
    else:
        acc = {}
        reps = 2
        for _ in range(reps):
            tm = {}
            flush.fill_(1)
            gd.sor_filter_auto(xyz, K_SOR, SIGMA, args.hash, timings=tm)
            for k_, v in tm.items():
                acc[k_] = acc.get(k_, 0.0) + v / reps
        stage = {k_: round(max_over_ranks(v, dev, world), 3) for k_, v in sorted(acc.items())}
        knn_avg_ms = stage.get("knn", float("nan"))

    # ---- roofline of the dominant kernel (k_sor_knn).  The kernel is INSTRUCTION-ISSUE bound (ncu: issue-active
    # ~83 %, DRAM ~2.5 % of peak): its roofline is the warp-instruction issue rate.  Instructions per launch come
    # from the committed ncu capture of the same config (profiles/r02_knn_ncu.json); the byte models are context.
    if world == 1:
        grid = sor.build_grid(xyz, ws)
        _, st = sor.mean_dists(grid, K_SOR, args.hash, out=means, want_stats=True)
    else:
        grid, sizes, seg = gd.build_grid_distributed(xyz)
        tmp = torch.zeros(n_total, dtype=torch.float32, device=dev)
        _, st = sor.mean_dists_strided(grid, K_SOR, args.hash, tmp, world, rank, want_stats=True)
        del tmp, grid
    pk = peaks()
    hbm = float(pk.get("hbm_gbs", 6650.0))
    sm_mhz = float(pk.get("sm_max_mhz", 1965.0))
    issue_peak = 148 * 4 * sm_mhz * 1e6 / 1e9          # G warp-instructions / s: 148 SMs x 4 schedulers x clock
    alg_bytes = st["queries"] * (16 + 27 * 8 + 4) + 16 * st["scanned"] + 32 * (st["box_tests"] + st.get("box_loads", 0))
    ref_model_bytes = st["queries"] * (16 + 27 * 8 + 4) + 16 * st["visits"]
    # the newest committed capture taken with THIS build of the query kernel (gsx_build_info) and this configuration
    from gsx import _abi as _gabi
    build_info = _gabi.lib.gsx_build_info().decode()
    prof = {}
    for cand in ("r02c_knn_ncu.json", "r02_knn_ncu.json"):
        try:
            c = json.loads((ROOT / "profiles" / cand).read_text())
        except Exception:
            continue
        if c.get("build_info", "knn=r02") == build_info or (cand == "r02_knn_ncu.json" and not prof):
            prof = dict(c, file=cand)
            if c.get("build_info") == build_info:
                break
    same_cfg = bool(prof) and world == 1 and n == prof.get("n") and args.kind == prof.get("kind") and \
        args.hash == prof.get("hash") and prof.get("build_info") == build_info
    winst = prof.get("warp_instructions_per_launch") if same_cfg else None
    traffic = prof.get("dram_bytes_per_launch") if same_cfg else None
    kname = (prof.get("kernel") or "k_sor_knn16 (K<=16) / k_sor_knn").split("(const")[0].replace("void ", "").strip()
    roofline = {"bound": "issue", "kernel": kname,
                "achieved": round(winst / (knn_avg_ms * 1e-3) / 1e9, 1) if winst else None,
                "peak": round(issue_peak, 1), "unit": "Gwarp-instr/s",
                "frac": round(winst / (knn_avg_ms * 1e-3) / 1e9 / issue_peak, 4) if winst else None,
                "peak_source": "148 SMs x 4 warp schedulers x sm_max_mhz of MEASURED_PEAKS.json",
                "traffic": traffic,
                "dram_frac": round(traffic / (knn_avg_ms * 1e-3) / 1e9 / hbm, 4) if traffic else None,
                "hbm_peak_gbs": hbm,
                "kernel_ms": round(knn_avg_ms, 3), "kernel_share_of_step": round(knn_avg_ms / ms_per_step, 3),
                "warp_instr_per_query": round(winst / prof["queries"], 1) if winst else None,
                "ncu_issue_active_pct": prof.get("issue_active_pct") if same_cfg else None,
                "ncu_capture": prof.get("file") if same_cfg else None, "build_info": build_info,
                "per_query": {"ref_visits_V": round(st["visits"] / st["queries"], 1),
                              "scanned": round(st["scanned"] / st["queries"], 1),
                              "box_tests": round(st["box_tests"] / st["queries"], 1)},
                "gather_model": {"algorithmic_bytes_per_launch": int(alg_bytes),
                                 "GBps": round(alg_bytes / (knn_avg_ms * 1e-3) / 1e9, 1),
                                 "frac_of_hbm": round(alg_bytes / (knn_avg_ms * 1e-3) / 1e9 / hbm, 4),
                                 "reference_model_GBps": round(ref_model_bytes / (knn_avg_ms * 1e-3) / 1e9, 1),
                                 "note": "bytes the pruned search gathers (L1/L2-served); SURVEY 8(d)'s un-pruned "
                                         "reference model (16 B x V visits) is reference_model_GBps; neither is DRAM "
                                         "traffic -- `traffic`/`dram_frac` are (ncu)"}}

    cfg = c2_config(args, world)
    line = {
        "metric": "Msplats/s SOR k=16", "value": round(value, 3), "unit": "Msplats/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "run": {"semantics": "taichi", "hash_mode": args.hash, "kept": kept,
                "l2": "256 MiB flush write before every step + working set (~0.6 GB/step) larger than L2",
                "parallelism": (f"dp{world}: owner-partitioned distributed grid build (all-to-all + ragged segment "
                                f"exchange), own-segment queries, reduce-scatter of the mean distances, sharded "
                                f"NumPy-order statistics" if use_dist_build else
                                f"dp{world}: all-gather xyz, replicated grid, sharded queries, one all-reduce")
                if world > 1 else "single GPU"},
        "stage_ms": stage, "gpu_launches": int(launches), "roofline": roofline,
    }
    if clk:
        line["clocks"] = clk

    if world == 1 and not args.no_extras:
        line["e2e"] = measure_e2e(xyz_np, args, pinned=True)
        line["e2e"]["pageable_input"] = measure_e2e(xyz_np, args, pinned=False)
        line["cpu_baseline"] = measure_cpu_baseline(xyz_np, args)
        line["like_for_like"] = measure_like_for_like(xyz, xyz_np, args, line["cpu_baseline"])
        line["other_modes"] = measure_other(xyz, ws, means, args)
        line["pipeline"] = measure_pipeline(xyz_np, args)
        try:
            line["host_rows"] = measure_host_rows(xyz_np)
        except Exception as e:  # noqa: BLE001  (an extra: never lose the bench line over it)
            line["host_rows"] = {"error": str(e)[:200]}
        del ws
        torch.cuda.empty_cache()
        line["kmeans"] = measure_kmeans(dev, full=True)
    elif world > 1:
        line["e2e"] = measure_e2e_sharded(xyz_np, args, dev, rank, world)
        if not args.no_extras:
            line["parity"] = measure_parity(xyz, mask, args, dev, rank, world)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def measure_parity(xyz, mask_local, args, dev, rank, world):
    """Outside the timed region: the N-rank masks against the single-GPU filters on the union cloud (rank 0)."""
    import torch
    from gsx import sor, density
    from gsx import dist as gd
    dmask_local, dinfo = gd.density_filter_sharded(xyz, sensitivity=0.5, keep_multicluster=True)
    xyz_all = gather_to_rank0(xyz, world, rank)
    mask_all = gather_to_rank0(mask_local.view(torch.uint8), world, rank)
    dmask_all = gather_to_rank0(dmask_local.view(torch.uint8), world, rank)
    out = None
    if rank == 0:
        torch.cuda.empty_cache()
        m1 = sor.sor_filter(xyz_all, K_SOR, SIGMA, hash_mode=args.hash).view(torch.uint8)
        d1, info1 = density.density_filter(xyz_all, sensitivity=0.5, keep_multicluster=True)
        d1 = d1.view(torch.uint8)
        out = {"what": f"{world}-rank keep-masks vs the single-GPU filter on the union cloud of {xyz_all.shape[0]} splats",
               "sor": {"mask_sha_nranks": sha(mask_all), "mask_sha_1gpu": sha(m1),
                       "equal": bool(torch.equal(mask_all, m1)), "kept": int(m1.sum().item())},
               "density": {"mask_sha_nranks": sha(dmask_all), "mask_sha_1gpu": sha(d1),
                           "equal": bool(torch.equal(dmask_all, d1)), "kept": int(d1.sum().item()),
                           "clusters": int(info1["clusters"])},
               }
        out["equal"] = out["sor"]["equal"] and out["density"]["equal"]
    return out


def measure_e2e(xyz_np, args, pinned: bool):
    """Same metric through the reference-facing plugin call with HOST buffers:
    gsconverter.processing.gpu_ops.filter_sor_gpu(np.ndarray) -> np.ndarray[bool];
    H2D of the xyz and D2H of the mask are inside the timed region.  pinned=False: a plain (pageable) NumPy array,
    which is what the reference call site passes (np.column_stack, data_processor.py:139)."""
    import torch
    os.environ["GSX_SOR_HASH"] = args.hash
    from gsconverter.processing import gpu_ops
    n = len(xyz_np)
    if pinned:
        buf = torch.empty((n, 3), dtype=torch.float32).pin_memory()
        host = buf.numpy()
        host[:] = xyz_np
    else:
        host = xyz_np.copy()
    for _ in range(2):
        m = gpu_ops.filter_sor_gpu(host, K_SOR, SIGMA)
    torch.cuda.synchronize()
    reps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(reps):
        m = gpu_ops.filter_sor_gpu(host, K_SOR, SIGMA)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    return {"value": round(n / dt / 1e6, 3), "unit": "Msplats/s", "ms_per_step": round(dt * 1e3, 3),
            "h2d_bytes_per_step": int(n * 12), "d2h_bytes_per_step": int(n), "host_input": "pinned" if pinned else "pageable",
            "api": "gsconverter.processing.gpu_ops.filter_sor_gpu(numpy[N,3]) -> numpy bool[N]", "kept": int(m.sum())}


def measure_e2e_sharded(xyz_np, args, dev, rank, world):
    """N>1: host slab -> device -> sharded global filter -> host mask, per rank; max over ranks."""
    import torch
    import torch.distributed as dist
    from gsx import dist as gd
    n = len(xyz_np)
    pinned = torch.empty((n, 3), dtype=torch.float32).pin_memory()
    pinned.numpy()[:] = xyz_np
    out = torch.empty(n, dtype=torch.bool).pin_memory()

    def once():
        x = pinned.to(dev, non_blocking=True)
        mask = gd.sor_filter_auto(x, K_SOR, SIGMA, args.hash)
        out.copy_(mask, non_blocking=True)
        torch.cuda.synchronize()
    once()
    dist.barrier()
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    dist.barrier()
    dt = max_over_ranks((time.perf_counter() - t0) / reps, dev, world)
    return {"value": round(n * world / dt / 1e6, 3), "unit": "Msplats/s", "ms_per_step": round(dt * 1e3, 3),
            "h2d_bytes_per_step": int(n * 12), "d2h_bytes_per_step": int(n), "host_input": "pinned",
            "api": "gsx.dist.sor_filter_auto(host slab per rank)"}


def measure_cpu_baseline(xyz_np, args):
    ns = min(args.cpu_sample, len(xyz_np))
    sample = np.ascontiguousarray(xyz_np[:ns])
    cores = os.cpu_count() or 1
    dt, kept = cpu_reference_sor(sample, K_SOR, SIGMA)
    dt2, kept2 = cpu_taichi_port_sor(sample, K_SOR, SIGMA, args.hash)
    dens = None
    try:   # SURVEY 8(d) CPU baseline (b): the reference's NumPy density filter (data_processor.py:11-117), same sample
        import oracle
        t0 = time.perf_counter()
        dmask, dinfo = oracle.density_mask(sample, sensitivity=0.5, keep_multicluster=True)
        dt3 = time.perf_counter() - t0
        dens = {"value": round(ns / dt3 / 1e6, 4), "unit": "Msplats/s", "seconds": round(dt3, 3), "kept": int(dmask.sum()),
                "what": "apply_density_filter(sensitivity=0.5, keep_multicluster) as NumPy (oracle/filters.py, pinned to the "
                        "imported reference by tests/golden/make_goldens.py), one thread, same sample"}
    except Exception as e:  # noqa: BLE001
        dens = {"error": str(e)[:200]}
    return {"density": dens, "value": round(ns / dt / 1e6, 4), "unit": "Msplats/s", "cores": cores, "kind": "port",
            "sample": f"first {ns} points of the bench cloud, one pass; reference CPU path = SciPy cKDTree "
                      f"(k+1)-NN on cpu_count()-1={max(1, cores - 1)} workers + mean/std mask "
                      f"(data_processor.py:155-180); the --impl reference arm times the full cloud",
            "seconds": round(dt, 3),
            "taichi_semantics_port": {"value": round(ns / dt2 / 1e6, 4), "unit": "Msplats/s", "seconds": round(dt2, 3),
                                      "what": "C/OpenMP oracle of the Taichi kernel (same results as the GPU path), "
                                              "all host cores, same sample"}}


def measure_like_for_like(xyz, xyz_np, args, cpu_bl):
    """The SAME function on both sides: exact float64 (k+1)-NN SOR (cKDTree semantics, data_processor.py:155-180) --
    gsx's GPU implementation of it (bit-identical to SciPy, tests/test_sor_ckdtree_gpu.py) against SciPy on the host
    cores, on the same prefix of the cloud."""
    import torch
    from gsx import sor
    out = {}
    try:
        ns = min(args.cpu_sample, len(xyz_np))
        xs = xyz[:ns].contiguous()
        for _ in range(2):
            sor.ckdtree_filter(xs, K_SOR, SIGMA)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(3):
            m = sor.ckdtree_filter(xs, K_SOR, SIGMA)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / 3
        host = np.ascontiguousarray(xyz_np[:ns])
        sor.ckdtree_filter_host(host, K_SOR, SIGMA)
        t0 = time.perf_counter()
        mh = sor.ckdtree_filter_host(host, K_SOR, SIGMA)
        dt = time.perf_counter() - t0
        out = {"semantics": "ckdtree (exact float64 KNN)", "points": ns,
               "gpu_device_ms": round(ms, 3), "gpu_device_msplats_s": round(ns / ms / 1e3, 2),
               "gpu_e2e_host_buffers_msplats_s": round(ns / dt / 1e6, 2),
               "cpu_scipy_msplats_s": cpu_bl["value"], "cpu_cores": cpu_bl["cores"],
               "ratio_device": round(ns / ms / 1e3 / cpu_bl["value"], 1),
               "ratio_e2e": round(ns / dt / 1e6 / cpu_bl["value"], 1),
               "kept": int(m.sum().item()), "kept_host_call": int(mh.sum())}
        # the full cloud on the GPU as well (the CPU side of that size is the --impl reference arm)
        sor.ckdtree_filter(xyz, K_SOR, SIGMA)          # warm-up at this size (the first call grows torch's allocator)
        torch.cuda.synchronize()
        a.record()
        mf = sor.ckdtree_filter(xyz, K_SOR, SIGMA)
        b.record()
        torch.cuda.synchronize()
        out["gpu_full_cloud"] = {"points": int(xyz.shape[0]), "ms": round(a.elapsed_time(b), 2),
                                 "msplats_s": round(xyz.shape[0] / a.elapsed_time(b) / 1e3, 2), "kept": int(mf.sum().item())}
    except Exception as e:  # noqa: BLE001
        out["error"] = str(e)[:300]
    return out


def measure_other(xyz, ws, means, args):
    """Whole-filter throughput for the other probe-hash mode and the uniform cloud (device-resident)."""
    import torch
    from gsx import sor, synth
    out = {}

    def timed(x, mode):
        for _ in range(2):
            sor.sor_filter(x, K_SOR, SIGMA, hash_mode=mode, ws=ws)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(5):
            sor.sor_filter(x, K_SOR, SIGMA, hash_mode=mode, ws=ws)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / 5

    try:   # the density filter alone on the resident cloud (BASELINE configs[1]: density_sensitivity 0.5)
        from gsx import density
        for _ in range(2):
            density.density_filter(xyz, sensitivity=0.5, keep_multicluster=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            dm, dinfo = density.density_filter(xyz, sensitivity=0.5, keep_multicluster=True)
        torch.cuda.synchronize()
        dms = (time.perf_counter() - t0) / 3 * 1e3
        out[f"density_0.5_multicluster_{args.kind}"] = {"ms": round(dms, 3), "msplats_s": round(xyz.shape[0] / dms / 1e3, 2),
                                                       "kept": int(dm.sum().item()), "clusters": int(dinfo["clusters"]),
                                                       "note": "wall clock incl. the host cluster selection between the "
                                                               "two device stages"}
    except Exception as e:  # noqa: BLE001
        out["density_error"] = str(e)[:200]
    other = "i64" if args.hash == "i32wrap" else "i32wrap"
    ms = timed(xyz, other)
    out[f"{args.kind}_{other}"] = {"ms": round(ms, 3), "msplats_s": round(xyz.shape[0] / ms / 1e3, 2)}
    if args.kind != "uniform":
        xu = torch.from_numpy(synth.xyz(xyz.shape[0], "uniform")).to(xyz.device)
        for mode in ("i32wrap", "i64"):
            ms = timed(xu, mode)
            out[f"uniform_{mode}"] = {"ms": round(ms, 3), "msplats_s": round(xu.shape[0] / ms / 1e3, 2)}
    return out


def measure_pipeline(xyz_np, args):
    """BASELINE configs[1] chained (converter.py:194-236 order): bbox -> alpha(5) -> density(0.5, multicluster)
    -> SOR k=16 on the 10 M cloud through gsx.pipeline.FilterChain: pinned host xyz+opacity in, surviving row
    indices out (the device-resident working set; host records are gathered once by the caller)."""
    import torch
    from gsx.pipeline import FilterChain
    n = len(xyz_np)
    op_np = np.random.default_rng(1).normal(0, 2, n).astype(np.float32)
    px = torch.empty((n, 3), dtype=torch.float32).pin_memory()
    px.numpy()[:] = xyz_np
    po = torch.empty(n, dtype=torch.float32).pin_memory()
    po.numpy()[:] = op_np

    def once():
        ch = FilterChain(px, po)
        c0 = ch.crop_by_bbox(-11, -11, -11, 11, 11, 11)
        c1 = ch.alpha(5)
        c2, _ = ch.density(sensitivity=0.5, keep_multicluster=True)
        c3 = ch.sor(K_SOR, SIGMA, hash_mode=args.hash)
        idx = ch.indices()
        return (c0, c1, c2, c3, len(idx))
    once()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        counts = once()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    return {"what": "bbox -> alpha(5) -> density(0.5, multicluster) -> SOR k=16, host columns in, surviving indices out",
            "ms": round(dt * 1e3, 2), "msplats_s": round(n / dt / 1e6, 2), "survivors_per_stage": list(counts[:4]),
            "h2d_bytes": int(n * 16), "d2h_bytes": int(counts[4] * 4)}


def measure_host_rows(xyz_np, n=1_000_000):
    """Host-resident records (a1: where the reference's time goes once the masks are cheap): np.column_stack of the
    filter columns and the `vertices[mask]` gather of 248-byte records, NumPy (one thread) vs libgsx's threaded
    gsx_host_extract_xyz_opacity / gsx_host_gather_rows, on a 1 M-record sample with 60 % survivors (NumPy's structured
    fancy index takes seconds per million records, so the sample is kept small).  CPU only."""
    from gsx import hostrows
    n = min(n, len(xyz_np))
    names = (["x", "y", "z", "nx", "ny", "nz", "f_dc_0", "f_dc_1", "f_dc_2"] + [f"f_rest_{i}" for i in range(45)] +
             ["opacity", "scale_0", "scale_1", "scale_2", "rot_0", "rot_1", "rot_2", "rot_3"])   # structures.py:23-59
    rec = np.zeros(n, dtype=[(nm, "f4") for nm in names])
    rec["x"], rec["y"], rec["z"] = xyz_np[:n, 0], xyz_np[:n, 1], xyz_np[:n, 2]
    idx = np.flatnonzero(np.random.default_rng(3).random(n) < 0.6).astype(np.int64)

    def best(fn, reps=3):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            r = fn()
            ts.append(time.perf_counter() - t0)
        return min(ts), r
    t_np, a = best(lambda: rec[idx], reps=1)
    t_gx, b = best(lambda: hostrows.take_rows(rec, idx))
    same = a.tobytes() == b.tobytes()
    del a, b
    t_np2, c = best(lambda: np.column_stack((rec["x"], rec["y"], rec["z"])), reps=2)
    t_gx2, d = best(lambda: hostrows.xyz_opacity(rec))
    same = same and c.tobytes() == d[0].tobytes()
    return {"records": n, "record_bytes": rec.dtype.itemsize, "survivors": int(len(idx)), "identical_bytes": bool(same),
            "gather_rows": {"numpy_ms": round(t_np * 1e3, 1), "gsx_ms": round(t_gx * 1e3, 1),
                            "gsx_GBps_read_plus_write": round(len(idx) * rec.dtype.itemsize * 2 / t_gx / 1e9, 1)},
            "column_stack_xyz": {"numpy_ms": round(t_np2 * 1e3, 1), "gsx_ms": round(t_gx2 * 1e3, 1)},
            "threads": os.environ.get("GSX_HOST_THREADS", "default (16 on a host with >= 32 cores)")}


# ----------------------------------------------------------------------------- c3: K-Means (secondary BASELINE metric)
def measure_kmeans(dev, full=True, nprob=64, rows=781_250, iters=10):
    """K-Means iterations/s on the SOG shN schedule (sog.py:527-549): 64 chunks x 781 250 x 45, K=256 (the 50 M-splat
    C3 config, 9 GB of SH rows), 10 Lloyd iterations -- the schedule's own count.  value = chunk-iterations / s.
    roofline: the iteration streams X twice (assign: score GEMM on the tensor cores; update: member walk) -> HBM."""
    import torch
    from gsx import kmeans as gk
    D, K = 45, 256
    X = device_sh_rows(nprob * rows, dev, 20260923, D)
    offs = [p * rows for p in range(nprob + 1)]
    init = torch.stack([X[offs[p]:offs[p] + K] for p in range(nprob)])
    pk = peaks()
    hbm = float(pk.get("hbm_gbs", 6650.0))
    out = {"metric": "K-Means chunk-iterations/s (781250x45, K=256)", "chunks": nprob, "iters": iters,
           "config": "BASELINE configs[2]: 50M-splat scene, SOG --compression_level 5 shN schedule"}
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    modes = ("tensor", "strict") if full else ("tensor",)
    for mode in modes:
        its = iters if mode == "tensor" else 2
        gk.kmeans_lloyd_batched(X, offs, K, 1, init, assign=mode)
        torch.cuda.synchronize()
        a.record()
        r = gk.kmeans_lloyd_batched(X, offs, K, its, init, assign=mode, want_stats=True)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        ci = nprob * its / (ms * 1e-3)
        if mode == "tensor":
            bytes_it = nprob * rows * (2 * (4 * D) + 4 + 4 + 4 + 4)   # X twice, labels w+r, member w+r
            flops_it = 2.0 * nprob * rows * K * 48
            out.update({"value": round(ci, 1), "unit": "chunk-iterations/s", "ms_total": round(ms, 2),
                        "ms_per_iteration": round(ms / its, 3), "assign": "tcgen05 TF32 score GEMM + exact re-check",
                        "mpoint_iters_per_s": round(nprob * rows * its / (ms * 1e-3) / 1e6, 1),
                        "candidates": r[3],
                        "roofline": {"bound": "hbm", "achieved": round(bytes_it * its / (ms * 1e-3) / 1e9, 1), "peak": hbm,
                                     "unit": "GB/s", "frac": round(bytes_it * its / (ms * 1e-3) / 1e9 / hbm, 4),
                                     "algorithmic_bytes_per_iteration": int(bytes_it),
                                     "tensor_tflops": round(flops_it * its / (ms * 1e-3) / 1e12, 1),
                                     "tensor_frac_of_bf16_sustained": round(flops_it * its / (ms * 1e-3) / 1e12 /
                                                                            float(pk.get("bf16_tflops_sustained", 1400.0)), 4),
                                     "traffic": None}})
            digest = sha(r[1][:1_000_000]) + sha(r[0])
            out["labels_centroids_sha"] = digest
        else:
            out["strict_cuda_core_assign"] = {"value": round(ci, 1), "ms_per_iteration": round(ms / its, 3),
                                              "labels_equal_tensor_after_2_iterations": None}
    del X
    torch.cuda.empty_cache()
    if full:
        # e2e through the plugin with HOST buffers: gpu_ops.kmeans on one chunk (140 MB H2D, labels + centroids D2H)
        try:
            from gsconverter.processing import gpu_ops
            xc = device_sh_rows(rows, dev, 7, D).cpu().numpy()
            np.random.seed(1)
            gpu_ops.kmeans(xc, K, max_iter=iters)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            reps = 3
            for _ in range(reps):
                gpu_ops.kmeans(xc, K, max_iter=iters)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / reps
            out["e2e"] = {"value": round(iters / dt, 1), "unit": "chunk-iterations/s", "ms_per_call": round(dt * 1e3, 2),
                          "h2d_bytes_per_step": int(xc.nbytes), "d2h_bytes_per_step": int(rows * 4 + K * D * 4),
                          "api": "gsconverter.processing.gpu_ops.kmeans(numpy[781250,45], 256, max_iter=10)"}
            from sklearn.cluster import MiniBatchKMeans
            t0 = time.perf_counter()
            MiniBatchKMeans(n_clusters=K, max_iter=10, batch_size=min(4096 * 4, len(xc)), n_init="auto",
                            compute_labels=True).fit(xc)
            dts = time.perf_counter() - t0
            out["cpu_reference_sklearn"] = {"seconds_per_chunk_max_iter10": round(dts, 2),
                                            "chunk_fits_per_s": round(1.0 / dts, 3), "cores": os.cpu_count(),
                                            "note": "the reference's fallback when Taichi is absent (gpu_ops.py:48-52: "
                                                    "MiniBatchKMeans, unseeded -- a different algorithm); one full chunk"}
        except Exception as e:  # noqa: BLE001
            out["e2e_error"] = str(e)[:300]
    return out


def run_c3(args):
    import torch
    sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(PKG))
    world, rank, local_rank, dev = setup_dist()
    from gsx import _abi
    clocks = ClockSampler(local_rank)
    clocks.start()
    clocks.window_begin()        # the whole measurement (seconds of K-Means) is the window
    l0 = _abi.lib.gsx_kernel_launches()
    km = measure_kmeans(dev, full=not args.no_extras)
    clocks.window_end()
    clk = clocks.stop()
    line = {"metric": "K-Means chunk-iterations/s", "value": km["value"], "unit": "chunk-iterations/s", "n_gpus": 1,
            "steps": km["iters"], "warmup": 1, "ms_per_step": km["ms_per_iteration"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 (tf32 tensor-core scores, exact f32 re-check)",
            "data": "synthetic", "config": {"workload": km["config"] + ": 64 chunks x 781250 x 45, K=256, 10 iterations"},
            "roofline": km["roofline"], "gpu_launches": int(_abi.lib.gsx_kernel_launches() - l0), "kmeans": km}
    if "e2e" in km:
        line["e2e"] = km["e2e"]
    if clk:
        line["clocks"] = clk
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- c4 / c5: the large sharded configs
def run_big(args):
    """c4: 4 x 50 M, SOR + density --keep_multicluster.  c5: 8 x 125 M, bbox -> alpha -> density -> SOR -> K-Means.
    Device-generated `mixed` cloud (seed + rank).  A step = the whole chain on the resident cloud; parity = the
    N-rank survivor digests against the same chain on ONE GPU over the union cloud (fits in 180 GB)."""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(PKG))
    world, rank, local_rank, dev = setup_dist()
    from gsx import synth, _abi, kmeans as gk
    from gsx import dist as gd
    from gsx.pipeline import FilterChain
    full_chain = args.config == "c5"
    n = args.n
    xyz, op = device_cloud(n, dev, synth.SEED + 1000 + rank, synth, want_opacity=True)
    n_total = n * world
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    class Chain1:  # single-process stand-in with the same interface (world == 1 and the parity run)
        def __init__(self, x, o):
            self.chain = FilterChain(x, o, device=x.device)

        def crop_by_bbox(self, *b): return self.chain.crop_by_bbox(*b)
        def alpha(self, a): return self.chain.alpha(a)
        def density(self, **kw): return self.chain.density(**kw)
        def sor(self, k, tf, hash_mode=None, timings=None): return self.chain.sor(k, tf, hash_mode=hash_mode)

        def local_indices(self):
            return torch.arange(self.chain.n0, device=dev) if self.chain.idx is None else self.chain.idx.to(torch.int64)

        @property
        def count(self): return self.chain.count

    def chain_once(x, o, sharded, timings=None):
        ch = gd.ShardedFilterChain(x, o) if sharded else Chain1(x, o)
        marks = [ev()]
        marks[0].record()
        counts = []
        if full_chain:
            counts.append(ch.crop_by_bbox(-11, -11, -11, 11, 11, 11))
            counts.append(ch.alpha(5))
            m = ev(); m.record(); marks.append(m)
            counts.append(ch.density(sensitivity=0.5, keep_multicluster=True)[0])
            m = ev(); m.record(); marks.append(m)
            counts.append(ch.sor(K_SOR, SIGMA, hash_mode=args.hash, timings=timings))
        else:   # c4: SOR + density --keep_multicluster, each on the full cloud (converter.py order: density, then SOR)
            counts.append(ch.density(sensitivity=0.5, keep_multicluster=True)[0])
            m = ev(); m.record(); marks.append(m)
            counts.append(ch.sor(K_SOR, SIGMA, hash_mode=args.hash, timings=timings))
        m = ev(); m.record(); marks.append(m)
        return ch, counts, marks

    def kmeans_once(n_surv, seed):
        """SOG schedule share of this rank: its survivors' SH rows in 64/world chunks, K=256, 10 iterations."""
        nch = max(1, 64 // world)
        rows = n_surv // nch
        X = device_sh_rows(rows * nch, dev, seed)
        offs = [p * rows for p in range(nch + 1)]
        init = torch.stack([X[offs[p]:offs[p] + 256] for p in range(nch)])
        gk.kmeans_lloyd_batched(X[: 2 * rows], offs[:3], 256, 1, init[:2])   # warm-up
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        C, L, cnt = gk.kmeans_lloyd_batched(X, offs, 256, 10, init)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b), nch, rows, sha(C), X, init

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    for _ in range(max(1, min(args.warmup, 2))):
        chain_once(xyz, op, world > 1)
    barrier(world)
    l0 = _abi.lib.gsx_kernel_launches()
    steps = max(1, args.steps)
    t0e, t1e = ev(), ev()
    barrier(world)
    clocks.window_begin()
    t0e.record()
    for _ in range(steps):
        ch, counts, marks = chain_once(xyz, op, world > 1)
    t1e.record()
    barrier(world)
    launches = _abi.lib.gsx_kernel_launches() - l0      # (the clock window stays open over the K-Means part below)
    ms_chain = max_over_ranks(t0e.elapsed_time(t1e), dev, world) / steps
    stage = {}
    names = (["bbox+alpha", "density", "sor"] if full_chain else ["density", "sor"])
    for nm, (a, b) in zip(names, zip(marks[:-1], marks[1:])):
        stage[nm] = round(max_over_ranks(a.elapsed_time(b), dev, world), 3)
    tm = {}
    ch, counts, _ = chain_once(xyz, op, world > 1, timings=tm)
    sor_break = {k_: round(max_over_ranks(v, dev, world), 3) for k_, v in sorted(tm.items())}
    surv_local = ch.local_indices()
    n_surv_local = int(surv_local.numel())
    tot = torch.tensor([n_surv_local], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tot)
    n_surv = int(tot.item())
    km = None
    ms_total = ms_chain
    if full_chain:
        del ch
        torch.cuda.empty_cache()
        ms_km, nch, rows, csha, Xk, initk = kmeans_once(n_surv_local, 555 + rank)
        ms_km = max_over_ranks(ms_km, dev, world)
        km = {"ms": round(ms_km, 2), "chunks_per_rank": nch, "rows_per_chunk": rows, "K": 256, "iters": 10,
              "chunk_iterations_per_s": round(nch * world * 10 / (ms_km * 1e-3), 1), "centroids_sha_rank0": csha,
              "sharding": "chunks are independent problems: no collective (SURVEY 8e)"}
        ms_total = ms_chain + ms_km
        # K-Means parity: rank 1's first chunk recomputed on rank 0 (same kernels, other GPU): bit-identical
        if world > 1:   # (the chunk length differs per rank: ship it first)
            blk = Xk[:rows].contiguous()
            ini = initk[0].contiguous()
            C1, _, _ = gk.kmeans_lloyd_batched(blk, [0, rows], 256, 10, ini.reshape(1, 256, -1))
            if rank == 1:
                dist.send(torch.tensor([rows], dtype=torch.int64, device=dev), dst=0)
                dist.send(blk, dst=0); dist.send(ini, dst=0); dist.send(C1.contiguous(), dst=0)
            if rank == 0:
                r1 = torch.zeros(1, dtype=torch.int64, device=dev)
                dist.recv(r1, src=1)
                r1 = int(r1.item())
                rb = torch.empty((r1, blk.shape[1]), dtype=torch.float32, device=dev)
                ri, rc = torch.empty_like(ini), torch.empty_like(C1)
                dist.recv(rb, src=1); dist.recv(ri, src=1); dist.recv(rc, src=1)
                C0, _, _ = gk.kmeans_lloyd_batched(rb, [0, r1], 256, 10, ri.reshape(1, 256, -1))
                km["parity_rank1_chunk_on_rank0"] = {"equal": bool(torch.equal(C0.view(torch.int32), rc.view(torch.int32))),
                                                    "rows": r1,
                                                    "max_rel_err": float(((C0 - rc).abs() / rc.abs().clamp_min(1e-30)).max().item())}
        del Xk, initk
        torch.cuda.empty_cache()
    clk = clocks.stop() if rank == 0 else None

    # ---- parity: the same chain on ONE GPU over the union cloud (rank 0); digests of the surviving global indices
    parity = None
    if world > 1 and not args.no_extras:
        base = rank * n
        surv_global = (surv_local + base).contiguous()
        surv_all = gather_to_rank0(surv_global, world, rank)
        xyz_all = gather_to_rank0(xyz, world, rank)
        op_all = gather_to_rank0(op, world, rank)
        if rank == 0:
            torch.cuda.empty_cache()
            t0 = time.perf_counter()
            ch1, counts1, _ = chain_once(xyz_all, op_all, False)
            torch.cuda.synchronize()
            dt1 = time.perf_counter() - t0
            s1 = ch1.local_indices()
            parity = {"what": f"{world}-rank survivors vs the same chain on one GPU over the union cloud of {n_total} splats",
                      "survivors_sha_nranks": sha(surv_all), "survivors_sha_1gpu": sha(s1),
                      "equal": bool(surv_all.shape == s1.shape and torch.equal(surv_all, s1)),
                      "survivors": int(s1.numel()), "stage_counts_1gpu": [int(c) for c in counts1],
                      "one_gpu_chain_s": round(dt1, 2)}
            del ch1, xyz_all, op_all
    cnt_g = []
    for c in counts:
        t = torch.tensor([int(c)], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t)
        cnt_g.append(int(t.item()))
    cfgname = ("BASELINE configs[4]: 1B-splat synthetic, bbox -> alpha(5) -> density(0.5) -> SOR k=16 -> K-Means (SOG level 5), "
               "8xB200" if full_chain else
               "BASELINE configs[3]: 200M-splat synthetic, SOR k=16 + density 0.5 --keep_multicluster, sharded 4xB200")
    line = {"metric": "Msplats/s full chain" if full_chain else "Msplats/s density+SOR", "value": round(n_total / (ms_total * 1e-3) / 1e6, 2),
            "unit": "Msplats/s", "n_gpus": world, "steps": steps, "warmup": max(1, min(args.warmup, 2)),
            "ms_per_step": round(ms_total, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic (device-generated SURVEY 8d mixed distribution, seed + rank)",
            "config": {"workload": cfgname, "splats_per_gpu": n, "splats_total": n_total, "k": K_SOR, "sigma": SIGMA,
                       "hash_mode": args.hash},
            "stage_ms": stage, "sor_breakdown_ms": sor_break, "survivors_per_stage": cnt_g, "survivors": n_surv,
            "chain_ms": round(ms_chain, 3), "gpu_launches": int(launches), "parity": parity}
    if km:
        line["kmeans"] = km
    if clk:
        line["clocks"] = clk
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "c2":
        run_c2(args)
    elif args.config == "c3":
        run_c3(args)
    else:
        run_big(args)


if __name__ == "__main__":
    main()
