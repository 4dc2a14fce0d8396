"""The 2^30-row switch-overs of stream compaction and the radix sort, and the documented size limits.

Below 2^30 rows both primitives chain 30-bit running counts through decoupled look-back words in one kernel; from
2^30 on they run count / scan / scatter kernels with 32-bit offsets (csrc/gsx_compact.cu, csrc/gsx_radix.cu).

(a) At real size (n > 2^30) on the shipped library: every output element is checked against a closed formula; nothing
    is sorted or nonzero()-ed at that size, and the checks run on the device in chunks of 2^26 elements.
(b) The fallback forms at ordinary sizes: the existing exact checks (torch's stable sort, the SOR oracle, NumPy
    lexsort, the Morton restatement, SciPy, NumPy boolean indexing) rerun in a subprocess against builds whose
    switch-over is 4096 rows.
(c) CPU: the workspace-size functions accept the largest documented n and refuse the next one.
"""
import ctypes as C
import json
import os
import re
import subprocess
import sys
import time
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
GIB = 1 << 30
CHUNK = 1 << 26
N_LIMIT = 2**31 - 64            # gsx.h: every point count n < 2^31 - 64
SWITCH = 4096                   # switch-over of the test builds


# ------------------------------------------------------------------ (c) documented limits, host calls only
def test_header_states_the_limit():
    src = (ROOT / "include" / "gsx.h").read_text()
    m = re.search(r"#define\s+GSX_N_LIMIT\s+(\d+)LL", src)
    assert m and int(m.group(1)) == N_LIMIT
    assert "N < 2^31 - 64" in src


@pytest.mark.parametrize("fn", ["gsx_sor_workspace_bytes", "gsx_sor_grid_workspace_bytes",
                                "gsx_compact_workspace_bytes", "gsx_lexsort_workspace_bytes",
                                "gsx_morton_workspace_bytes", "gsx_knn_exact_workspace_bytes"])
def test_workspace_sizes_pin_the_point_limit(fn, gsx_lib):
    f = getattr(gsx_lib, fn)
    assert f(N_LIMIT - 1) > 0
    assert f(N_LIMIT) < 0 and b"out of range" in gsx_lib.gsx_last_error()
    assert f(1 << 40) < 0
    assert f(1) > 0


def test_sort_pairs_workspace_size_pins_its_limit(gsx_lib):
    """gsx_sort_pairs is a generic primitive: 1 <= n < 2^32 (32-bit offsets of the three-kernel passes)."""
    f = gsx_lib.gsx_sort_pairs_workspace_bytes
    assert f(2**32 - 1) > 0
    assert f(2**32) < 0 and b"out of range" in gsx_lib.gsx_last_error()
    assert f(N_LIMIT) > 0


def test_python_wrappers_raise_on_refused_sizes(gsx_lib):
    from gsx import GsxError
    from gsx._abi import workspace_size
    with pytest.raises(GsxError, match="out of range"):
        workspace_size("gsx_compact_workspace_bytes", N_LIMIT)
    assert workspace_size("gsx_compact_workspace_bytes", N_LIMIT - 1) > 0


# ------------------------------------------------------------------ (a) at size, shipped library
def _need(nbytes, what):
    import torch
    free, _ = torch.cuda.mem_get_info()
    want = nbytes + 8 * GIB
    if free < want:
        pytest.skip(f"{what}: needs {want / GIB:.1f} GiB free on the device ({nbytes / GIB:.1f} GiB + 8 GiB margin), "
                    f"has {free / GIB:.1f} GiB: short by {(want - free) / GIB:.1f} GiB")


def _chunks(n):
    for a in range(0, n, CHUNK):
        yield a, min(n, a + CHUNK)


def _free():
    import gc
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _xyz_of(i):
    """Row number -> coordinates, exact in float32 for i < 2^31."""
    import torch
    return torch.stack(((i & ((1 << 23) - 1)).float(), (i >> 23).float(), (i % 7).float()), 1)


def _opacity_of(i):
    return (((i * 5) & ((1 << 24) - 1)) - (1 << 23)).float()


# keep row i  <=>  (i mod P) >= D  and  i < L.  Survivor j is row (j // Q) * P + D + j mod Q with Q = P - D, and L is
# chosen so that exactly `count` rows survive.  P is prime: the dropped rows fall at every offset of the 2048-row
# tiles and 1024-row blocks.
COMPACT_N = (1 << 30) + (1 << 20) + 7
COMPACT_CASES = [((1 << 30) - 1, 3001, 2), (1 << 30, 4099, 3), ((1 << 30) + (1 << 19), 8191, 1)]


def _cut(count, P, D):
    Q = P - D
    return (count // Q) * P + (D + count % Q if count % Q else 0)


@pytest.mark.gpu
@pytest.mark.parametrize("with_opacity", [True, False], ids=["opacity", "no_opacity"])
def test_compact_at_size(with_opacity, cuda, gsx_lib):
    """n = 2^30 + 2^20 + 7 rows; exactly 2^30 - 1, 2^30 and 2^30 + 2^19 survivors."""
    import torch
    from gsx.pipeline import compact
    n = COMPACT_N
    _need(n * (1 + 12 + 12 + 4 + (8 if with_opacity else 0)) + 2 * GIB, "compact at size")
    t0 = time.perf_counter()
    xyz = torch.empty((n, 3), dtype=torch.float32, device=cuda)
    opacity = torch.empty(n, dtype=torch.float32, device=cuda) if with_opacity else None
    mask = torch.empty(n, dtype=torch.bool, device=cuda)
    for a, b in _chunks(n):
        i = torch.arange(a, b, dtype=torch.int64, device=cuda)
        xyz[a:b] = _xyz_of(i)
        if with_opacity:
            opacity[a:b] = _opacity_of(i)
    for count, P, D in COMPACT_CASES:
        L = _cut(count, P, D)
        assert L <= n
        for a, b in _chunks(n):
            i = torch.arange(a, b, dtype=torch.int64, device=cuda)
            mask[a:b] = ((i % P) >= D) & (i < L)
        x_o, o_o, idx_o, m = compact(mask, xyz, opacity, None)
        assert m == count, f"survivors: got {m}, want {count}"
        Q = P - D
        for a, b in _chunks(m):
            j = torch.arange(a, b, dtype=torch.int64, device=cuda)
            i = (j // Q) * P + D + j % Q
            assert torch.equal(idx_o[a:b], i.to(torch.int32)), f"idx_out wrong in [{a}, {b}) of {count} survivors"
            assert torch.equal(x_o[a:b], _xyz_of(i)), f"xyz_out wrong in [{a}, {b}) of {count} survivors"
            if with_opacity:
                assert torch.equal(o_o[a:b], _opacity_of(i)), f"opacity_out wrong in [{a}, {b}) of {count} survivors"
        assert (o_o is None) == (not with_opacity)
        del x_o, o_o, idx_o
        _free()
    print(f"\ncompact at size ({'with' if with_opacity else 'without'} opacity, n={n}, 3 masks): "
          f"{time.perf_counter() - t0:.1f} s")
    del xyz, opacity, mask
    _free()


SORT_N = (1 << 30) + 4097


def _block_order(p, n, B):
    """Rows in blocks of B equal keys whose key DEcreases with the block: the stable ascending order is the blocks
    reversed (the short last block first), ascending rows inside each block.  Output position p -> row."""
    import torch
    nb = (n + B - 1) // B
    s = n - (nb - 1) * B
    q = p - s
    return torch.where(p < s, (nb - 1) * B + p, (nb - 2 - q // B) * B + q % B)


def _pair_key(i, n, B):
    nb = (n + B - 1) // B
    field = nb - 1 - i // B                                     # bits [5, 29): the sorted field, 3 digit passes
    hi = (i * 2654435761) & 0x7FFFFFFF                          # bits [32, 63): above end_bit, carried along
    lo = ((i * 40503) >> 3) & 31                                # bits [0, 5): below begin_bit, must be ignored
    return (hi << 32) | (field << 5) | lo


@pytest.mark.gpu
def test_sort_pairs_at_size(cuda, gsx_lib):
    import torch
    from gsx import sor
    n, B = SORT_N, 1000
    _need(gsx_lib.gsx_sort_pairs_workspace_bytes(n) + 12 * n + 2 * GIB, "sort_pairs at size")
    t0 = time.perf_counter()
    keys = torch.empty(n, dtype=torch.int64, device=cuda)
    vals = torch.empty(n, dtype=torch.int32, device=cuda)
    for a, b in _chunks(n):
        i = torch.arange(a, b, dtype=torch.int64, device=cuda)
        keys[a:b] = _pair_key(i, n, B)
        vals[a:b] = i.to(torch.int32)
    sor.sort_pairs(keys, vals, 5, 29)
    for a, b in _chunks(n):
        i = _block_order(torch.arange(a, b, dtype=torch.int64, device=cuda), n, B)
        assert torch.equal(vals[a:b], i.to(torch.int32)), f"values out of order in [{a}, {b})"
        assert torch.equal(keys[a:b], _pair_key(i, n, B)), f"keys wrong in [{a}, {b})"
    print(f"\nsort_pairs at size (n={n}): {time.perf_counter() - t0:.1f} s")
    del keys, vals
    _free()


@pytest.mark.gpu
def test_sort_keys_only_at_size(cuda, gsx_lib):
    """vals=None: the packed words of the grid build (row number below begin_bit), n >= 2^30."""
    import torch
    from gsx import sor
    n, B = SORT_N, 777
    nb = (n + B - 1) // B

    def word(i):
        return ((((i * 2654435761) >> 11) & 0xFF) << 55) | ((nb - 1 - i // B) << 31) | i

    _need(gsx_lib.gsx_sort_pairs_workspace_bytes(n) + 8 * n + 2 * GIB, "keys-only sort at size")
    t0 = time.perf_counter()
    words = torch.empty(n, dtype=torch.int64, device=cuda)
    for a, b in _chunks(n):
        words[a:b] = word(torch.arange(a, b, dtype=torch.int64, device=cuda))
    sor.sort_pairs(words, None, 31, 55)
    for a, b in _chunks(n):
        i = _block_order(torch.arange(a, b, dtype=torch.int64, device=cuda), n, B)
        assert torch.equal(words[a:b], word(i)), f"words out of order in [{a}, {b})"
    print(f"\nkeys-only sort at size (n={n}): {time.perf_counter() - t0:.1f} s")
    del words
    _free()


# ------------------------------------------------------------------ (b) fallback forms at ordinary sizes
VARIANTS = {
    "radix": ("gsx_radix.cu", f"-DGSX_RADIX_ONESWEEP_MAX_N={SWITCH}"),
    "compact": ("gsx_compact.cu", f"-DGSX_COMPACT_ONEPASS_MAX_N={SWITCH}"),
}


@pytest.fixture(scope="session")
def switch_variants(gsx_lib, tmp_path_factory):
    """libgsx.so builds whose radix sort / compaction switch to the >= 2^30 form at 4096 rows (built in a temporary
    directory with scripts/build_variants.sh; nvcc is all they need)."""
    out = tmp_path_factory.mktemp("gsx_variants")
    env = dict(os.environ, GSX_VARIANT_DIR=str(out))
    env.pop("CC", None)
    libs = {}
    for name, (tu, flags) in VARIANTS.items():
        subprocess.run(["bash", str(ROOT / "scripts" / "build_variants.sh"), tu, f"sw{name}:{flags}"], env=env,
                       check=True, capture_output=True, text=True, timeout=600)
        libs[name] = out / f"libgsx_sw{name}.so"
        assert libs[name].exists()
    return libs


def _run_py(lib, code):
    env = dict(os.environ, GSX_LIB=str(lib))
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


# kernel launches of one sort (2 digit passes) and one compaction at n rows, and which library answered
_LAUNCHES = """
import json, sys
sys.path[:0] = ['.', '3dgsconverter_b200']
import torch
from gsx import _abi, sor
from gsx.pipeline import compact
lib, dev, out = _abi.lib, torch.device('cuda:0'), {'lib': str(_abi.LIB_PATH)}
for n in (4095, 4096):
    keys = torch.arange(n, 0, -1, dtype=torch.int64, device=dev)
    c0 = lib.gsx_kernel_launches(); sor.sort_pairs(keys.clone(), torch.arange(n, dtype=torch.int32, device=dev), 0, 16)
    c1 = lib.gsx_kernel_launches(); sor.sort_pairs(keys.clone(), None, 0, 16)
    c2 = lib.gsx_kernel_launches(); compact(torch.ones(n, dtype=torch.bool, device=dev), torch.zeros((n, 3), device=dev), None, None)
    c3 = lib.gsx_kernel_launches()
    out[n] = [c1 - c0, c2 - c1, c3 - c2]
print(json.dumps(out))
"""


@pytest.mark.gpu
def test_switch_variants_take_the_fallback(switch_variants, cuda, gsx_lib):
    """The shipped library runs the one-kernel forms at 4095 and 4096 rows; each test build changes form exactly at
    4096 (more kernels: histogram / scan / scatter per digit, count / scan / scatter)."""
    from gsx import _abi
    shipped = _run_py(_abi.LIB_PATH, _LAUNCHES)
    assert shipped["4095"] == shipped["4096"]
    radix = _run_py(switch_variants["radix"], _LAUNCHES)
    assert radix["lib"] == str(switch_variants["radix"])
    assert radix["4095"] == shipped["4095"]
    assert radix["4096"][0] > shipped["4096"][0] and radix["4096"][1] > shipped["4096"][1]
    assert radix["4096"][2] == shipped["4096"][2]
    comp = _run_py(switch_variants["compact"], _LAUNCHES)
    assert comp["4095"] == shipped["4095"]
    assert comp["4096"][:2] == shipped["4096"][:2] and comp["4096"][2] > shipped["4096"][2]


_SOR_IDS = [f"tests/test_sor_gpu.py::test_sor_matches_oracle[100000-{k}-{mode}-mixed]"
            for k in (16, 27) for mode in ("i32wrap", "i64")]
SUITES = {
    "radix-sort": ("radix", ["tests/test_radix_sort_gpu.py"]),
    "radix-sor": ("radix", _SOR_IDS + ["tests/test_sor_gpu.py::test_sor_edge_cases"]),
    "radix-lexsort-morton-ckdtree": ("radix", [
        "tests/test_sog_helpers_gpu.py::test_lexsort_matches_numpy",
        "tests/test_morton_gpu.py::test_morton_order_matches_reference_algorithm",
        "tests/test_morton_gpu.py::test_morton_degenerate_clouds",
        "tests/test_sor_ckdtree_gpu.py::test_ckdtree_edge_cases"]),
    "compact": ("compact", [
        "tests/test_dropin_api_gpu.py::test_compact_points_matches_numpy",
        "tests/test_dropin_api_gpu.py::test_compact_points_unaligned_mask_and_chained_index"]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("suite", list(SUITES))
def test_existing_checks_on_switch_variant(suite, switch_variants, cuda):
    variant, ids = SUITES[suite]
    env = dict(os.environ, GSX_LIB=str(switch_variants[variant]))
    r = subprocess.run([sys.executable, "-m", "pytest", "-p", "no:cacheprovider", "-q", "-m", "gpu", *ids], cwd=ROOT,
                       env=env, capture_output=True, text=True, timeout=560)
    tail = (r.stdout + r.stderr)[-4000:]
    assert r.returncode == 0, tail
    assert re.search(r"\d+ passed", tail) and "skipped" not in tail and "deselected" not in tail, tail
