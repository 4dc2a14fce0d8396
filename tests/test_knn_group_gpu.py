"""GPU: the group path of the SOR query kernel (GSX_KNN_GROUP) returns the same bits as the per-query walk.

Two extra builds of gsx_sor.cu go to a temporary directory: one without the group path and one whose list holds only
2 entries, so that almost every group batch overflows and falls back to the per-query path.  The mean distances of
both must equal the shipped build's bit for bit on three clouds, both hash modes, k in {1, 7, 16, 27}.  A launch with
stats confirms that the shipped build really answers queries through the group path."""
import hashlib
import json
import os
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
pytestmark = pytest.mark.gpu

VARIANTS = {"nogroup": "-DGSX_KNN_GROUP=0", "list2": "-DGSX_KNN_GROUP_LIST=2"}

_MEANS = r"""
import hashlib, json, sys
sys.path[:0] = ['.', '3dgsconverter_b200']
import numpy as np, torch
from gsx import _abi, sor, synth
out = {'build_info': _abi.lib.gsx_build_info().decode(), 'digests': {}, 'group_queries': {}}
for kind in ('mixed', 'uniform', 'clustered'):
    x = torch.from_numpy(synth.xyz(300_000, kind)).cuda()
    ws = sor.workspace(len(x), x.device)
    grid = sor.build_grid(x, ws)
    for mode in ('i32wrap', 'i64'):
        for k in (1, 7, 16, 27):
            m, st = sor.mean_dists(grid, k, mode, want_stats=True)
            key = f'{kind}/{mode}/{k}'
            out['digests'][key] = hashlib.sha256(m.cpu().numpy().tobytes()).hexdigest()
            out['group_queries'][key] = st['group_queries']
print(json.dumps(out))
"""


@pytest.fixture(scope="module")
def variant_libs(tmp_path_factory):
    out = tmp_path_factory.mktemp("knn_group_variants")
    env = dict(os.environ, GSX_VARIANT_DIR=str(out))
    env.pop("CC", None)
    libs = {}
    for name, flags in VARIANTS.items():
        subprocess.run(["bash", str(ROOT / "scripts" / "build_variants.sh"), "gsx_sor.cu", f"{name}:{flags}"], env=env,
                       check=True, capture_output=True, text=True, timeout=900)
        libs[name] = out / f"libgsx_{name}.so"
        assert libs[name].exists()
    return libs


def _means(lib=None):
    env = dict(os.environ)
    if lib is not None:
        env["GSX_LIB"] = str(lib)
    r = subprocess.run([sys.executable, "-c", _MEANS], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_group_path_is_bit_identical_to_the_per_query_walk(variant_libs, gsx_lib):
    shipped = _means()
    assert "group=1" in shipped["build_info"], shipped["build_info"]
    # the group path really runs on the clustered parts, at every k <= 32 (K > 32 keeps the per-query walk only)
    for key, gq in shipped["group_queries"].items():
        if not key.startswith("uniform"):
            assert gq > 0, (key, gq)
    for name, lib in variant_libs.items():
        got = _means(lib)
        assert got["digests"] == shipped["digests"], name
        if name == "nogroup":
            assert "group=0" in got["build_info"] and not any(got["group_queries"].values())
        else:   # a 2-entry list overflows in most batches, so far fewer queries take the group path
            assert sum(got["group_queries"].values()) < sum(shipped["group_queries"].values()) // 2
