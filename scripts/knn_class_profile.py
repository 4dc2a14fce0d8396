"""Where the SOR query kernel's cycles go, by the size of the centre probe's bucket (the query's own bucket).

    scripts/build_variants.sh gsx_sor.cu prof:"-DGSX_KNN_PROFILE=1" prof_nogroup:"-DGSX_KNN_PROFILE=1 -DGSX_KNN_GROUP=0"
    GSX_LIB=3dgsconverter_b200/lib/variants/libgsx_prof.so python scripts/knn_class_profile.py [--n 10000000] [--out F]

Needs a library built with -DGSX_KNN_PROFILE=1: lane 0 of every 16-query batch adds the clock64 cycles of the batch
and its query count to one of 4 classes by the centre bucket's size (taken at the batch's first query).  Prints one
JSON object per cloud (the bench's `mixed` cloud, k = 16, i32wrap, and the uniform cloud): per class the share of the
queries, the share of the summed cycles and the mean cycles per query.  The cycles are summed over all warps, so they
weigh the classes against each other; they are not a kernel time."""
import argparse
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "3dgsconverter_b200")]

CLASSES = ("<=64", "<=1024", "<=16384", ">16384")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10_000_000)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from gsx import _abi, sor, synth
    info = _abi.lib.gsx_build_info().decode()
    if "profile=1" not in info:
        sys.exit(f"knn_class_profile: {_abi.LIB_PATH} was not built with -DGSX_KNN_PROFILE=1 ({info})")
    res = {"lib": Path(str(_abi.LIB_PATH)).name, "build_info": info, "n": a.n, "k": a.k, "hash": "i32wrap",
           "gpu": torch.cuda.get_device_name(0), "clouds": {}}
    for kind in ("mixed", "uniform"):
        x = torch.from_numpy(synth.xyz(a.n, kind)).cuda()
        ws = sor.workspace(a.n, x.device)
        grid = sor.build_grid(x, ws)
        sor.mean_dists(grid, a.k, "i32wrap")   # warm-up
        _, st = sor.mean_dists(grid, a.k, "i32wrap", want_stats=True)
        cyc, qs = st["class_cycles"], st["class_queries"]
        tc, tq = max(sum(cyc), 1), max(sum(qs), 1)
        res["clouds"][kind] = {
            "queries": st["queries"], "group_queries": st["group_queries"],
            "classes": {c: {"query_share": round(qs[i] / tq, 4), "cycle_share": round(cyc[i] / tc, 4),
                            "cycles_per_query": round(cyc[i] / qs[i], 1) if qs[i] else None}
                        for i, c in enumerate(CLASSES)},
            "long_bucket_cycle_share": round(sum(cyc[1:]) / tc, 4)}
        del x, ws, grid
        print(kind, json.dumps(res["clouds"][kind]), flush=True)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
