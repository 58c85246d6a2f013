"""Exhaustive ranking rate on the GPU: trees per second of azb_exhaustive_best over the whole enumeration at each N (the
device time the call reports, host wall clock beside it), k = 100 against k = 65 536, the one-off table build, and the
optimum with the number of trees below the star's key sqrt(N - 1) + 1; at N = 30 and 32 only the table build.

    python tools/exhaustive_probe.py --out DIR [--n 19 22 23 24 26]      (writes DIR/exhaustive_probe.json)
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from azdopt_b200 import capi  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    if q.returncode != 0:
        raise RuntimeError("nvidia-smi failed: no GPU to measure on")
    return q.stdout.strip().splitlines()[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for exhaustive_probe.json")
    ap.add_argument("--n", type=int, nargs="+", default=[19, 22, 23, 24, 26])
    ap.add_argument("--ks", type=int, nargs="+", default=[100, 65536])
    ap.add_argument("--tables-only", type=int, nargs="*", default=[30, 32],
                    help="sizes whose table build is timed without ranking the whole range")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    res = dict(card=gpu_info(), cases=[])
    for n in args.n:
        total = capi.free_tree_count(n)
        with capi.Handle(capi.default_config(n, 1)) as h:
            t0 = time.perf_counter()
            h.free_trees(0, 1)  # builds and uploads the tables
            tables_s = time.perf_counter() - t0
            h.exhaustive_best(0, min(total, 1 << 20), k=100)  # warm-up: modules, CUB, the slab
            case = dict(n=n, trees=total, tables_s=round(tables_s, 3), device_bytes=h.device_bytes(), runs=[])
            for k in args.ks:
                t0 = time.perf_counter()
                r = h.exhaustive_best(k=k)
                wall = time.perf_counter() - t0
                case["runs"].append(dict(k=k, ms=round(r["ms"], 2), wall_s=round(wall, 3),
                                         trees_per_s=round(total / (r["ms"] * 1e-3)), n_below=r["n_below"]))
            best = r
            case.update(best_index=int(best["index"][0]), best_parents=best["parents"][0].tolist(),
                        best_key=float(best["mu"][0]) + float(best["lambda1"][0]), best_eval=float(best["eval"][0]),
                        star_key=math.sqrt(n - 1) + 1)
            print(json.dumps(case), flush=True)
            res["cases"].append(case)
    res["tables"] = []
    for n in args.tables_only:
        with capi.Handle(capi.default_config(n, 1)) as h:
            before = h.device_bytes()
            t0 = time.perf_counter()
            h.free_trees(0, 1)
            rec = dict(n=n, tables_s=round(time.perf_counter() - t0, 3), first_call_bytes=h.device_bytes() - before)
        print(json.dumps(rec), flush=True)
        res["tables"].append(rec)
    with open(os.path.join(args.out, "exhaustive_probe.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
