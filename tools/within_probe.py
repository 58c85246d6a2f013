"""azb_trees_within on the GPU: for each N and each bound (the star's key, + 0.5, + 1) the size of every level, the
children and distinct evaluations per level, the call's device time (host wall clock beside it), and the result's
counts; a configuration whose level outgrows --max-level is recorded as a capacity stop with the level it reached.  At
N = 26 it also times azb_exhaustive_best over the whole range, the other exact answer there.

    python tools/within_probe.py --out DIR [--n 26 32 40 48 64] [--max-level 2000000]   (writes DIR/within_probe.json)
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from azdopt_b200 import capi  # noqa: E402

LINE = re.compile(r"azb_trees_within: N (\d+) level (\d+): (\d+) classes, (\d+) children, (\d+) evaluated, ([\d.]+) ms")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    if q.returncode != 0:
        raise RuntimeError("nvidia-smi failed: no GPU to measure on")
    return q.stdout.strip().splitlines()[0]


def traced(call):
    """call() with the library's per-level trace (AZB_TRACE_WITHIN, written to stderr) captured: (result, levels)."""
    os.environ["AZB_TRACE_WITHIN"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tmp:
        os.dup2(tmp.fileno(), 2)
        try:
            res = call()
        except capi.AzbError as e:
            res = e
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["AZB_TRACE_WITHIN"]
        tmp.seek(0)
        levels = [dict(n=int(m.group(2)), classes=int(m.group(3)), children=int(m.group(4)), evaluated=int(m.group(5)),
                       ms=float(m.group(6))) for m in map(LINE.match, tmp.read().splitlines()) if m]
    return res, levels


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for within_probe.json")
    ap.add_argument("--n", type=int, nargs="+", default=[26, 32, 40, 48, 64])
    ap.add_argument("--offsets", type=float, nargs="+", default=[0.0, 0.5, 1.0], help="bounds: the star's key + offset")
    ap.add_argument("--max-level", type=int, default=2_000_000)
    ap.add_argument("--k", type=int, default=100)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    res = dict(card=gpu_info(), max_level=args.max_level, cases=[])
    for n in args.n:
        with capi.Handle(capi.default_config(n, 1)) as h:
            lam, mu, _, _ = h.eval_costs(np.zeros((1, n), dtype=np.uint8))  # the star, the default bound
            star_key = float(mu[0]) + float(lam[0])
            h.trees_within(star_key - 0.5, k=1, max_level=args.max_level)  # warm-up: modules, CUB, the slab
            for off in args.offsets:
                bound = None if off == 0.0 else star_key + off
                t0 = time.perf_counter()
                r, levels = traced(lambda: h.trees_within(bound, k=args.k, max_level=args.max_level))
                wall = time.perf_counter() - t0
                case = dict(n=n, offset=off, bound=star_key + off, wall_s=round(wall, 3),
                            levels=levels, children=sum(x["children"] for x in levels),
                            evaluated=sum(x["evaluated"] for x in levels), device_bytes=h.device_bytes())
                if isinstance(r, capi.AzbError):
                    case.update(capacity=r.code == capi.ERR_CAPACITY, error=str(r))
                else:
                    case.update(ms=round(r["ms"], 2), n_within=r["n_within"], n_below=r["n_below"],
                                best_key=float(r["mu"][0]) + float(r["lambda1"][0]) if len(r["mu"]) else None,
                                best_parents=r["parents"][0].tolist() if len(r["mu"]) else None)
                print(json.dumps({k: v for k, v in case.items() if k != "levels"}), flush=True)
                res["cases"].append(case)
            if n == 26:
                h.exhaustive_best(0, 1 << 20, k=100)
                t0 = time.perf_counter()
                ex = h.exhaustive_best(k=100)
                res["exhaustive_26"] = dict(ms=round(ex["ms"], 2), wall_s=round(time.perf_counter() - t0, 3),
                                            n_below=ex["n_below"])
                print(json.dumps(res["exhaustive_26"]), flush=True)
    with open(os.path.join(args.out, "within_probe.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
