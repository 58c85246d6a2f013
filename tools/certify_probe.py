"""The c21 key certificates on the GPU: azb_certify_keys in trees per second (N = 19, 33, 64; random recursive trees,
the library's root generator, against sqrt(N - 1) + 1), with the share of each verdict; the same at N = 64 on trees near
the bound (the 27 618 classes azb_trees_within returns at the star's key, repeated to the same batch size); and the time
azb_trees_within_proof adds to azb_trees_within with the default bound (N = 26, 48, 64; plain and proof calls
alternated, each --reps times), with the proof words.  The card's name and power limit are recorded with the numbers.

    python tools/certify_probe.py --out DIR [--reps 3]   (writes DIR/certify_probe.json)
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from azdopt_b200 import capi  # noqa: E402
from within_probe import gpu_info  # noqa: E402


def certify_rate(n, m, reps, near=False):
    with capi.Handle(capi.default_config(n, 1)) as h:
        if near:
            cls = h.trees_within(k=65536)["parents"]
            parents = np.ascontiguousarray(np.resize(cls, (m, n)))
        else:
            parents = capi.generate_roots(n, 0, m, n)[0]
        h.certify_keys(parents[:1024])  # warm up
        ms = []
        for _ in range(reps):
            t0 = time.perf_counter()
            r = h.certify_keys(parents)
            ms.append(((time.perf_counter() - t0) * 1e3, r["ms"]))
        lam, _, _, cost_ms = h.eval_costs(parents)
    dev = min(d for _, d in ms)
    v = r["verdict"]
    return dict(n=n, trees=m, batch="trees_within classes at the star's key" if near else "random recursive",
                device_ms=dev, wall_ms=min(w for w, _ in ms), trees_per_s=m / dev * 1e3, cost_kernel_ms=cost_ms, verdicts={str(k): int(np.sum(v == k)) for k in (-1, 0, 1, 2)},
                enclosed=int(np.sum(np.isfinite(r["lambda1_lo"]))))


def proof_cost(n, reps):
    out = dict(n=n, plain_ms=[], proof_ms=[])
    with capi.Handle(capi.default_config(n, 1)) as h:
        h.trees_within(k=1)  # warm up
        for _ in range(reps):
            a = h.trees_within(k=100)
            b = h.trees_within(k=100, prove=True)
            out["plain_ms"].append(a["ms"])
            out["proof_ms"].append(b["ms"])
        assert (a["n_within"], a["n_below"]) == (b["n_within"], b["n_below"])
        out.update(n_within=b["n_within"], n_below=b["n_below"], proof=b["proof"],
                   added_ms=min(out["proof_ms"]) - min(out["plain_ms"]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--trees", type=int, default=1 << 20)
    ap.add_argument("--within-n", type=int, nargs="*", default=[26, 48, 64])
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    res = dict(gpu=gpu_info(), certify=[], proof=[])
    for n in (19, 33, 64):
        res["certify"].append(certify_rate(n, a.trees, a.reps))
        print(json.dumps(res["certify"][-1]), flush=True)
    res["certify"].append(certify_rate(64, a.trees, a.reps, near=True))
    print(json.dumps(res["certify"][-1]), flush=True)
    for n in a.within_n:
        res["proof"].append(proof_cost(n, a.reps))
        print(json.dumps(res["proof"][-1]), flush=True)
    with open(os.path.join(a.out, "certify_probe.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
