"""PUCT selection (azb_config.selection = AZB_SELECT_PUCT) against the reference's next_action: simulations/s of K timed
steps, the two modes alternating on the same roots, for the one-launch hash mode (N = 19 at 4096 and 65 536 roots,
N = 64 at 4096 roots) and the asynchronous kernel with the tensor-core model (N = 19, 4096 roots).

    python tools/puct_probe.py [--steps K] [--reps R] [--c-puct C]

Prints the card's name and power limit, one line per timed run, and a JSON summary (median per mode and shape).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from azdopt_b200 import capi  # noqa: E402

SHAPES = [  # (name, N, roots, config)
    ("hash_n19_b4096", 19, 4096, dict(prior_mode=capi.PRIOR_HASH)),
    ("hash_n19_b65536", 19, 65536, dict(prior_mode=capi.PRIOR_HASH)),
    ("async_tc_n19_b4096", 19, 4096, dict(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, async_workers=capi.ASYNC_AUTO)),
    ("hash_n64_b4096", 64, 4096, dict(prior_mode=capi.PRIOR_HASH)),
]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.TimeoutExpired):
        return "unknown"


def run(n, b, kw, selection, c_puct, steps, warmup):
    parents, masks = capi.generate_roots(0, 0, b, n)
    cfg = capi.default_config(n, b, max_steps=steps + warmup + 8, selection=selection, puct_c=c_puct, **kw)
    with capi.Handle(cfg) as h:
        h.set_counter_mode(False)
        if kw.get("prior_mode") == capi.PRIOR_MLP:
            h.mlp_init(1)
        h.set_roots(parents, masks)
        h.init_trees()
        h.step(warmup)
        h.reset_counters()
        ms, _ = h.step_timed(steps)
        live = h.counters()["n_live"]
        return live / (ms * 1e-3), ms, h.argmin()["eval"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--c-puct", type=float, default=1.0)
    ap.add_argument("--only", default="", help="comma-separated shape names")
    a = ap.parse_args()
    print(f"card: {card()}", flush=True)
    shapes = [s for s in SHAPES if not a.only or s[0] in a.only.split(",")]
    res = {}
    for name, n, b, kw in shapes:
        for rep in range(a.reps):
            for sel in (capi.SELECT_REFERENCE, capi.SELECT_PUCT):
                sims, ms, best = run(n, b, kw, sel, a.c_puct, a.steps, a.warmup)
                mode = "puct" if sel else "reference"
                res.setdefault(name, {}).setdefault(mode, []).append(sims)
                print(f"{name:22s} rep {rep} {mode:9s}: {ms:9.2f} ms for {a.steps} steps  {sims / 1e6:8.3f} M sims/s  "
                      f"argmin {best:.5f}", flush=True)
    summary = {name: {mode: statistics.median(v) for mode, v in d.items()} for name, d in res.items()}
    for name, d in summary.items():
        d["puct_over_reference"] = d["puct"] / d["reference"]
    print(json.dumps(dict(card=card(), steps=a.steps, reps=a.reps, c_puct=a.c_puct, median_sims_per_s=summary)))


if __name__ == "__main__":
    main()
