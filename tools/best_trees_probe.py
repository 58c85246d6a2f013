"""Cost of azb_best_trees at the search's own shapes: N = 19 after 800 steps at 4096 and 16 384 roots, N = 64 after
200 steps at 1024 roots, k = 1, 100 and 10 000 each, on the example's workload (device MLP on tensor cores, the
library's default step layout).
usage: python tools/best_trees_probe.py [out.jsonl]     prints the card, then one JSON line per (shape, k)
Per line: the epoch's search time (azb_step_timed, device events), the call's device time (torch.profiler: the sum of
the kernels one call launches, and the span from the first kernel's start to the last one's end), the whole C-ABI call
(host clock around the synchronous call, median of 5), and the selection rounds and candidates, replayed on the host
from the tree dumps (node costs) and azb_tree_codes with the library's rule (first M = 4k, then twice the candidates)."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from azdopt_b200 import build, capi  # noqa: E402
from best_trees_util import replay  # noqa: E402

SHAPES = [(19, 4096, 800), (19, 16384, 800), (64, 1024, 200)]
KS = (1, 100, 10000)


def f2ord(bits):
    bits = bits.astype(np.uint64)
    return np.where(bits & 0x80000000, (~bits) & 0xFFFFFFFF, bits | 0x80000000)


def rounds(h, k, dumps):
    """(rounds, candidates of the last round, classes found, nodes) of the selection for k, from dumps + azb_tree_codes."""
    roots_p, roots_m = h.get_roots()
    ords, where = [], []
    for t, d in enumerate(dumps):
        o = f2ord(d["nodes"][:, 0])
        ords.append(o)
        where.extend((t, i) for i in range(len(o)))
    ords = np.concatenate(ords)
    srt = np.sort(ords)
    total, m, r = len(ords), 4 * k, 0
    while True:
        r += 1
        thr = srt[min(m, total) - 1]
        sel = np.nonzero(ords <= thr)[0]
        par = np.stack([replay(roots_p[where[j][0]], roots_m[where[j][0]], dumps[where[j][0]]["keys"][where[j][1]], h.n)[0]
                        for j in sel])
        n_cls = len({tuple(c) for c in h.tree_codes(par).tolist()})
        if n_cls >= k or len(sel) >= total:
            return r, int(len(sel)), n_cls, total
        m = 2 * len(sel)


def device_ms(h, k):
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        h.best_trees(k)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.device_time_total > 0
          and not e.name.startswith("Memcpy") and not e.name.startswith("Memset")]
    busy = sum(e.device_time_total for e in ev) / 1e3
    span = (max(e.time_range.end for e in ev) - min(e.time_range.start for e in ev)) / 1e3 if ev else 0.0
    return busy, span, len(ev)


def main():
    build()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print(card, flush=True)
    out = open(sys.argv[1], "w") if len(sys.argv) > 1 else None
    for n, b, steps in SHAPES:
        cfg = capi.default_config(n, b, prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, max_steps=steps,
                                  async_workers=capi.ASYNC_AUTO)
        with capi.Handle(cfg) as h:
            h.mlp_init(1)
            h.set_roots(*capi.generate_roots(0, 0, b, n))
            h.init_trees()
            search_ms, _ = h.step_timed(steps)
            dumps = [h.dump_tree(t) for t in range(h.b)]
            for k in KS:
                h.best_trees(k)  # warm: slab growth, first launches
                try:
                    busy, span, n_kernels = device_ms(h, k)
                except Exception as e:  # the profiler is a measurement aid; the other figures still stand
                    print("profiler:", e, flush=True)
                    busy = span = n_kernels = None
                walls = []
                for _ in range(5):
                    t0 = time.perf_counter()
                    res = h.best_trees(k)
                    walls.append((time.perf_counter() - t0) * 1e3)
                r, cand, n_cls, total = rounds(h, k, dumps)
                rec = dict(card=card, n=n, roots=b, steps=steps, k=k, returned=int(len(res["eval"])), nodes=total,
                           rounds=r, candidates=cand, classes_found=n_cls, search_ms=round(search_ms, 2),
                           device_kernel_ms=busy and round(busy, 3), device_span_ms=span and round(span, 3), kernels=n_kernels,
                           call_ms=round(float(np.median(walls)), 3), device_bytes=h.device_bytes())
                print(json.dumps(rec), flush=True)
                if out:
                    out.write(json.dumps(rec) + "\n")
                    out.flush()
    return 0


if __name__ == "__main__":
    sys.exit(main())
