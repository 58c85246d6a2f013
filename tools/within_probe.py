"""azb_trees_within on the GPU: for each N and each bound (the star's key, + 0.5, + 1) the size of every level, the
children and distinct evaluations per level, the call's device time (host wall clock beside it), and the result's
counts; a configuration whose level outgrows --max-level is recorded as a capacity stop with the level it reached.  At
N = 26 it also times azb_exhaustive_best over the whole range, the other exact answer there.

    python tools/within_probe.py --out DIR [--n 26 32 40 48 64] [--max-level 2000000]   (writes DIR/within_probe.json)

With --gpus G it times azb_comm_trees_within instead: G ranks, one process and one GPU each, attached to one
communicator (--share-gpu: all on GPU 0, exchanging through host sockets, for the counts of G ranks without the
times).  Per level it records the global size, the largest and smallest rank share, the codes that crossed
between ranks (16 bytes each) and the slowest rank's time.  A case that runs past --time-limit seconds is stopped (its
ranks are terminated) and recorded with the levels it finished.  One JSON line per case is appended to
DIR/within_sharded.jsonl.

    python tools/within_probe.py --out DIR --gpus 8 --n 64 --offsets 0 0.5 1 --max-level 0 [--time-limit 600]
"""
import argparse
import json
import multiprocessing
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
RANK_LINE = re.compile(r"azb_comm_trees_within: N (\d+) level (\d+) rank (\d+): (\d+) classes owned, (\d+) global, (\d+) children, "
                       r"(\d+) codes sent, (\d+) received, (\d+) evaluated, ([\d.]+) ms")


def gpu_info(every=False):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    if q.returncode != 0:
        raise RuntimeError("nvidia-smi failed: no GPU to measure on")
    lines = q.stdout.strip().splitlines()
    return lines if every else lines[0]


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


def _rank(rank, world, n, offset, max_level, k, tmp, share_gpu):
    """One rank of a sharded case: its trace goes to tmp/trace<rank>.txt, its result to tmp/rank<rank>.json."""
    if share_gpu:  # every rank on GPU 0, each its own NCCL host so that NCCL accepts them (sockets over loopback)
        os.environ.update(NCCL_HOSTID=f"azb-rank-{rank}", NCCL_SOCKET_IFNAME="lo", NCCL_IB_DISABLE="1")
    fd = os.open(os.path.join(tmp, f"trace{rank}.txt"), os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
    os.dup2(fd, 2)
    path = os.path.join(tmp, "nccl_id")
    if rank == 0:
        with open(path + ".tmp", "wb") as f:
            f.write(capi.comm_unique_id())
        os.replace(path + ".tmp", path)
    while not os.path.exists(path):
        time.sleep(0.05)
    with capi.Handle(capi.default_config(n, 1, device=0 if share_gpu else rank)) as h:
        h.comm_init(open(path, "rb").read(), rank, world)
        lam, mu, _, _ = h.eval_costs(np.zeros((1, n), dtype=np.uint8))
        star_key = float(mu[0]) + float(lam[0])
        h.comm_trees_within(star_key - 0.5, k=1, max_level=max_level)  # warm-up: NCCL channels, modules, CUB, the slab
        res = dict(bound=star_key + offset)
        if world == 1:  # the local call beside it, same process and device
            t0 = time.perf_counter()
            try:
                r = h.trees_within(None if offset == 0.0 else star_key + offset, k=k, max_level=max_level)
                res.update(local_ms=round(r["ms"], 2), local_wall_s=round(time.perf_counter() - t0, 3))
            except capi.AzbError as e:
                res.update(local_error=str(e))
        os.environ["AZB_TRACE_WITHIN"] = "1"
        t0 = time.perf_counter()
        try:
            r = h.comm_trees_within(None if offset == 0.0 else star_key + offset, k=k, max_level=max_level)
            res.update(ms=round(r["ms"], 2), n_within=r["n_within"], n_below=r["n_below"],
                       best_key=float(r["mu"][0]) + float(r["lambda1"][0]) if len(r["mu"]) else None)
        except capi.AzbError as e:
            res.update(capacity=e.code == capi.ERR_CAPACITY, error=str(e))
        res.update(wall_s=round(time.perf_counter() - t0, 3), device_bytes=h.device_bytes())
    with open(os.path.join(tmp, f"rank{rank}.json"), "w") as f:
        json.dump(res, f)


def sharded_case(args, n, offset):
    """One azb_comm_trees_within case on args.gpus ranks: the ranks' results and the per-level table of their traces."""
    world = args.gpus
    with tempfile.TemporaryDirectory() as tmp:
        ctx = multiprocessing.get_context("spawn")
        procs = [ctx.Process(target=_rank, args=(r, world, n, offset, args.max_level, args.k, tmp, args.share_gpu)) for r in range(world)]
        for p in procs:
            p.start()
        deadline = time.monotonic() + args.time_limit
        for p in procs:
            p.join(max(0.0, deadline - time.monotonic()))
        stopped = any(p.is_alive() for p in procs)
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(10)
            if p.is_alive():
                p.kill()
                p.join()
        ranks = []
        for r in range(world):
            f = os.path.join(tmp, f"rank{r}.json")
            ranks.append(json.load(open(f)) if os.path.exists(f) else None)
        rows = {}
        for r in range(world):
            for m in map(RANK_LINE.match, open(os.path.join(tmp, f"trace{r}.txt")).read().splitlines()):
                if m:
                    rows.setdefault(int(m.group(2)), []).append([int(x) for x in m.groups()[3:9]] + [float(m.group(10))])
    levels = []
    for lv in sorted(rows):
        x = rows[lv]
        levels.append(dict(n=lv, ranks=len(x), classes=x[0][1], share_max=max(v[0] for v in x), share_min=min(v[0] for v in x),
                           children=sum(v[2] for v in x), sent=sum(v[3] for v in x), received=sum(v[4] for v in x),
                           evaluated=sum(v[5] for v in x), ms=max(v[6] for v in x)))
    case = dict(gpus=world, share_gpu=args.share_gpu, n=n, offset=offset, max_level=args.max_level, time_limit_s=args.time_limit, stopped=stopped,
                ranks=ranks, levels=levels, children=sum(x["children"] for x in levels), evaluated=sum(x["evaluated"] for x in levels),
                bytes_exchanged=16 * sum(x["sent"] for x in levels))
    return case


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for within_probe.json")
    ap.add_argument("--n", type=int, nargs="+", default=[26, 32, 40, 48, 64])
    ap.add_argument("--offsets", type=float, nargs="+", default=[0.0, 0.5, 1.0], help="bounds: the star's key + offset")
    ap.add_argument("--max-level", type=int, default=2_000_000)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--gpus", type=int, default=0, help="time azb_comm_trees_within on this many ranks (0: azb_trees_within)")
    ap.add_argument("--time-limit", type=float, default=600.0, help="--gpus: seconds before a case's ranks are stopped")
    ap.add_argument("--share-gpu", action="store_true",
                    help="--gpus: every rank on GPU 0 (level shares and codes exchanged are those of G GPUs, times are not)")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    if args.gpus:
        card = gpu_info(every=True)[:1 if args.share_gpu else args.gpus]
        for n in args.n:
            for off in args.offsets:
                case = dict(card=card, **sharded_case(args, n, off))
                print(json.dumps({k: v for k, v in case.items() if k not in ("levels", "ranks")} | dict(rank0=case["ranks"][0])),
                      flush=True)
                with open(os.path.join(args.out, "within_sharded.jsonl"), "a") as f:
                    f.write(json.dumps(case) + "\n")
        return
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
