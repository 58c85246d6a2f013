#!/usr/bin/env python
"""bench.py — MCTS simulations/sec of the batched c21 search step (BASELINE.json's metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one NablaOptimizer::par_roll_out_episodes over the whole batch of roots
(az-discrete-opt/src/nabla/optimizer/mod.rs:121-191): walks + pack + MLP forward + add_actions + argmin.
One simulation = one root advanced by one step that ended on a newly expanded node; exhausted-root no-ops are
counted separately and excluded.  Workload at N GPUs: `--roots` (4096, BASELINE configs[1]) roots PER GPU,
N = 19, random-init MLP 304-512-1024-512-152, synthetic roots of the example's distribution (weak scaling; roots
shard across ranks with no collective inside a step).

torch is used here only for torch.distributed (NCCL process group: barrier, max/sum over ranks, the broadcast of the
library's communicator id) and torch.cuda.synchronize — the product is libazb.so.

Extra objects in the JSON line (VERDICT round 1, item 7): `same_priors` (the GPU lock step on the CPU arm's hash priors:
the two arms then build the same trees), `c4` (N = 64) at one GPU, `c3` (8192 roots per GPU) at eight, and at N > 1
`epoch_boundary` (azb_comm_init + azb_update_model + azb_comm_argmin over NCCL, timed outside the step metric).
The oracle (oracle/) is used only by the cpu_baseline leg and by --impl reference.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # no bytecode caches for the modules it imports from the tree (which may be read-only)

METRIC = "mcts_simulations_per_sec"
UNIT = "simulations/s"


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"  # /opt/skills/guides/B200_PROFILING.md


def algorithmic_bytes(k: dict, n: int) -> float:
    """SURVEY.md §8(d): compact record sizes x the workload counters of the launches (DESIGN.md §5)."""
    a = (n - 1) * (n - 2) // 2 - 1
    w = (a + 31) // 32
    NODE, EDGE, PRED = 32, 20, 12
    KEY, ST, VEC, H = 4 * w + 4, 4 * ((n + 3) // 4) + 4 * w, 8 * a, 4 * a
    tree = (k["n_sel"] * NODE + k["d_sel"] * (EDGE + NODE) + k["n_cand"] * PRED + k["n_probe"] * KEY
            + k["n_ins"] * (NODE + KEY) + k["n_arc"] * (EDGE + 4) + k["n_pred"] * PRED + k["n_cn"] * 2 * NODE
            + k["d_cn"] * EDGE)
    state = k["n_reset"] * ST + k["n_live"] * (2 * ST + VEC + H)
    return float(tree + state)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md's clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.thread = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.2] or [r for (_, r) in self.rows]
        if not rows:
            return None
        sm = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({nm for r in rows for nm, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(rows)}


def cpu_reference_run(n, roots, steps, warmup, seed, threads, budget_s=None):
    """The restated reference (oracle/azb_oracle.cpp: dense eigensolve, leaf-stripping matching, ordered maps) on
    the host cores.  Tree + state + cost are timed; priors are the counter hash (the reference evaluates its MLP on
    a GPU through dfdx — nabla/model/dfdx.rs:81-83 — so no CPU forward is part of its CPU path).
    With `budget_s` the steps run in chunks of 50 and the run stops after the chunk that crosses the budget (a
    bounded sample: the steps actually run are returned)."""
    from oracle import oracle

    oracle.build()
    a = oracle.action_dim(n)
    parents, masks = oracle.generate_roots(seed, 0, roots, n)
    o = oracle.Optimizer(n, roots, lambda_method=oracle.LAMBDA_DENSE, n_threads=threads)
    o.set_roots(parents, masks)
    o.init_trees(oracle.hash_priors(seed, 0, roots, a, 0))
    if warmup:
        o.steps_hash(seed, 0, 1, warmup)
    o.reset_counters()
    t0 = time.perf_counter()
    done = 0
    while done < steps:
        c = min(50, steps - done) if budget_s else steps
        o.steps_hash(seed, 0, 1 + warmup + done, c)
        done += c
        if budget_s and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    k = o.counters()
    k["steps_run"] = done
    return k["n_live"] / dt, dt, k


def dump_outputs(out_dir, h, capi, n_improved, seed, world=1, budget=64_000_000, row_budget=40_000_000, max_trees=32):
    """Writes what the timed steps computed, as of their last step, to out_dir/<name>.npy in float32 or float64 (counts
    and indices as exact integers): the step counters and improvement count, the argmin, and per tree the model's
    priors, the state vectors it read, the walker's path length and the tree sizes, then the node records of a few
    whole trees.  A tree whose root is exhausted did not expand in the step (path length 0): its prior and state rows
    are zeros.  With `world` ranks each rank gets 1/world of both byte budgets, so the dumps of all ranks together stay
    within them.  When all rows do not fit the row budget, a fixed sample of trees drawn from `seed` is written, in
    tree order."""
    budget //= world
    row_budget //= world
    os.makedirs(out_dir, exist_ok=True)
    out = {"counters": np.array([h.counters()[f] for f in capi.COUNTER_FIELDS], dtype=np.float64),
           "n_improved": np.array([n_improved], dtype=np.float64)}
    am = h.argmin()
    out.update(argmin_eval=np.array([am["eval"]], dtype=np.float32), argmin_lambda1=np.array([am["lambda1"]]),
               argmin_mu=np.array([am["mu"]], dtype=np.float64), argmin_parents=am["parents"].astype(np.float64),
               argmin_permitted=am["permitted"].astype(np.float64))
    k = min(h.b, row_budget // (4 * 3 * h.a + 8 * 4))
    rows = np.arange(h.b) if k == h.b else np.sort(np.random.default_rng(seed).choice(h.b, k, replace=False))
    priors, states = h.priors()[rows], h.state_vecs()[rows]
    path_len = h.walkers()["path_len"][rows]
    priors[path_len == 0] = 0.0
    states[path_len == 0] = 0.0
    out.update(priors=priors, state_vecs=states, walker_path_len=path_len.astype(np.float64),
               tree_sizes=np.array([h.tree_sizes(int(i)) for i in rows], dtype=np.float64))
    # whole trees, one record per node: tree, c, c*, n_t, exhausted children, prediction range lo, hi (include/azb.h);
    # as many sampled trees as the byte budget leaves room for
    used = sum(a.nbytes for a in out.values()) + 128 * (len(out) + 1)  # each .npy file adds a 128-byte header
    nodes = []
    for i in rows[np.linspace(0, len(rows) - 1, min(max_trees, len(rows))).astype(np.int64)]:
        nd = h.dump_tree(int(i))["nodes"]
        costs = np.ascontiguousarray(nd[:, :2]).view(np.float32)  # c and c* are stored as their f32 bit patterns
        rec = np.concatenate([np.full((len(nd), 1), i, dtype=np.float64), costs.astype(np.float64),
                              nd[:, 2:].astype(np.float64)], axis=1)
        if used + rec.nbytes > budget:
            break
        nodes.append(rec)
        used += rec.nbytes
    out["tree_nodes"] = np.concatenate(nodes) if nodes else np.zeros((0, 7))
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def timed_config(capi, n, b, workers, steps, warmup, seed, rank, local_rank, prior_hash=False, mlp_mode=None):
    """K device-timed steps of another configuration on this rank's GPU (inputs resident, W warm-up steps first).
    Returns (simulations, ms, cost evals, device bytes)."""
    kw = dict(device=local_rank, first_root=rank * b, max_steps=warmup + steps + 8)
    if prior_hash:
        kw.update(prior_mode=capi.PRIOR_HASH, prior_seed=seed)
    else:
        kw.update(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC if mlp_mode is None else mlp_mode, async_workers=workers)
    parents, masks = capi.generate_roots(seed, rank * b, b, n)
    with capi.Handle(capi.default_config(n, b, **kw)) as h:
        if not prior_hash:
            h.mlp_init(seed + 1)
        h.set_roots(parents, masks)
        h.init_trees()
        h.step(warmup)
        h.reset_counters()
        h.set_counter_mode(False)
        ms, _ = h.step_timed(steps)
        k = h.counters()
        return float(k["n_live"]), float(ms), float(k["n_ins"]), h.device_bytes()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=800, help="timed steps (800 = one epoch of the example)")
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--roots", type=int, default=4096, help="roots per GPU (BASELINE configs[1])")
    ap.add_argument("--vertices", type=int, default=19)
    ap.add_argument("--mlp", default=os.environ.get("AZB_MLP", "tc"), choices=["fp32", "tc", "tc3"],
                    help="tc: bf16 tensor cores (default); tc3: bf16x3 tensor cores at f32 accuracy; fp32: CUDA cores")
    ap.add_argument("--max-episodes", type=int, default=int(os.environ.get("AZB_MAX_EPISODES", "0")))
    ap.add_argument("--groups", type=int, default=int(os.environ.get("AZB_GROUPS", "1")),
                    help="concurrent tree groups per GPU (own CUDA stream each); needs --max-episodes 0")
    ap.add_argument("--async-workers", type=int, default=int(os.environ.get("AZB_ASYNC_WORKERS", "-1")),
                    help="tensor-core worker SMs of the asynchronous search kernel; 0 = lock step; -1 = auto")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-baseline-roots", type=int, default=4096)
    ap.add_argument("--cpu-baseline-seconds", type=float, default=20.0, help="time bound of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the same_priors / c3 / c4 objects")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what they computed to DIR/<name>.npy (rank r > 0: DIR/rank<r>/); "
                         "the inputs depend only on the arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    # stdout carries exactly ONE line, the JSON: everything else a library prints there (NCCL's version banner, ...) goes
    # to stderr for the rest of the run
    sys.stdout.flush()
    out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n, b = args.vertices, args.roots
    host_threads = os.cpu_count() or 1

    # ------------------------------------------------------------------ reference arm: CPU path on the host cores
    if args.impl == "reference":
        if rank != 0:
            return 0
        sample_roots = b  # the whole per-GPU batch; bounded in time instead (a step = one pass over these roots)
        val, dt, k = cpu_reference_run(n, sample_roots, args.steps, args.warmup, args.seed, host_threads, budget_s=60.0)
        line = {
            "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / k["steps_run"] * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
            "config": {"workload": f"06-c21 (snapshot: 04-c21-tree.rs) N={n}, {sample_roots} roots (one GPU's batch), "
                                   f"n_as_tol=[200,50,50]->25, hash priors", "vertices": n, "roots": sample_roots,
                       "steps_run": k["steps_run"], "seconds": dt},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": host_threads, "kind": "port",
                             "sample": f"{sample_roots} roots x {k['steps_run']} steps ({dt:.1f} s) after {args.warmup} warm-up; the "
                                       "reference is Rust and cannot be built here, so this is its C++ restatement "
                                       "(oracle/), tree+state+cost on all host threads, MLP forward excluded"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        out.write(json.dumps(line) + "\n")
        out.flush()
        return 0

    # ------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist

    backend = None
    if world > 1:
        # roots shard across ranks with no collective inside a step; the cross-rank traffic of this benchmark is the
        # barrier, a few scalar reductions and the communicator id — over NCCL like everything else on this box
        import datetime

        torch.cuda.set_device(local_rank)
        try:
            dist.init_process_group("nccl", timeout=datetime.timedelta(seconds=180),
                                    device_id=torch.device("cuda", local_rank))
            backend = "nccl"
        except Exception as e:  # pragma: no cover - the line says so
            sys.stderr.write(f"bench: NCCL process group failed ({e}); using gloo for the scalars\n")
            dist.init_process_group("gloo", timeout=datetime.timedelta(seconds=180))
            backend = "gloo"
    from azdopt_b200 import capi

    a = capi.action_dim(n)
    total_steps = args.warmup + args.steps
    prof_steps = min(args.steps, 100)
    aw = args.async_workers
    if aw < 0:  # auto: the library's choice for this root count (AZB_ASYNC_AUTO; include/azb.h)
        aw = capi.ASYNC_AUTO if not args.max_episodes and args.groups == 1 else 0
    cfg = capi.default_config(n, b, device=local_rank, first_root=rank * b, prior_mode=capi.PRIOR_MLP,
                              mlp_mode={"tc": capi.MLP_TC, "tc3": capi.MLP_TC3, "fp32": capi.MLP_FP32}[args.mlp],
                              max_steps=total_steps + prof_steps + 8, max_episodes=args.max_episodes,
                              n_groups=1 if args.max_episodes else args.groups, async_workers=aw)
    parents, masks = capi.generate_roots(args.seed, rank * b, b, n)
    mlp_note = args.mlp
    try:
        h = capi.Handle(cfg)
    except capi.AzbError as e:  # e.g. no tensor-map driver entry point: still a CUDA path, and the line says so
        if args.mlp == "fp32":
            raise
        cfg.mlp_mode = capi.MLP_FP32
        cfg.async_workers = aw = 0
        h = capi.Handle(cfg)
        mlp_note = f"fp32 (tensor-core path unavailable: {e})"
        args.mlp = "fp32"
    aw = cfg.async_workers = int(h.cfg.async_workers)  # the resolved choice
    h.mlp_init(args.seed + 1)  # same seed on every rank: replicated weights

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    dev = torch.device("cuda", local_rank) if backend == "nccl" else torch.device("cpu")

    def allreduce(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    # ---- device-resident timing: inputs in HBM, W warm-up steps, K timed steps
    h.set_roots(parents, masks)
    h.init_trees()
    try:
        h.step(args.warmup)
    except capi.AzbError as e:
        if not aw:
            raise
        # the persistent kernel could not run here (e.g. no cooperative launch): same path, lock-step launches
        sys.stderr.write(f"bench: asynchronous kernel unavailable ({e}); falling back to the lock step\n")
        h.close()
        cfg.async_workers = aw = 0
        h = capi.Handle(cfg)
        h.mlp_init(args.seed + 1)
        h.set_roots(parents, masks)
        h.init_trees()
        h.step(args.warmup)
    h.reset_counters()
    h.set_counter_mode(False)  # timed pass: only n_live / n_noop / n_ins are counted
    launches0 = h.kernel_launches()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.25)
    barrier()
    t0 = time.time()
    ms, n_improved = h.step_timed(args.steps)
    barrier()
    t1 = time.time()
    clocks = sampler.stop(t0, t1)
    launches = h.kernel_launches() - launches0
    k = h.counters()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs if rank == 0 else os.path.join(args.dump_outputs, f"rank{rank}"), h, capi,
                     n_improved, args.seed, world=world)
    h.set_counter_mode(True)
    ms_max = allreduce(ms, dist.ReduceOp.MAX if world > 1 else None)
    sims = allreduce(float(k["n_live"]), dist.ReduceOp.SUM if world > 1 else None)
    evals = allreduce(float(k["n_ins"]), dist.ReduceOp.SUM if world > 1 else None)
    noops = allreduce(float(k["n_noop"]), dist.ReduceOp.SUM if world > 1 else None)
    value = sims / (ms_max * 1e-3)

    # ---- roofline of the dominant kernel (the search kernel): events over a continuation of the run with all
    #      workload counters on.  Lock step: one launch per step, per-launch events.  Asynchronous kernel: ONE launch
    #      runs all prof_steps steps (search + in-kernel model forward), so "per launch" is that whole launch.
    h.reset_counters()
    hbm_peak, peak_src = _peaks()
    if aw:
        prof_ms, _ = h.step_timed(prof_steps)
        kp = h.counters()
        tree_ms, mlp_ms = prof_ms, 0.0
        bytes_per_launch = algorithmic_bytes(kp, n)
        tree_launch_s = prof_ms * 1e-3
    else:
        tree_ms, mlp_ms = h.step_profile(prof_steps)
        kp = h.counters()
        bytes_per_launch = algorithmic_bytes(kp, n) / prof_steps
        tree_launch_s = tree_ms * 1e-3 / prof_steps
    achieved = bytes_per_launch / tree_launch_s / 1e9
    traffic = None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel (ncu --set full, profiles/)
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tr = json.load(f)
        if tr.get("roots") == b and tr.get("vertices") == n and tr.get("kernel") == ("azb_async_kernel" if aw else "azb_tree_kernel"):
            traffic = tr["dram_bytes_per_launch"] * (prof_steps / tr.get("steps_per_launch", prof_steps) if aw else 1)
    except Exception:
        pass
    # what actually bounds the search kernel (DESIGN.md §4.4): instruction issue and single-warp latency, not bytes.  The
    # warp-instruction count per launch is ncu's (same capture as `traffic`); the duration is this run's
    issue = None
    try:
        if traffic is not None and tr.get("warp_instructions_per_launch"):
            n_sm, sm_hz = torch.cuda.get_device_properties(local_rank).multi_processor_count, 1.965e9
            wi = tr["warp_instructions_per_launch"] * (prof_steps / tr.get("steps_per_launch", prof_steps) if aw else 1)
            issue = {"warp_instructions_per_launch": wi, "achieved_ginst_per_s": wi / tree_launch_s / 1e9,
                     "peak_ginst_per_s": n_sm * 4 * sm_hz / 1e9, "frac": wi / tree_launch_s / (n_sm * 4 * sm_hz),
                     "what": "warp instructions per launch (ncu smsp__inst_executed.sum, profiles/r02_traffic.json) / this run's launch "
                             "duration, against 4 issue slots per SM per clock at 1965 MHz"}
    except Exception:
        issue = None
    roofline = {"bound": "hbm", "kernel": "azb_async_kernel" if aw else "azb_tree_kernel", "achieved": achieved,
                "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_per_launch, "launch_us": tree_launch_s * 1e6,
                "steps_per_launch": prof_steps if aw else 1,
                "mlp_us_per_step": None if aw else mlp_ms * 1e3 / prof_steps,
                "tree_share_of_step": None if aw else tree_ms / max(tree_ms + mlp_ms, 1e-9), "issue": issue}
    dev_bytes = h.device_bytes()

    # ---- e2e: a whole epoch through the C ABI with HOST buffers: roots H2D (set_roots), init, K per-step calls each
    #      reading back the step's result (improvement record + status), final argmin D2H
    h2 = h  # same handle: the reference's optimizer also re-seeds its trees in place (par_reset_trees)
    barrier()
    e0 = time.perf_counter()
    h2.set_roots(parents, masks)
    h2.init_trees()
    n_live_before = h2.counters()["n_live"]
    n_imp, imp_log = h2.step(args.steps, cap=args.steps)  # the epoch's K steps in one call, improvement log to the host
    am = h2.argmin()
    torch.cuda.synchronize()
    e1 = time.perf_counter()
    e2e_sims = h2.counters()["n_live"] - n_live_before
    e2e_s = allreduce(e1 - e0, dist.ReduceOp.MAX if world > 1 else None)
    e2e_sims = allreduce(float(e2e_sims), dist.ReduceOp.SUM if world > 1 else None)
    roots_bytes = parents.nbytes + masks.nbytes
    e2e = {"value": e2e_sims / e2e_s, "unit": UNIT,
           "h2d_bytes_per_step": roots_bytes / args.steps,
           "d2h_bytes_per_step": (48 + 16 * min(n_imp, args.steps) + n + 4 * capi.mask_words(n) + 16) / args.steps,
           "what": "one epoch through the C ABI with host buffers: azb_set_roots(host roots, H2D) + azb_init_trees + "
                   "azb_step(K steps, per-step improvement log D2H) + azb_get_argmin(D2H); wall clock, max over ranks"}
    # the same epoch driven one step per call, like the reference's loop body (04-c21-tree.rs:143): every call
    # synchronises and reads the step's improvement record back
    for _ in range(3):  # warm-up of the single-step path (its CUDA graph and lazily loaded kernels are first used here)
        h2.step(1, cap=4)
    barrier()
    p0 = time.perf_counter()
    h2.set_roots(parents, masks)
    h2.init_trees()
    n_live_before = h2.counters()["n_live"]
    for _ in range(args.steps):
        h2.step(1, cap=4)
    am1 = h2.argmin()
    torch.cuda.synchronize()
    p1 = time.perf_counter()
    ps_sims = allreduce(float(h2.counters()["n_live"] - n_live_before), dist.ReduceOp.SUM if world > 1 else None)
    ps_s = allreduce(p1 - p0, dist.ReduceOp.MAX if world > 1 else None)
    e2e["per_step_calls"] = {"value": ps_sims / ps_s, "unit": UNIT,
                             "what": "same, K x azb_step(1) (one CUDA-graph launch + sync + read-back per step)",
                             "same_argmin": bool(am1["eval"] == am["eval"])}
    # ... and with the trees running ahead of the caller: azb_step_enqueue(K), then one azb_step_poll per step (the
    # step's ArgminImprovement as soon as every tree has finished it), azb_step(0) to complete
    barrier()
    q0 = time.perf_counter()
    h2.set_roots(parents, masks)
    h2.init_trees()
    n_live_before = h2.counters()["n_live"]
    h2.step_enqueue(args.steps)
    n_pol = 0
    for _ in range(args.steps):
        n_pol += 1 if h2.step_poll()[0] else 0
    h2.step(0)
    am2 = h2.argmin()
    torch.cuda.synchronize()
    q1 = time.perf_counter()
    pq_sims = allreduce(float(h2.counters()["n_live"] - n_live_before), dist.ReduceOp.SUM if world > 1 else None)
    pq_s = allreduce(q1 - q0, dist.ReduceOp.MAX if world > 1 else None)
    e2e["per_step_polled"] = {"value": pq_sims / pq_s, "unit": UNIT,
                              "what": "same, azb_step_enqueue(K) + K x azb_step_poll (each step's improvement record read back "
                                      "as soon as every tree has finished it, later steps still running) + azb_step(0)",
                              "d2h_bytes_per_step": 8 * b, "same_argmin": bool(am2["eval"] == am["eval"]),
                              "same_improvements": bool(n_pol == n_imp)}
    # ---- epoch boundary over NCCL (N > 1): the library's own communicator (azb_comm_init), the sharded training step
    #      (weight sum, 1 284 248-float gradient and loss all-reduced inside azb_update_model) and the all-gather of the
    #      per-rank best (azb_comm_argmin).  Timed separately; none of it is inside the step metric.
    epoch_boundary = None
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid = torch.frombuffer(bytearray(capi.comm_unique_id()), dtype=torch.uint8).to(dev)
        dist.broadcast(uid, 0)
        try:
            h.comm_init(uid.cpu().numpy().tobytes(), rank, world)
            n_obs_tol = min(200, max(1, args.steps // 4))  # the example's 200 after a whole 800-step epoch
            barrier()
            h.update_model(n_obs_tol)  # first call: buffers, NCCL channel set-up
            barrier()
            u0 = time.perf_counter()
            loss = h.update_model(n_obs_tol)
            torch.cuda.synchronize()
            u1 = time.perf_counter()
            gbest = h.comm_argmin()
            torch.cuda.synchronize()
            u2 = time.perf_counter()
            ar_ms = h.comm_allreduce_bench(20)
            epoch_boundary = {
                "collective": "NCCL (libazb's communicator: ncclAllReduce x3 in azb_update_model, ncclAllGather in azb_comm_argmin)",
                "nccl_ranks": world, "update_model_ms": allreduce((u1 - u0) * 1e3, dist.ReduceOp.MAX),
                "comm_argmin_ms": allreduce((u2 - u1) * 1e3, dist.ReduceOp.MAX),
                "gradient_allreduce_ms": allreduce(ar_ms, dist.ReduceOp.MAX), "gradient_floats": h.mlp_num_params(),
                "loss": float(loss), "global_best_eval": float(gbest[4]), "global_best_owner_rank": int(gbest[5]),
                "n_obs_tol": n_obs_tol}
        except capi.AzbError as e:
            epoch_boundary = {"error": str(e), "nccl_ranks": world}
    h.close()

    # ---- the other configurations BASELINE.json names, as objects beside the headline (same timing rules: W warm-up
    #      steps, inputs resident, events on the library's stream, max over ranks)
    extra = {}
    xsteps = min(args.steps, 400)
    if world == 1 and not args.no_extra:
        # the GPU on the CPU arm's own priors (counter hash; lock step, no model): identical trees in both arms
        sp_steps = min(args.steps, 200)
        sp_sims, sp_ms, _, _ = timed_config(capi, n, b, 0, sp_steps, args.warmup, args.seed, rank, local_rank, prior_hash=True)
        extra["same_priors"] = {"value": sp_sims / (sp_ms * 1e-3), "unit": UNIT, "steps": sp_steps, "ms_per_step": sp_ms / sp_steps,
                                "what": f"N={n}, {b} roots, hash priors (the reference arm's), no model forward: the search (tree + state + cost) "
                                        "kernel ALONE, one launch for all the steps (every warp takes its tree through them; hash priors "
                                        "are computed in add_actions, so no tree waits for anybody)",
                                "hbm_frac_algorithmic": (sp_sims / (sp_ms * 1e-3)) * (algorithmic_bytes(kp, n) / max(kp["n_live"], 1)) / 1e9 / hbm_peak}
        try:  # the issue roofline of the search kernel alone: ncu's warp instructions per tree-step x this run's tree-steps/s
            wi_step = tr["tree_kernel_alone"]["warp_instructions_per_tree_step"]
            n_sm = torch.cuda.get_device_properties(local_rank).multi_processor_count
            extra["same_priors"]["issue_frac"] = (b * sp_steps / (sp_ms * 1e-3)) * wi_step / (n_sm * 4 * 1.965e9)
            extra["same_priors"]["issue_note"] = ("warp instructions per tree-step from profiles/r02_traffic.json (ncu of this kernel at 65 536 "
                                                  "roots: issue slots 69.5 % busy) x tree-steps/s of this run / (SMs x 4 x 1965 MHz)")
        except Exception:
            pass
        # the f32-accurate tensor-core model (AZB_MLP_TC3: bf16 hi + lo operands, three products per dot product): what the
        # reference's f32 forward costs on the tensor cores; the default stays bf16 because it is the faster step
        if args.mlp == "tc" and aw:
            t3_steps = min(args.steps, 200)
            t3_sims, t3_ms, _, _ = timed_config(capi, n, b, aw, t3_steps, args.warmup, args.seed, rank, local_rank, mlp_mode=capi.MLP_TC3)
            extra["f32_accurate_model"] = {"value": t3_sims / (t3_ms * 1e-3), "unit": UNIT, "steps": t3_steps, "ms_per_step": t3_ms / t3_steps,
                                           "what": "same workload with mlp_mode = AZB_MLP_TC3 (priors within 1e-5 relative of the f32 forward; "
                                                   "tests/test_gpu_parity.py) instead of bf16 (2e-2 absolute)"}
        # C4: 64-vertex trees (cost path dominated): 4096 roots, the library's layout for N >= 47 (16 model SMs)
        c4_roots, c4_steps = 4096, min(args.steps, 64)
        try:
            c4_sims, c4_ms, ev4, bytes4 = timed_config(capi, 64, c4_roots, capi.ASYNC_AUTO, c4_steps, max(3, min(args.warmup, 8)), args.seed, rank, local_rank)
            extra["c4"] = {"value": c4_sims / (c4_ms * 1e-3), "unit": UNIT, "vertices": 64, "roots": c4_roots, "steps": c4_steps,
                           "ms_per_step": c4_ms / c4_steps, "cost_evals_per_sec": ev4 / (c4_ms * 1e-3), "device_bytes": bytes4,
                           "what": "BASELINE configs[3]: N=64 (A=1952, MLP 3904-512-1024-512-1952), asynchronous kernel, 16 model SMs "
                                   "(AZB_ASYNC_AUTO), 16 tree warps per SM taking over each other's runnable trees"}
        except capi.AzbError as e:
            extra["c4"] = {"error": str(e)}
    if world == 8 and not args.no_extra:
        # C3: 65 536 roots over the 8 GPUs = 8192 per GPU, the library's layout (36 model SMs)
        c3_sims, c3_ms, ev3, _ = timed_config(capi, n, 8192, capi.ASYNC_AUTO, xsteps, args.warmup, args.seed, rank, local_rank)
        ms3 = allreduce(c3_ms, dist.ReduceOp.MAX)
        sims3 = allreduce(c3_sims, dist.ReduceOp.SUM)
        extra["c3"] = {"value": sims3 / (ms3 * 1e-3), "unit": UNIT, "roots_total": 8192 * world, "roots_per_gpu": 8192,
                       "steps": xsteps, "ms_per_step": ms3 / xsteps,
                       "what": "BASELINE configs[2]: 65 536 roots sharded over 8 GPUs, no collective inside a step"}

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload on the host cores
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = min(b, args.cpu_baseline_roots)
        val, dt, kc = cpu_reference_run(n, cb, args.steps, 4, args.seed, host_threads, budget_s=args.cpu_baseline_seconds)
        cpu = {"value": val, "unit": UNIT, "cores": host_threads, "kind": "port",
               "sample": f"{cb} roots x {kc['steps_run']} steps ({dt:.1f} s); restated reference (C++ oracle), tree+state+cost on "
                         "all host threads, hash priors, MLP forward excluded"}

    if cpu and "same_priors" in extra:
        extra["same_priors"]["cpu_value"] = cpu["value"]
        extra["same_priors"]["ratio_vs_cpu"] = extra["same_priors"]["value"] / cpu["value"]
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 search + f64 lambda_1 + " + {"tc": "bf16 tensor-core MLP", "tc3": "bf16x3 tensor-core MLP (f32 accuracy)", "fp32": "f32 MLP"}[args.mlp],
            "data": "synthetic",
            "config": {"workload": f"06-c21 (snapshot: 04-c21-tree.rs) N={n}, {b} roots per GPU x {world} GPU, "
                                   f"random-init MLP {2 * a}-512-1024-512-{a}, n_as_tol=[200,50,50]->25",
                       "vertices": n, "roots_per_gpu": b, "roots_total": b * world, "mlp": mlp_note, "max_episodes_per_launch": args.max_episodes, "tree_groups": 1 if args.max_episodes else args.groups,
                       "search": (f"asynchronous: ONE persistent cooperative kernel per azb_step call — {148 - aw} SMs walk trees, "
                                  f"{aw} SMs run the tensor-core model (setmaxnreg role split)" if aw
                                  else "lock step: one search launch + model forward per step"),
                       "l2": f"per-GPU arenas {dev_bytes / 1e6:.0f} MB > 126 MB L2; no flush between steps",
                       "simulations_in_timed_region": sims, "noop_root_steps": noops,
                       "cost_evals_per_sec": evals / (ms_max * 1e-3)},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "argmin_eval": float(am["eval"]),
        }
        line.update(extra)
        if epoch_boundary is not None:
            line["epoch_boundary"] = epoch_boundary
        out.write(json.dumps(line) + "\n")
        out.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
