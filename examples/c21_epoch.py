#!/usr/bin/env python
"""The reference's example loop (graph-state/examples/04-c21-tree.rs:76-208) on the B200 path, through the Python
mirror of NablaOptimizer (azdopt_b200/nabla.py) — same constants, same outputs:

    python examples/c21_epoch.py [--batch 512] [--epochs 3] [--episodes 800] [--out out_dir] [--checkpoint DIR [--resume]]
                                 [--exhaustive]

Per epoch: `episodes` search steps fused on the device (improvements are printed with their step like the example's
process_argmin), par_update_model (loss), par_reset_trees with the example's modify_root policy.  Writes a TensorBoard
event file with the example's scalar tags, the best tree as graph6 and the first search DAG as Graphviz DOT.
With --checkpoint DIR the run is saved after every epoch (search and training state, the BestTrees accumulator and the
epoch count); --resume continues from the last save exactly where the interrupted run would have gone on.
With --exhaustive every tree on N vertices is ranked on the device before the first epoch (each rank its share of the
enumeration, like the roots) and every epoch logs the gap between the run's best and that exact optimum.
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from azdopt_b200 import capi, nabla, observe, shard  # noqa: E402

N = 19                       # 04-c21-tree.rs:33
C_LOWER, C_UPPER = 2.0, 15.0  # :58-68 for N = 19


def squish(c):  # :70-74
    return (c - C_LOWER) / (C_UPPER - C_LOWER)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)       # :54
    ap.add_argument("--epochs", type=int, default=3)        # :133 (250 in the example)
    ap.add_argument("--episodes", type=int, default=800)    # :134
    ap.add_argument("--n-obs-tol", type=int, default=200)   # :135
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default="c21_out")
    ap.add_argument("--best", type=int, default=0, metavar="K",
                    help="also keep the K best non-isomorphic trees over all epochs in best_trees.g6")
    ap.add_argument("--checkpoint", metavar="DIR", help="save the run here after every epoch")
    ap.add_argument("--resume", action="store_true", help="continue from the last checkpoint in --checkpoint DIR")
    ap.add_argument("--exhaustive", action="store_true",
                    help="rank every tree on N vertices first and log each epoch's gap to the exact optimum")
    args = ap.parse_args()
    if args.resume and not args.checkpoint:
        ap.error("--resume needs --checkpoint DIR")
    os.makedirs(args.out, exist_ok=True)
    space = nabla.ROTModifyParentsOnce(n=N)
    model = nabla.ActionModel(seed=args.seed + 1, arithmetic="tc")
    first_epoch, best = 1, (nabla.BestTrees(args.best) if args.best else None)
    if args.resume:
        progress = np.load(os.path.join(args.checkpoint, "progress.npz"))
        first_epoch = int(progress["epoch"]) + 1
        if best and "best_k" in progress:
            best = nabla.BestTrees.from_state({k[5:]: progress[k] for k in progress.files if k.startswith("best_")})
        opt = nabla.NablaOptimizer.resume(shard.checkpoint_paths(args.checkpoint), space, model, args.batch,
                                          max_steps=args.episodes)
    else:
        roots = capi.generate_roots(args.seed, 0, args.batch, N)  # ROTWithActionPermissions::generate, k ~ U{5..A/2} (:85,108-112)
        opt = nabla.NablaOptimizer.par_new(space, roots, model, args.batch, max_steps=args.episodes)
    goal = squish(5.2)                                         # :117
    optimum = None
    if args.exhaustive:
        rank, world = 0, 1                                     # one process here; each rank of a sharded run takes its range
        total = capi.free_tree_count(N)
        lo, hi = shard.shard_range(total, rank, world)
        ex = shard.global_exhaustive_best(opt.h.exhaustive_best(lo, hi - lo, k=1), 1)
        optimum = float(ex["eval"][0])
        print(f"exact optimum over all {total} trees: eval {optimum:.6f} lambda_1={ex['lambda1'][0]:.6f} mu={ex['mu'][0]} "
              f"(index {ex['index'][0]}); {ex['n_below']} trees below the star's sqrt(N - 1) + 1")

    def save_checkpoint(epoch):
        os.makedirs(args.checkpoint, exist_ok=True)
        opt.save(shard.checkpoint_path(args.checkpoint, 0))
        extra = {f"best_{k}": v for k, v in best.state().items()} if best else {}
        tmp = os.path.join(args.checkpoint, "progress.tmp.npz")
        np.savez(tmp, epoch=epoch, **extra)    # the TensorBoard steps continue from episodes * epoch
        os.replace(tmp, os.path.join(args.checkpoint, "progress.npz"))

    # a resumed run appends to the event file the interrupted run wrote
    with open(os.path.join(args.out, "tfevents-losses"), "ab" if args.resume else "wb") as f:
        writer = observe.TensorboardWriter(f)
        if not args.resume:
            writer.write_file_version()

        def process_argmin(a, step):                           # :119-130
            print(f"{a.eval:12.6f}\tlambda_1={a.lambda_1:.6f} mu={a.mu}")
            writer.write_cost(step, a.lambda_1, a.mu)
            writer.flush()
            return a.eval < goal

        if not args.resume:
            process_argmin(opt.argmin_data(), 0)
        for epoch in range(first_epoch, args.epochs + 1):
            print(f"==== EPOCH: {epoch} ====")
            improved = opt.roll_out(args.episodes)             # the inner loop :141-150, fused on the device
            if best:                                           # every node of this epoch's trees, before the reset
                best.add(opt.best_trees(args.best))
            for (step, tree, node, ev) in improved:
                print(f"  step {args.episodes * (epoch - 1) + step + 1}: tree {tree} node {node} eval {ev:.6f}")
            if optimum is not None:
                print(f"  gap to the exact optimum: {opt.argmin_data().eval - optimum:.6f}")
            if improved and process_argmin(opt.argmin_data(), args.episodes * epoch):
                print("state is optimal:", opt.argmin_data().parents.tolist())
                break
            loss = opt.par_update_model(args.n_obs_tol)        # :163
            writer.write_loss(args.episodes * epoch, loss)
            writer.write_cost(args.episodes * epoch, opt.argmin_data().lambda_1, opt.argmin_data().mu)
            writer.flush()
            print(f"  loss {loss:.6f}")
            with open(os.path.join(args.out, "tree.dot"), "w") as g:   # :153-157 (the example renders PNGs)
                g.write(opt.tree_dot(0))
            opt.par_reset_trees(seed=args.seed + 7)            # :172-207
            if args.checkpoint:
                save_checkpoint(epoch)
    with open(os.path.join(args.out, "best.g6"), "wb") as g:
        g.write(opt.argmin_graph6() + b"\n")
    print("best tree (graph6):", opt.argmin_graph6().decode())
    cert = opt.h.certify_keys(opt.argmin_data().parents[None])   # proven against sqrt(N - 1) + 1, or open
    verdict = {-1: "proven below", 0: "proven equal to", 1: "proven above", 2: "open against"}[int(cert["verdict"][0])]
    print(f"best tree's key mu + lambda_1 (lambda_1 in ({cert['lambda1_lo'][0]!r}, {cert['lambda1_hi'][0]!r}), "
          f"mu = {cert['mu'][0]}): {verdict} sqrt(N - 1) + 1")
    if best:
        with open(os.path.join(args.out, "best_trees.g6"), "wb") as g:
            for t in best.result():
                g.write(observe.graph6_of_state(t.parents) + f" {t.eval:.9g}\n".encode())
    opt.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
