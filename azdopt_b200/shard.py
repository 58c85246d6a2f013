"""Sharding of roots over one process per GPU (SURVEY.md §8e): contiguous blocks of roots per rank, no collective
inside a step; epoch-boundary collectives over torch.distributed (NCCL on GPUs, gloo in CPU tests)."""
from __future__ import annotations

import glob
import os

import numpy as np


def shard_range(total: int, rank: int, world: int):
    """Contiguous block [lo, hi) of rank's roots; sizes differ by at most one."""
    base, rem = divmod(total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def global_argmin(local_eval: float, local_parents: np.ndarray, local_permitted: np.ndarray, dist=None, device="cpu"):
    """All-gather of each rank's (best eval, state) and a first-minimum over ranks (optimizer/mod.rs:221: lowest
    index wins ties).  Returns (eval, rank, parents, permitted)."""
    import torch

    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        return float(local_eval), 0, local_parents, local_permitted
    world = dist.get_world_size()
    rec = np.concatenate([np.array([local_eval], dtype=np.float32).view(np.uint8), local_parents.astype(np.uint8),
                          local_permitted.astype(np.uint32).view(np.uint8)])
    t = torch.from_numpy(rec.copy()).to(device)
    out = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    recs = [o.cpu().numpy() for o in out]
    evals = [float(r[:4].view(np.float32)[0]) for r in recs]
    best = min(range(world), key=lambda r: (evals[r], r))
    r = recs[best]
    n = local_parents.size
    return evals[best], best, r[4:4 + n].copy(), r[4 + n:].view(np.uint32).copy()


def sum_counters(counters: dict, dist=None, device="cpu") -> dict:
    """Sum the workload counters of all ranks (whole-job simulations = sum of n_live)."""
    import torch

    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        return dict(counters)
    keys = sorted(counters)
    t = torch.tensor([counters[k] for k in keys], dtype=torch.int64, device=device)
    dist.all_reduce(t)
    return {k: int(v) for k, v in zip(keys, t.cpu().tolist())}


def global_best_trees(local: list, k: int, dist=None) -> list:
    """The k best isomorphism classes over all ranks: every rank's best_trees list (nabla.BestTree records) gathered
    and merged in rank order, so a class found on several ranks at one value keeps the lowest rank's representative —
    the lowest global root, as one unsharded handle would pick."""
    from .nabla import BestTrees

    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        return BestTrees(k).add(local).result()
    lists = [None] * dist.get_world_size()
    dist.all_gather_object(lists, list(local))
    acc = BestTrees(k)
    for lst in lists:
        acc.add(lst)
    return acc.result()


def merge_exhaustive_best(results: list, k: int) -> dict:
    """The k best of several Handle.exhaustive_best results over disjoint index ranges, by (key, index) with key =
    mu + lambda1 in f64 as the library computes it, so the merge equals one call over the union; n_below is summed."""
    cat = {name: np.concatenate([r[name] for r in results]) for name in ("index", "parents", "lambda1", "mu", "eval")}
    key = cat["mu"].astype(np.float64) + cat["lambda1"]
    order = np.lexsort((cat["index"], key))[:k]
    out = {name: a[order] for name, a in cat.items()}
    out["n_below"] = sum(int(r["n_below"]) for r in results)
    return out


def global_exhaustive_best(local: dict, k: int, dist=None) -> dict:
    """The k best free trees over all ranks, each rank having ranked its shard_range(A000055(N), rank, world) of the
    enumeration with Handle.exhaustive_best: gathered and merged by (key, index), equal to one call over the whole range;
    n_below is summed."""
    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        return merge_exhaustive_best([local], k)
    lists = [None] * dist.get_world_size()
    dist.all_gather_object(lists, {name: local[name] for name in ("index", "parents", "lambda1", "mu", "eval", "n_below")})
    return merge_exhaustive_best(lists, k)


def checkpoint_path(directory: str, rank: int) -> str:
    """Where rank `rank` keeps its checkpoint blob inside a run's checkpoint directory."""
    return os.path.join(directory, f"rank{rank:05d}.azbckpt")


def checkpoint_paths(directory: str) -> list:
    """Every rank's checkpoint blob in `directory`, in rank order (temporary files of an interrupted save excluded)."""
    return sorted(p for p in glob.glob(os.path.join(directory, "rank*.azbckpt")) if os.path.isfile(p))


def resume_sharded(directory: str, space, model, total: int, rank: int, world: int, **kw):
    """This rank's NablaOptimizer over its shard_range of `total` roots, loaded from EVERY rank's file in `directory`
    (written by a run with any number of ranks): each file is memory-mapped, so only the headers and the records of this
    rank's roots are read."""
    from .nabla import NablaOptimizer

    lo, hi = shard_range(total, rank, world)
    paths = checkpoint_paths(directory)
    if not paths:
        raise FileNotFoundError(f"no checkpoint in {directory}")
    return NablaOptimizer.resume(paths, space, model, hi - lo, first_root=lo, **kw)
