"""Merging best-trees lists (nabla.BestTrees across epochs, shard.global_best_trees across ranks over gloo) equals the
top k of the union, on synthetic lists with ties in value and in code (CPU)."""
import os
import pickle
import sys

import numpy as np
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _nodes(rng, roots, n_nodes):
    """Synthetic node records (eval, code, global root, node) with many ties in eval and in code."""
    out = []
    for r in roots:
        for i in range(n_nodes):
            ev = np.float32(rng.integers(0, 12) / 16.0)
            code = (int(rng.integers(0, 6)) << 60 | 1 << 63, int(rng.integers(0, 3)))
            out.append((ev, code, int(r), i))
    return out


def _top(nodes, k):
    """What azb_best_trees returns for these nodes: per code the minimum (eval, root, node), then (eval, code), k first."""
    from azdopt_b200.nabla import BestTree

    best = {}
    for ev, code, r, i in nodes:
        if code not in best or (ev, r, i) < (best[code][0], best[code][2], best[code][3]):
            best[code] = (ev, code, r, i)
    rows = sorted(best.values(), key=lambda t: (t[0], t[1]))[:k]
    return [BestTree(ev, 0.0, 0, np.zeros(1, np.uint8), np.zeros(1, np.uint32), code, r, i) for ev, code, r, i in rows]


def _key(trees):
    return [(float(t.eval), t.code, t.root, t.node) for t in trees]


def test_epochs_and_shards_merge_to_the_union_top_k():
    from azdopt_b200.nabla import BestTrees

    rng = np.random.default_rng(3)
    for k in (1, 2, 3, 5, 40):
        shards = [_nodes(rng, range(8 * s, 8 * s + 8), 6) for s in range(4)]  # contiguous roots, rank order
        union = [x for s in shards for x in s]
        acc = BestTrees(k)
        for s in shards:
            acc.add(_top(s, k))
        assert _key(acc.result()) == _key(_top(union, k))
        # adding a list twice or an empty list changes nothing
        acc.add(_top(shards[0], k)).add([])
        assert _key(acc.result()) == _key(_top(union, k))


def test_equal_value_keeps_the_existing_entry():
    from azdopt_b200.nabla import BestTree, BestTrees

    a = BestTree(np.float32(0.5), 1.0, 1, np.zeros(1, np.uint8), np.zeros(1, np.uint32), (1 << 63, 0), 7, 3)
    b = BestTree(np.float32(0.5), 2.0, 2, np.zeros(1, np.uint8), np.zeros(1, np.uint32), (1 << 63, 0), 1, 0)
    c = BestTree(np.float32(0.25), 3.0, 3, np.zeros(1, np.uint8), np.zeros(1, np.uint32), (1 << 63, 0), 9, 9)
    acc = BestTrees(4).add([a]).add([b])
    assert acc.result() == [a]
    assert BestTrees(4).add([a]).add([c]).result() == [c]


def _worker(rank, world, port, k, out_dir):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from azdopt_b200 import shard

    rng = np.random.default_rng(11)
    shards = [_nodes(rng, range(8 * s, 8 * s + 8), 6) for s in range(world)]
    res = shard.global_best_trees(_top(shards[rank], k), k, dist)
    with open(os.path.join(out_dir, f"b{rank}.pkl"), "wb") as f:
        pickle.dump(_key(res), f)
    dist.barrier()
    dist.destroy_process_group()


def test_global_best_trees_over_gloo(tmp_path):
    world, k = 2, 5
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(world, port, k, str(tmp_path)), nprocs=world, join=True)
    rng = np.random.default_rng(11)
    union = [x for s in range(world) for x in _nodes(rng, range(8 * s, 8 * s + 8), 6)]
    want = _key(_top(union, k))
    for r in range(world):
        with open(tmp_path / f"b{r}.pkl", "rb") as f:
            assert pickle.load(f) == want
