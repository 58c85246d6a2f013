"""The free-tree enumeration of include/azb.h on the CPU: its plain restatement (free_trees_ref.py) against Otter's count,
networkx and the canonical code, and azb_free_tree_count (host only).  No kernel is launched here."""
import ctypes as C
from fractions import Fraction

import networkx as nx
import numpy as np
import pytest

import free_trees_ref as R
from azdopt_b200 import observe


def _a000081(nmax):
    """Rooted trees: a(n+1) = (1/n) sum_{k=1..n} (sum_{d | k} d a(d)) a(n-k+1), a(1) = 1."""
    a = [0, 1]
    for n in range(1, nmax):
        s = sum(sum(d * a[d] for d in range(1, k + 1) if k % d == 0) * a[n - k + 1] for k in range(1, n + 1))
        a.append(s // n)
    return a


def _otter(n, a):
    """A000055(n) = a(n) - (sum_{i=1..n-1} a(i) a(n-i) - [n even] a(n/2)) / 2."""
    conv = sum(a[i] * a[n - i] for i in range(1, n))
    if n % 2 == 0:
        conv -= a[n // 2]
    return int(a[n] - Fraction(conv, 2))


def _is_centroid(par, v):
    n = len(par)
    g = nx.Graph([(u, int(par[u])) for u in range(1, n)])
    g.remove_node(v)
    return max(len(c) for c in nx.connected_components(g)) <= n // 2


def test_counts_equal_otters_formula(capi):
    a = _a000081(32)
    for n in range(5, 33):
        want = _otter(n, a)
        assert R.free_tree_count(n) == want, n
        got = C.c_uint64()
        assert capi.lib().azb_free_tree_count(n, C.byref(got)) == capi.OK
        assert got.value == want == capi.free_tree_count(n), n
    for s in range(1, 17):
        assert R.rooted_count(s) == a[s]
    assert capi.free_tree_count(32) == 109972410221 and R.free_tree_count(19) == 317955


def test_count_refuses_sizes_outside_5_to_32(capi):
    got = C.c_uint64()
    for n in (0, 4, 33, 64):
        assert capi.lib().azb_free_tree_count(n, C.byref(got)) == capi.ERR_INVALID
    assert capi.lib().azb_free_tree_count(19, None) == capi.ERR_INVALID
    with pytest.raises(capi.AzbError):
        capi.free_tree_count(33)


@pytest.mark.parametrize("n", range(5, 13))
def test_restatement_lists_every_tree_once(n):
    rows = R.free_trees(n, 0, R.free_tree_count(n))
    for p in rows:
        assert all(p[v] < v for v in range(1, n))
        assert _is_centroid(p, 0)
    codes = [observe.tree_code(p) for p in rows]
    want = sorted(observe.tree_code(_parents_of(T)) for T in nx.nonisomorphic_trees(n))
    assert len(set(codes)) == len(codes) == len(want)
    assert sorted(codes) == want


def _parents_of(T):
    """parents[v] < v form of a networkx tree: BFS from vertex 0."""
    order = list(nx.bfs_tree(T, 0))
    idx = {v: i for i, v in enumerate(order)}
    par = [0] * len(order)
    for u, v in nx.bfs_edges(T, 0):
        par[idx[v]] = idx[u]
    return par


def test_rooted_ids_follow_size_then_sequence_order():
    # size 3: the sequences of sum 2 are [0, 0] (two leaves) < [1] (a path below the root)
    assert R.rooted(2) == (0, 0, 0) and R.rooted(3) == (0, 0, 1)
    starts, _ = R._tables()
    for s in range(2, 9):
        seqs = []
        for g in range(starts[s - 1], starts[s]):
            kids = R._sequence(s - 1, g - starts[s - 1], starts[s - 1] - 1)
            assert kids == sorted(kids, reverse=True) and sum(R.size_of(c) for c in kids) == s - 1
            seqs.append(kids)
        assert seqs == sorted(seqs) and len({tuple(q) for q in seqs}) == len(seqs)


@pytest.mark.parametrize("n", [30, 32])
def test_sampled_indices_at_30_and_32(n):
    total, u = R.free_tree_count(n), R.unicentroidal_count(n)
    rng = np.random.default_rng(n)
    idx = sorted({0, 1, u - 1, u, total - 1, *map(int, rng.integers(0, total, 300)), *map(int, rng.integers(u, total, 40))})
    codes = set()
    for i in idx:
        p = R.free_tree(n, i)
        assert p.shape == (n,) and all(p[v] < v for v in range(1, n))
        assert _is_centroid(p, 0)
        codes.add(observe.tree_code(p))
    assert len(codes) == len(idx)
    assert R.free_tree(n, 0).tolist() == [0] * n  # the star: n - 1 copies of id 0
    # even n: the last index is the pair of the last rooted tree of size n / 2 with itself (two paths: the path P_n)
    t = R.rooted_count(n // 2)
    assert total - u == t * (t + 1) // 2
    assert R.free_tree(n, total - 1).tolist() == [0, 0] + list(range(1, n // 2)) + [0] + list(range(n // 2 + 1, n - 1))
    with pytest.raises(IndexError):
        R.free_tree(n, total)


def test_shard_merge_orders_by_key_then_index():
    from azdopt_b200 import shard

    rng = np.random.default_rng(3)
    m = 500
    lam = rng.choice([2.0, 2.5, 3.0 + 1e-12], m)  # many exact ties in mu + lambda1
    mu = rng.integers(1, 4, m).astype(np.uint32)
    whole = dict(index=np.arange(m, dtype=np.uint64), parents=rng.integers(0, 9, (m, 9)).astype(np.uint8), lambda1=lam, mu=mu,
                 eval=(mu + lam).astype(np.float32))
    key = mu.astype(np.float64) + lam
    want = np.lexsort((np.arange(m), key))[:40]
    cuts = [0, 7, 8, 300, m]
    parts = [dict({name: a[lo:hi] for name, a in whole.items()}, n_below=hi - lo) for lo, hi in zip(cuts, cuts[1:])]
    got = shard.merge_exhaustive_best(parts[::-1], 40)
    assert got["index"].tolist() == want.tolist() and got["n_below"] == m
    assert np.array_equal(got["parents"], whole["parents"][want])
    assert shard.global_exhaustive_best(dict(whole, n_below=5), 40)["index"].tolist() == want.tolist()
