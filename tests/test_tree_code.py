"""The canonical tree code of include/azb.h, as observe.tree_code states it, against networkx (CPU)."""
import networkx as nx
import numpy as np
import pytest

from azdopt_b200 import observe
from best_trees_util import parents_of, random_parents, relabel


@pytest.mark.parametrize("n,count", [(5, 3), (6, 6), (7, 11), (8, 23), (9, 47), (10, 106), (11, 235), (12, 551)])
def test_nonisomorphic_trees_get_distinct_codes(n, count):
    codes = [observe.tree_code(parents_of(T)) for T in nx.nonisomorphic_trees(n)]
    assert len(codes) == count and len(set(codes)) == count  # OEIS A000055
    for hi, lo in codes:
        s = format(hi, "064b") + format(lo, "064b")
        assert s[0] == "1" and s.count("1") == n and set(s[2 * n:]) <= {"0"}  # 2n bits, n ones, zero padded


def test_relabelling_keeps_the_code():
    rng = np.random.default_rng(1)
    for n in (5, 9, 19, 33, 64):
        for _ in range(20):
            p = random_parents(rng, n)
            c = observe.tree_code(p)
            for _ in range(3):
                assert observe.tree_code(relabel(rng, p)) == c


def test_equal_codes_iff_isomorphic():
    rng = np.random.default_rng(2)
    seen_equal_degrees = 0
    for _ in range(300):
        n = int(rng.integers(5, 20))
        a, b = random_parents(rng, n), random_parents(rng, n)
        if rng.random() < 0.3:
            b = relabel(rng, a)
        Ta = nx.Graph([(v, int(a[v])) for v in range(1, n)])
        Tb = nx.Graph([(v, int(b[v])) for v in range(1, n)])
        same_deg = sorted(d for _, d in Ta.degree()) == sorted(d for _, d in Tb.degree())
        iso = nx.is_isomorphic(Ta, Tb)
        seen_equal_degrees += same_deg and not iso
        assert (observe.tree_code(a) == observe.tree_code(b)) == iso
    # pairs that a degree sequence cannot tell apart
    for n in range(8, 13):
        trees = list(nx.nonisomorphic_trees(n))
        by_deg = {}
        for T in trees:
            by_deg.setdefault(tuple(sorted(d for _, d in T.degree())), []).append(T)
        for group in by_deg.values():
            codes = {observe.tree_code(parents_of(T)) for T in group}
            assert len(codes) == len(group)
            seen_equal_degrees += len(group) > 1
    assert seen_equal_degrees > 0


def _word_pair(s):
    bits = int(s.ljust(128, "0"), 2)
    return bits >> 64, bits & ((1 << 64) - 1)


@pytest.mark.parametrize("n", [5, 6, 19, 20, 63, 64])
def test_closed_forms(n):
    star = np.zeros(n, dtype=np.uint8)
    assert observe.tree_code(star) == _word_pair("1" + "10" * (n - 1) + "0")
    path = np.array([0] + list(range(n - 1)), dtype=np.uint8)
    if n % 2:  # one centre: two arms of (n - 1) / 2 vertices
        arm = "1" * ((n - 1) // 2) + "0" * ((n - 1) // 2)
        want = "1" + arm + arm + "0"
    else:  # two centres: rooted at either, one arm of n/2 - 1 and one of n/2
        want = "1" + "1" * (n // 2) + "0" * (n // 2) + "1" * (n // 2 - 1) + "0" * (n // 2 - 1) + "0"
    assert observe.tree_code(path) == _word_pair(want)


def test_rejects_bad_parent_arrays():
    with pytest.raises(ValueError):
        observe.tree_code(np.array([0, 0, 2, 1, 1], dtype=np.uint8))
