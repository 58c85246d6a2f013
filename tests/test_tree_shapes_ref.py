"""The shape families and the exact lambda_1 / mu reference of tree_shapes.py (CPU), and the evidence behind the 4-ulp
bound of the GPU tests: the oracle's mirror of the kernel is within 4 ulp of the exact lambda_1 on every input those
tests use."""
import math
from fractions import Fraction

import networkx as nx
import numpy as np
import pytest

import tree_shapes as ts
from azdopt_b200 import observe


def _all_inputs():
    for n in range(5, 65):
        for name, p in ts.shape_batch(n):
            yield n, name, p


def test_families_are_trees_in_parent_order():
    for n, name, p in _all_inputs():
        assert len(p) == n and p[0] == 0 and all(p[v] < v for v in range(1, n)), (n, name)


def test_inertia_count_at_eigenvalues_and_zero_pivots():
    """At x = -1, 0, 1/2, 1, 2 many pivots are zero (every odd tree has the eigenvalue 0, the star on 5 vertices has 2):
    the count equals the number of eigvalsh values above x."""
    rng = np.random.default_rng(3)
    trees = [f(n) for n in (5, 6, 7, 10, 17, 23) for f in ts.FAMILIES.values()]
    trees += [ts.random_tree(n, rng) for n in (5, 6, 8, 9, 12) for _ in range(20)]
    zero_rule = 0
    for p in trees:
        ev = np.linalg.eigvalsh(nx.to_numpy_array(nx.Graph(ts.edges_of(p)), nodelist=range(len(p))))
        for x in (Fraction(-1), Fraction(0), Fraction(1, 2), Fraction(1), Fraction(2)):
            want = int((ev > float(x) + 1e-9).sum())
            assert ts.eigen_count_above(p, int(x * 2 ** ts.SCALE)) == want, (p.tolist(), x)
            zero_rule += bool(np.any(np.abs(ev - float(x)) < 1e-9))
    assert zero_rule > 50


@pytest.mark.parametrize("n", range(5, 65))
def test_closed_forms(n):
    r, lo, hi = ts.exact_lambda1(ts.star(n))
    assert lo * lo < n - 1 <= hi * hi and r == math.sqrt(n - 1)  # sqrt is correctly rounded, so bit for bit
    r, lo, hi = ts.exact_lambda1(ts.path(n))
    assert abs(r - 2 * math.cos(math.pi / (n + 1))) <= math.ulp(r)
    assert hi - lo < Fraction(2) ** -92 * r
    assert ts.exact_mu(ts.star(n)) == 1 and ts.exact_mu(ts.path(n)) == n // 2


def test_reference_agrees_with_eigvalsh_and_networkx():
    for n, name, p in _all_inputs():
        r = ts.exact_lambda1(p)[0]
        dense = ts.lambda1_dense(p)
        assert abs(r - dense) <= 1e-13 * r, (n, name, r, dense)
        assert ts.exact_mu(p) == len(nx.max_weight_matching(nx.Graph(ts.edges_of(p)), maxcardinality=True)), (n, name)


def test_stack_program_extremes():
    """The inputs fill the kernel's stack: T(k) needs k slots, as many as azb_stack_depth allows at 22, 23, 46, 47 and
    64 vertices, and the comb of cherries has the longest program, 94 ops at 64 vertices."""
    assert [len(ts.t_k(k)) for k in range(1, 6)] == [2, 5, 11, 23, 47]
    assert [ts.slots(ts.t_k(k)) for k in range(1, 6)] == [1, 2, 3, 4, 5]
    for n, k in ((22, 3), (23, 4), (46, 4), (47, 5), (64, 5)):
        assert ts.slots(ts.stack_extremal(n)) == k == ts.stack_depth(n)
    for n in range(5, 65):
        assert ts.program_length(ts.longest_program(n)) == n + (n - 1) // 2 - 1
        for name, p in ts.shape_batch(n):
            assert ts.slots(p) <= ts.stack_depth(n), (n, name)  # a subtree needing k slots has >= 3 * 2^(k-1) - 1 vertices
            assert ts.program_length(p) <= n + (n - 1) // 2 - 1, (n, name)
    assert ts.program_length(ts.longest_program(64)) == 94


def test_relabel_and_pruefer():
    rng = np.random.default_rng(4)
    for n in (5, 23, 64):
        for f in ts.FAMILIES.values():
            p = f(n)
            q = ts.relabel(p, rng)
            assert all(q[v] < v for v in range(1, n)) and observe.tree_code(q) == observe.tree_code(p)
    # 125 labelled trees on 5 vertices: 5 stars, 60 paths, 60 of the third shape
    counts = {}
    for _ in range(3000):
        code = observe.tree_code(ts.random_tree(5, rng))
        counts[code] = counts.get(code, 0) + 1
    got = sorted(counts.values())
    assert len(got) == 3 and abs(got[0] - 120) < 40 and all(abs(c - 1440) < 150 for c in got[1:])


def test_oracle_mirror_within_4_ulp_of_exact(orc):
    """LAMBDA_MULTISECTION (the matching polynomial up to 22 vertices, sectioning beyond, as the kernel) against the
    exact lambda_1.  Measured worst: 0.66 ulp for the polynomial method, 2.3 ulp for sectioning; with 9 section rounds
    instead of 11 the worst is 44 ulp, which the 1e-12 check against LAPACK cannot see."""
    worst = {}
    for n, name, p in _all_inputs():
        lam, mu, _, rc = orc.cost(p, method=orc.LAMBDA_MULTISECTION)
        u = ts.ulps(lam, p)
        assert rc == 0 and u <= 4.0, (n, name, p.tolist(), u)
        assert mu == ts.exact_mu(p)
        worst[n <= 22] = max(worst.get(n <= 22, 0.0), u)
    assert worst[True] < 1.0  # the polynomial method is within one ulp
