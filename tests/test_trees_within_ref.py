"""The plain restatement of azb_trees_within (trees_within_ref.py) on the CPU: growing leaf by leaf gives exactly the
classes a filter over every free tree gives, the known count at 19 vertices, and the canonical decode of a code.  No
kernel is launched here."""
import numpy as np
import pytest

import free_trees_ref as F
import trees_within_ref as W
from azdopt_b200 import observe


@pytest.fixture(scope="module")
def cost(orc):
    def f(parents):
        lam, mu, _, rc = orc.cost(parents, method=orc.LAMBDA_MULTISECTION)
        assert rc == 0
        return lam, mu

    return f


@pytest.mark.parametrize("n", range(5, 15))
def test_growth_equals_a_filter_over_every_tree(cost, n):
    every = {}
    for p in F.free_trees(n, 0, F.free_tree_count(n)):
        code = observe.tree_code(p)
        every[code] = W.key_of(cost, W.decode(code, n))
    assert len(every) == F.free_tree_count(n)
    star = W.star_key(cost, n)
    for bound in (star - 0.3, star, star + 0.5, star + 1.5, 0.0):
        want = sorted((k, c) for c, k in every.items() if k <= bound)
        got, sizes, _ = W.trees_within(n, bound, cost)
        assert got == want, bound
        assert sizes[-1] == len(want) or (not want and min(sizes) == 0)


def test_nineteen_vertices_at_the_stars_key(cost):
    star = W.star_key(cost, 19)
    got, _, _ = W.trees_within(19, star, cost)
    assert len(got) == 3 and sum(k < star for k, _ in got) == 2
    assert got[-1] == (star, observe.tree_code([0] * 19))  # the star itself closes the set


@pytest.mark.parametrize("n", [5, 8, 11, 12, 24, 40, 64])
def test_decode_is_canonical(n):
    rng = np.random.default_rng(n)
    rows = F.free_trees(n, 0, F.free_tree_count(n)) if n <= 12 else [
        np.array([0] + [int(rng.integers(0, v)) for v in range(1, n)], dtype=np.uint8) for _ in range(300)]
    for p in rows:
        code = observe.tree_code(p)
        q = W.decode(code, n)
        assert all(q[v] < v for v in range(1, n))
        assert observe.tree_code(q) == code
        assert W.decode(observe.tree_code(q), n).tolist() == q.tolist()
