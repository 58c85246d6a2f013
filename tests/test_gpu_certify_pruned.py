"""The grow side of azb_trees_within_proof on the GPU, the word proof[4] rests on:

- azb_certify_pruned_kernel itself (through tests/certify_kernel_harness.cu, one class per launch) decides every class
  as the CPU restatement does, also for lambda_1 moved far from the truth, and never counts a class as proven above
  the bound unless exact arithmetic agrees;
- proof[4] of the whole call equals the restatement's count along trees_within_ref's growth, and is 1 where the binary64
  filter drops a tree within the bound (N = 24 and 33, one double below the star's computed key: the star);
- with proof[3] = proof[4] = 0, the counts the proof makes a theorem equal an exact count over every free tree
  (N = 10 and 12)."""
import math

import numpy as np
import pytest

import certify_oracle as co
import free_trees_ref as F
import trees_within_ref as W
from azdopt_b200 import observe

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cost(orc):
    def f(parents):
        lam, mu, _, rc = orc.cost(parents, method=orc.LAMBDA_MULTISECTION)
        assert rc == 0
        return lam, mu

    return f


def _handle(capi, n):
    return capi.Handle(capi.default_config(n, 1))


def test_kernel_decides_as_the_restatement_and_soundly(capi, cost):
    cases = co.pruned_cases(cost)
    got = np.zeros(len(cases), dtype=bool)
    # one harness call per (n, bound): the harness takes one bound for all its classes
    groups = {}
    for i, (p, c, mu, thr, bound, n) in enumerate(cases):
        groups.setdefault((n, bound), []).append(i)
    for (n, bound), idx in groups.items():
        got[idx] = co.kernel_unproven(np.stack([cases[i][0] for i in idx]), [cases[i][1] for i in idx],
                                      [cases[i][2] for i in idx], [cases[i][3] for i in idx], bound, n)
    n_open = 0
    for (p, c, mu, thr, bound, n), g in zip(cases, got):
        assert g == co.unproven(p, c, mu, thr, bound, n), (p.tolist(), c, bound)
        if g:
            n_open += 1
        else:
            assert co.exact_sign(p, bound) == 1, (p.tolist(), c, bound)
    assert 0 < n_open < len(cases)


@pytest.mark.parametrize("n", [24, 33])
def test_a_tree_within_the_bound_dropped_by_the_filter_is_left_unproven(capi, cost, n):
    bound = math.nextafter(W.star_key(cost, n), -math.inf)
    star = np.zeros(n, dtype=np.uint8)
    assert co.exact_sign(star, bound) == -1  # sqrt(n - 1) + 1 < bound < the star's computed key
    _, want, dropped = co.grow_with_proof(n, bound, cost)
    assert want == 1 and [p.tolist() for p, _, _, u in dropped if u] == [star.tolist()]
    with _handle(capi, n) as h:
        r = h.trees_within(bound, k=65536, prove=True)
        code = h.tree_codes(star[None])[0]
    assert not any(np.array_equal(c, code) for c in r["code"])  # the filter dropped the star
    assert r["proof"]["unproven_pruned"] == 1  # so the counts are not claimed as a theorem


@pytest.mark.parametrize("n", [10, 12])
def test_the_theorem_against_every_free_tree(capi, cost, n):
    codes = {observe.tree_code(p) for p in F.free_trees(n, 0, F.free_tree_count(n))}
    trees = [W.decode(c, n) for c in codes]
    keys = sorted({W.key_of(cost, p) for p in trees})
    star = W.star_key(cost, n)
    near = sorted(keys, key=lambda k: abs(k - star))[:4]
    bounds = [-1.0] + [b for k in near for b in (math.nextafter(k, -math.inf), k)]
    theorems = 0
    with _handle(capi, n) as h:
        for bound in bounds:
            r = h.trees_within(None if bound < 0 else bound, k=65536, prove=True)
            pf = r["proof"]
            _, want, _ = co.grow_with_proof(n, bound, cost)
            assert pf["unproven_pruned"] == want, bound
            if pf["open"] == 0 and pf["unproven_pruned"] == 0:
                theorems += 1
                signs = [co.exact_sign(p, bound) for p in trees]
                assert None not in signs
                assert r["n_within"] - pf["above"] == sum(s <= 0 for s in signs), bound
                assert pf["below"] == signs.count(-1), bound
    assert theorems >= 1
