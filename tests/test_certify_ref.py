"""The CPU restatement of the c21 key certificates (certify_oracle.cpp, bit-identical to azb_certify_keys) against exact
arithmetic, at the tree shapes of tree_shapes.shape_batch for every N from 5 to 64, with the oracle's mirror of the
cost kernel's lambda_1 as the starting point c.

A certificate may fail to decide (verdict 2, open); it may never be wrong.  The share of open verdicts is recorded, with
no threshold."""
import math
from fractions import Fraction

import numpy as np
import pytest

import certify_oracle as co
import tree_shapes as ts
import trees_within_ref as W

OPEN = {}


def _batch(orc, n):
    batch = ts.shape_batch(n)
    parents = np.stack([p for _, p in batch])
    c = np.array([orc.cost(p, method=orc.LAMBDA_MULTISECTION)[0] for p in parents])
    return batch, parents, c


def _key_rounded(p):
    """The binary64 nearest to mu + lambda_1."""
    _, lo, hi = ts.exact_lambda1(p)
    return float(ts.exact_mu(p) + (lo + hi) / 2)


@pytest.mark.parametrize("n", range(5, 65))
def test_certificates_are_right(orc, n, record_property):
    batch, parents, c = _batch(orc, n)
    out = co.certify(parents, c)
    n_open = n_checked = 0
    for i, (name, p) in enumerate(batch):
        where = f"n {n} {name} row {i}"
        _, elo, ehi = ts.exact_lambda1(p)
        mu = int(out["mu"][i])
        assert mu == ts.exact_mu(p), where
        lo, hi = out["lambda1_lo"][i], out["lambda1_hi"][i]
        assert Fraction(lo) <= elo and Fraction(hi) > ehi, f"{where}: ({lo!r}, {hi!r}) does not enclose lambda_1"
        # every decided count is the exact count at that point
        t_lo, t_hi = co.points(n, mu, -1.0)
        d0 = math.ulp(c[i])
        for x in (lo, hi, t_lo, t_hi, c[i] - d0, c[i] + d0, c[i] - 16 * d0, c[i] + 16 * d0):
            k = co.jt(p, x)
            if k >= 0:
                assert k == co.above(p, x), f"{where}: JT at {x!r} counts {k}"
        # verdicts: the default bound, and the doubles one ulp either side of the correctly rounded key
        key = _key_rounded(p)
        for bound in (-1.0, math.nextafter(key, -math.inf), math.nextafter(key, math.inf)):
            v = int(out["verdict"][i]) if bound < 0 else int(co.certify(p[None], c[i:i + 1], bound)["verdict"][0])
            n_checked += 1
            if v == 2:
                n_open += 1
                continue
            want = co.exact_sign(p, bound)
            assert want is not None and v == want, f"{where}: verdict {v} against {bound!r}, exact {want}"
    OPEN[n] = (n_open, n_checked)
    record_property("open_verdicts", f"{n_open}/{n_checked}")
    print(f"n {n}: {n_open} of {n_checked} verdicts open")


def test_star_and_points():
    """The star ties the default bound (verdict 0); the bound points enclose sqrt(N - 1) + 1 - mu."""
    for n in (5, 10, 17, 19, 26, 64):
        s = ts.star(n)
        out = co.certify(s[None], np.array([math.sqrt(n - 1)]))
        assert out["verdict"][0] == 0 and out["mu"][0] == 1
        # a bound >= 0 ties the star only when (bound - 1)^2 = n - 1
        b = math.sqrt(n - 1) + 1.0
        v = int(co.certify(s[None], np.array([math.sqrt(n - 1)]), b)["verdict"][0])
        if math.isqrt(n - 1) ** 2 == n - 1:
            assert v == 0
        else:
            assert v == co.exact_sign(s, b) or v == 2
        for mu in (1, 2, 7):
            t_lo, t_hi = co.points(n, mu, -1.0)
            s_lo, s_hi = Fraction(t_lo) - 1 + mu, Fraction(t_hi) - 1 + mu  # around sqrt(n - 1)
            assert s_lo * s_lo <= n - 1 <= s_hi * s_hi and s_lo > 0
            assert t_hi - t_lo <= 4 * math.ulp(t_hi + mu)


def test_greedy_mu_is_exact_on_random_trees():
    rng = np.random.default_rng(7)
    for n in (5, 9, 19, 33, 64):
        for _ in range(40):
            p = ts.random_tree(n, rng)
            assert co.greedy_mu(p) == ts.exact_mu(p)


@pytest.fixture(scope="module")
def cost(orc):
    def f(parents):
        lam, mu, _, rc = orc.cost(parents, method=orc.LAMBDA_MULTISECTION)
        assert rc == 0
        return lam, mu

    return f


def test_dropped_classes_are_proven_only_when_above(cost):
    """The grow side of azb_trees_within_proof, restated: a class the keep test drops counts as proven above the bound
    only when it is, also when c is far from lambda_1 (the keep test then drops classes within the bound)."""
    n_proven = n_decided_zero = 0
    for p, c, mu, thr, bound, n in co.pruned_cases(cost):
        if co.unproven(p, c, mu, thr, bound, n):
            continue
        n_proven += 1
        want = co.exact_sign(p, bound)
        assert want == 1, (p.tolist(), c, bound, want)
    for p, c, mu, thr, bound, n in co.pruned_cases(cost):
        if co.jt(p, co.points(n, co.greedy_mu(p), bound)[1]) == 0:  # lambda_1 < t_hi proven: within the bound
            n_decided_zero += 1
            assert co.unproven(p, c, mu, thr, bound, n)
    assert n_proven > 0 and n_decided_zero > 0  # both sides of the decision occur


def test_grown_dropped_classes(cost):
    """Along the growth of trees_within_ref, a dropped class is left unproven where the binary64 filter dropped a tree
    within the bound: at N = 24 one double below the star's computed key, the star (whose computed key lies above the
    next double of its true key) is such a tree."""
    n = 24
    star = W.star_key(cost, n)
    bound = math.nextafter(star, -math.inf)
    assert co.exact_sign(ts.star(n), bound) == -1  # the true key sqrt(23) + 1 is below the bound
    classes, unproven, dropped = co.grow_with_proof(n, bound, cost)
    assert unproven == 1
    assert [p.tolist() for p, _, _, u in dropped if u] == [[0] * n]
    for p, _, _, u in dropped:
        if not u:
            assert co.exact_sign(p, bound) == 1
