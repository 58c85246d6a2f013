"""azb_trees_within (include/azb.h) on the GPU: against the exhaustive ranking (N = 8 .. 24), against the plain
restatement (trees_within_ref.py, N = 33 and 40), self-consistency and agreement with the search at 48 and 64 vertices,
chunked growth, the refusals, the capacity limit, and the read-only property."""
import math

import numpy as np
import pytest

import trees_within_ref as W

pytestmark = pytest.mark.gpu


def _handle(capi, n, b=1, **kw):
    return capi.Handle(capi.default_config(n, b, **kw))


def _star_key(h):
    lam, mu, _, _ = h.eval_costs(np.zeros((1, h.n), dtype=np.uint8))
    return float(mu[0]) + float(lam[0])


def _keys(r):
    return r["mu"].astype(np.float64) + r["lambda1"]


def _codes(r):
    return [tuple(int(x) for x in c) for c in r["code"]]


def _self_consistent(h, r):
    """Every entry is what azb_eval_costs / azb_tree_codes give for its canonical parents, in (key, code) order."""
    n = len(r["mu"])
    assert n == min(r["n_within"], len(r["code"]))
    par = r["parents"]
    assert all(int(p[v]) < v for p in par for v in range(1, h.n))
    lam, mu, ev, _ = h.eval_costs(par)
    assert np.array_equal(lam.view(np.uint64), r["lambda1"].view(np.uint64))
    assert np.array_equal(mu, r["mu"]) and np.array_equal(ev.view(np.uint32), r["eval"].view(np.uint32))
    assert np.array_equal(h.tree_codes(par), r["code"])
    for p, c in zip(par, r["code"]):
        assert W.decode(c, h.n).tolist() == p.tolist()
    order = sorted(zip(_keys(r).tolist(), _codes(r)))
    assert order == list(zip(_keys(r).tolist(), _codes(r)))
    assert len(set(_codes(r))) == n


def _against_exhaustive(h, bound, exact):
    """trees_within(bound) against azb_exhaustive_best over the whole range, filtered to key <= bound."""
    ex = h.exhaustive_best(k=65536, bound=bound)
    le = h.exhaustive_best(k=1, bound=float(np.nextafter(bound, np.inf)))["n_below"]  # keys <= bound
    w = h.trees_within(bound, k=65536)
    _self_consistent(h, w)
    assert w["n_within"] == le and w["n_below"] == ex["n_below"]
    kex = _keys(ex)
    sel = kex <= bound
    if le > 65536:  # the exhaustive list is cut: compare the classes strictly ahead of its last key
        sel = kex < kex[-1]
        wsel = _keys(w) < kex[-1]
    else:
        wsel = np.ones(len(w["mu"]), dtype=bool)
    assert int(sel.sum()) == int(wsel.sum())
    want = {tuple(int(x) for x in c): i for i, c in enumerate(h.tree_codes(ex["parents"][sel]))}
    got = {c: i for i, c in enumerate(_codes(w)) if wsel[i]}
    assert set(want) == set(got)
    lam_ex, mu_ex, ev_ex = ex["lambda1"][sel], ex["mu"][sel], ex["eval"][sel]
    for c, i in got.items():
        j = want[c]
        assert w["mu"][i] == mu_ex[j]
        if exact:  # up to 22 vertices lambda1 does not depend on the labelling
            assert w["lambda1"][i].view(np.uint64) == lam_ex[j].view(np.uint64)
            assert w["eval"][i].view(np.uint32) == ev_ex[j].view(np.uint32)
        else:
            assert abs(w["lambda1"][i] - lam_ex[j]) <= 1e-12 * lam_ex[j]
    return w


@pytest.mark.parametrize("n", range(8, 23))
def test_equals_the_exhaustive_ranking(capi, n):
    with _handle(capi, n) as h:
        star = _star_key(h)
        for off in (0.0, 0.5, 1.5):
            w = _against_exhaustive(h, star + off, exact=True)
            if off == 0.0:  # the default bound is the star's key, and the star is in the set
                d = h.trees_within(k=65536)
                assert _codes(d) == _codes(w) and (d["n_within"], d["n_below"]) == (w["n_within"], w["n_below"])
                assert [0] * n in d["parents"].tolist()


def _clear_bound(h, target):
    """A bound near target that no key comes within 1e-9 of (checked with the exhaustive counts)."""
    for b in (target, target + 0.0371, target - 0.0413, target + 0.0837):
        lo = h.exhaustive_best(k=1, bound=b - 1e-9)["n_below"]
        hi = h.exhaustive_best(k=1, bound=b + 1e-9)["n_below"]
        if lo == hi:
            return b
    raise AssertionError(f"no clear bound near {target}")


@pytest.mark.parametrize("n", [23, 24])
def test_equals_the_exhaustive_ranking_with_the_section_method(capi, n):
    with _handle(capi, n) as h:
        star = _star_key(h)
        for off in (0.25, 0.5, 1.0):
            _against_exhaustive(h, _clear_bound(h, star + off), exact=False)


@pytest.fixture(scope="module")
def oracle_cost(orc):
    def f(parents):
        lam, mu, _, rc = orc.cost(parents, method=orc.LAMBDA_MULTISECTION)
        assert rc == 0
        return lam, mu

    return f


@pytest.mark.parametrize("n", [33, 40])
def test_equals_the_restatement(capi, oracle_cost, n):
    with _handle(capi, n) as h:
        star = _star_key(h)
        assert star == W.star_key(oracle_cost, n)
        want, _, _ = W.trees_within(n, star, oracle_cost)
        got = h.trees_within(k=65536)
        _self_consistent(h, got)
        assert got["n_within"] == len(want) and got["n_below"] == sum(k < star for k, _ in want)
        assert [(k, c) for k, c in zip(_keys(got).tolist(), _codes(got))] == want


def _hash_handle(capi, n, b, seed=0, **kw):
    h = capi.Handle(capi.default_config(n, b, prior_mode=capi.PRIOR_HASH, prior_seed=seed, max_steps=400, **kw))
    p, m = capi.generate_roots(seed, 0, b, n)
    h.set_roots(p, m)
    h.init_trees()
    return h


@pytest.mark.parametrize("n,offset", [(48, 0.5), (64, 0.0)])
def test_large_n_is_consistent_with_the_cost_and_the_search(capi, n, offset):
    with _hash_handle(capi, n, 64, seed=n) as h:
        h.step(200)
        bound = _star_key(h) + offset
        w = h.trees_within(bound, k=65536)
        _self_consistent(h, w)
        assert w["n_within"] <= 65536  # the whole set came back
        assert np.all(_keys(w) <= bound) and w["n_below"] == int(np.sum(_keys(w) < bound))
        codes = set(_codes(w))
        assert tuple(int(x) for x in h.tree_codes(np.zeros((1, n), dtype=np.uint8))[0]) in codes  # the star
        best = h.best_trees(200)
        lam, mu, _, _ = h.eval_costs(best["parents"])
        for c, key in zip(best["code"], mu.astype(np.float64) + lam):
            if key <= bound - 1e-9:  # keys within a few ulps of the bound may fall on either side between labellings
                assert tuple(int(x) for x in c) in codes


def test_chunks_and_merges_give_the_same_result(capi, monkeypatch):
    n = 26
    with _handle(capi, n) as h:
        star = _star_key(h)
        whole = h.trees_within(star + 0.5, k=65536)
    monkeypatch.setenv("AZB_TEST_GROW_CHUNK", "97")
    with _handle(capi, n) as h:
        part = h.trees_within(star + 0.5, k=65536)
        for name in ("code", "parents", "lambda1", "mu", "eval"):
            assert np.array_equal(part[name], whole[name]), name
        assert (part["n_within"], part["n_below"]) == (whole["n_within"], whole["n_below"])
        small = h.trees_within(star + 0.5, k=3)
        assert _codes(small) == _codes(whole)[:3] and small["n_within"] == whole["n_within"]


def test_refusals_and_the_capacity_limit(capi):
    with _handle(capi, 20) as h:
        for kw in (dict(k=0), dict(k=65537), dict(bound=math.nan)):
            with pytest.raises(capi.AzbError) as e:
                h.trees_within(**{"k": 10, **kw})
            assert e.value.code == capi.ERR_INVALID, kw
        full = h.trees_within(k=10)
        with pytest.raises(capi.AzbError) as e:
            h.trees_within(k=10, max_level=4)
        assert e.value.code == capi.ERR_CAPACITY and "level" in str(e.value) and "more than 4 classes" in str(e.value)
        again = h.trees_within(k=10)  # the refused call left nothing behind
        assert _codes(again) == _codes(full) and again["n_within"] == full["n_within"]
        none = h.trees_within(1.0, k=10)  # below every key
        assert none["n_within"] == 0 and len(none["code"]) == 0


def test_a_call_between_steps_changes_nothing(capi):
    n, b = 30, 64
    with _hash_handle(capi, n, b, seed=3) as a, _hash_handle(capi, n, b, seed=3) as c:
        ia, ic = a.step(40), c.step(40)
        before = a.checkpoint_save().copy()
        got = a.trees_within(k=500)
        assert got["n_within"] >= 1
        assert np.array_equal(a.checkpoint_save(), before)
        wa, wc = a.walkers(), c.walkers()
        for key in wa:
            assert np.array_equal(wa[key], wc[key]), key
        ga, gc = a.argmin(), c.argmin()
        assert ga["parents"].tolist() == gc["parents"].tolist() and ga["eval"] == gc["eval"]
        assert a.step(60) == c.step(60) and ia == ic
        assert a.argmin()["eval"] == c.argmin()["eval"]
        assert a.counters() == c.counters()
