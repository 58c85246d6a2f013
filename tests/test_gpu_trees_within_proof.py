"""azb_trees_within_proof (include/azb.h) on the GPU: its outputs are bit for bit azb_trees_within's, its proof words
are the verdicts azb_certify_keys gives the returned classes, counted once each, they agree with an exact
classification of the returned classes for N <= 24, and the counts of the project's headline results are proven
(N = 19 and N = 64 against sqrt(N - 1) + 1).

Where N - 1 is a square the bound sqrt(N - 1) + 1 is an integer, and another tree can tie it exactly: at N = 17 two
stars K1,7 whose centres are joined through a middle vertex (lambda_1 = 3, mu = 2), at N = 26 the double star with 12
and 12 leaves (lambda_1 = 4, mu = 2).  Only the star's tie is decided, so these stay open."""
import numpy as np
import pytest

import certify_oracle as co

pytestmark = pytest.mark.gpu

WORDS = ("below", "equal", "above", "open", "unproven_pruned")


def _handle(capi, n):
    return capi.Handle(capi.default_config(n, 1))


def _same(a, b):
    for name in ("code", "parents", "lambda1", "mu", "eval"):
        assert np.array_equal(a[name].view(np.uint8), b[name].view(np.uint8)), name
    assert (a["n_within"], a["n_below"]) == (b["n_within"], b["n_below"])


def _run(h, bound=None):
    plain = h.trees_within(bound, k=65536)
    proved = h.trees_within(bound, k=65536, prove=True)
    _same(plain, proved)
    pf = proved["proof"]
    assert sum(pf[w] for w in WORDS[:4]) == proved["n_within"] <= 65536
    v = h.certify_keys(proved["parents"], bound)["verdict"]
    assert [pf[w] for w in WORDS[:4]] == [int(np.sum(v == x)) for x in (-1, 0, 1, 2)]
    return proved, pf, v


def _tie(n):
    """The tree on n = 17 or 26 vertices other than the star whose key is sqrt(n - 1) + 1 exactly."""
    p = np.zeros(n, dtype=np.uint8)
    if n == 17:  # centres 0 and 2, joined through 1, with 7 leaves each
        p[2], p[10:] = 1, 2
    else:  # centres 0 and 1 with 12 leaves each
        p[14:] = 1
    return p


@pytest.mark.parametrize("n", list(range(8, 25)))
def test_equals_trees_within_and_the_exact_classification(capi, n):
    with _handle(capi, n) as h:
        r, pf, v = _run(h)
        for p, got in zip(r["parents"], v.tolist()):
            exact = co.exact_sign(p, -1.0)
            assert got == exact or (got == 2 and exact == 0), (p.tolist(), got, exact)  # only exact ties stay open
        assert pf["equal"] == 1 and pf["above"] == 0 and pf["unproven_pruned"] == 0
        assert pf["open"] == (1 if n == 17 else 0)


def test_exact_ties_stay_open(capi):
    for n in (17, 26):
        tie = _tie(n)
        assert co.exact_sign(tie, -1.0) == 0
        with _handle(capi, n) as h:
            assert h.certify_keys(tie[None])["verdict"][0] == 2
            r, pf, v = _run(h)
            code = h.tree_codes(tie[None])[0]
            assert [i for i in range(len(v)) if v[i] == 2] == [i for i, c in enumerate(r["code"]) if np.array_equal(c, code)]


@pytest.mark.parametrize("n", [26, 33, 40, 48])
def test_equals_trees_within(capi, n):
    with _handle(capi, n) as h:
        _, pf, _ = _run(h)
        assert pf["equal"] == 1 and pf["above"] == 0 and pf["unproven_pruned"] == 0
        assert pf["open"] == (1 if n == 26 else 0)


def test_star_plus_half_and_chunks(capi, monkeypatch):
    n = 26
    with _handle(capi, n) as h:
        lam, mu, _, _ = h.eval_costs(np.zeros((1, n), dtype=np.uint8))
        bound = float(mu[0]) + float(lam[0]) + 0.5
        whole, pw, _ = _run(h, bound)
    monkeypatch.setenv("AZB_TEST_GROW_CHUNK", "97")
    with _handle(capi, n) as h:
        part, pp, _ = _run(h, bound)
        _same(part, whole)
        # result classes are counted once each whatever the chunks; a dropped class met in several chunks counts in each
        assert [pp[w] for w in WORDS[:4]] == [pw[w] for w in WORDS[:4]]
        assert pp["unproven_pruned"] >= pw["unproven_pruned"]


def test_n19_proves_two_below_and_the_star(capi):
    with _handle(capi, 19) as h:
        _, pf, _ = _run(h)
        assert pf == dict(below=2, equal=1, above=0, open=0, unproven_pruned=0)


def test_n64_headline(capi):
    with _handle(capi, 64) as h:
        r, pf, _ = _run(h)
        assert (r["n_within"], r["n_below"]) == (27618, 27617)
        assert pf == dict(below=27617, equal=1, above=0, open=0, unproven_pruned=0)


def test_refusals(capi):
    with _handle(capi, 20) as h:
        for kw in (dict(k=0), dict(k=65537), dict(bound=float("nan"))):
            with pytest.raises(capi.AzbError) as e:
                h.trees_within(**{"k": 10, **kw}, prove=True)
            assert e.value.code == capi.ERR_INVALID, kw
