"""azb_free_trees and azb_exhaustive_best (include/azb.h) on the GPU: the enumeration byte for byte against its plain
restatement (free_trees_ref.py), the k best against a CPU ranking with the oracle's cost, chunking and sharding, the
refusals, the read-only property, and consistency with what the search finds."""
import functools
import math

import numpy as np
import pytest

import free_trees_ref as R
from azdopt_b200 import shard

pytestmark = pytest.mark.gpu


def _handle(capi, n, b=1, **kw):
    return capi.Handle(capi.default_config(n, b, **kw))


@functools.lru_cache(maxsize=None)
def _ranked(n, start, count, orc):
    """CPU ranking of [start, start + count): rows, lambda1, mu, eval (the oracle's LAMBDA_MULTISECTION, the method the
    parity tests use) and the order by (mu + lambda1, index)."""
    rows = R.free_trees(n, start, count)
    lam = np.zeros(count, np.float64)
    mu = np.zeros(count, np.uint32)
    ev = np.zeros(count, np.float32)
    for i, p in enumerate(rows):
        lam[i], mu[i], ev[i], rc = orc.cost(p, method=orc.LAMBDA_MULTISECTION)
        assert rc == 0
    key = mu.astype(np.float64) + lam
    return rows, lam, mu, ev, key, np.lexsort((np.arange(count), key))


def _check(orc, got, n, start, count, k):
    rows, lam, mu, ev, key, order = _ranked(n, start, count, orc)
    top = order[:min(k, count)]
    assert np.array_equal(got["index"], (start + top).astype(np.uint64))
    assert np.array_equal(got["parents"], rows[top])
    assert np.array_equal(got["lambda1"].view(np.uint64), lam[top].view(np.uint64))
    assert np.array_equal(got["mu"], mu[top])
    assert np.array_equal(got["eval"].view(np.uint32), ev[top].view(np.uint32))
    assert got["n_below"] == int(np.sum(key < math.sqrt(n - 1) + 1))


def _same(a, b):
    for name in ("index", "parents", "lambda1", "mu", "eval"):
        assert np.array_equal(np.asarray(a[name]).view(np.uint8), np.asarray(b[name]).view(np.uint8)), name
    assert a["n_below"] == b["n_below"]


@pytest.mark.parametrize("n", range(5, 17))
def test_free_trees_whole_range(capi, n):
    total = capi.free_tree_count(n)
    with _handle(capi, n) as h:
        assert np.array_equal(h.free_trees(0, total), R.free_trees(n, 0, total))


@pytest.mark.parametrize("n", [19, 24, 30, 32])
def test_free_trees_windows(capi, n):
    total, u, w = R.free_tree_count(n), R.unicentroidal_count(n), 1500
    with _handle(capi, n) as h:
        before = h.device_bytes()
        for s in sorted({0, total - w, max(u - w // 2, 0)}):
            m = min(w, total - s)
            assert np.array_equal(h.free_trees(s, m), R.free_trees(n, s, m)), s
        assert h.device_bytes() > before  # the tables count in azb_device_bytes


def test_free_trees_straddle_chunk_boundaries(capi, monkeypatch):
    monkeypatch.setenv("AZB_TEST_ENUM_CHUNK", "1000")
    n = 20
    with _handle(capi, n) as h:
        for s, m in ((500, 3700), (999, 2), (0, 1), (7000, 1001)):
            assert np.array_equal(h.free_trees(s, m), R.free_trees(n, s, m)), (s, m)


@pytest.mark.parametrize("n", range(8, 20))
def test_exhaustive_best_whole_range(capi, orc, n):
    total = capi.free_tree_count(n)
    with _handle(capi, n) as h:
        for k in (1000, min(total + 5, 65536)):
            got = h.exhaustive_best(k=k)
            assert len(got["index"]) == min(k, total)
            _check(orc, got, n, 0, total, k)


@pytest.mark.parametrize("n,where", [(23, "middle"), (24, "centroids")])
def test_exhaustive_best_windows_with_the_section_method(capi, orc, n, where):
    total, u, w = R.free_tree_count(n), R.unicentroidal_count(n), 200_000
    start = total // 3 if where == "middle" else u - w // 2  # at 24: straddles the bicentroidal trees
    with _handle(capi, n) as h:
        got = h.exhaustive_best(start, w, k=2000)
    _check(orc, got, n, start, w, 2000)


def test_chunks_and_uneven_shards_equal_one_call(capi, monkeypatch):
    n, k = 16, 300
    total = capi.free_tree_count(n)
    with _handle(capi, n) as h:
        whole = h.exhaustive_best(k=k)
    monkeypatch.setenv("AZB_TEST_ENUM_CHUNK", "777")
    with _handle(capi, n) as h:
        _same(h.exhaustive_best(k=k), whole)
        cuts = [0, 5, 4000, 4001, 12000, total]
        parts = [h.exhaustive_best(a, b - a, k=k) for a, b in zip(cuts, cuts[1:])]
        _same(shard.merge_exhaustive_best(parts, k), whole)
        _same(shard.global_exhaustive_best(h.exhaustive_best(k=k), k), whole)  # one rank: the local result
        small = h.exhaustive_best(k=1)
        assert small["index"].tolist() == whole["index"][:1].tolist()


def test_refusals(capi):
    with _handle(capi, 12) as h:
        total = capi.free_tree_count(12)
        for kw in (dict(k=0), dict(k=65537), dict(count=0), dict(start=total, count=1), dict(start=total - 3, count=4),
                   dict(start=total + 10, count=1)):
            with pytest.raises(capi.AzbError) as e:
                h.exhaustive_best(**{"k": 10, **kw})
            assert e.value.code == capi.ERR_INVALID, kw
        for s, m in ((total, 1), (total - 1, 2), (0, 0)):
            with pytest.raises(capi.AzbError) as e:
                h.free_trees(s, m)
            assert e.value.code == capi.ERR_INVALID
        assert len(h.exhaustive_best(total - 3, 3, k=65536)["index"]) == 3
    with _handle(capi, 40) as h:
        for call in (lambda: h.exhaustive_best(0, 10, k=5), lambda: h.free_trees(0, 4)):
            with pytest.raises(capi.AzbError) as e:
                call()
            assert e.value.code == capi.ERR_INVALID


def _hash_handle(capi, n, b, seed=0, **kw):
    h = capi.Handle(capi.default_config(n, b, prior_mode=capi.PRIOR_HASH, prior_seed=seed, max_steps=400, **kw))
    p, m = capi.generate_roots(seed, 0, b, n)
    h.set_roots(p, m)
    h.init_trees()
    return h


def test_a_call_between_steps_changes_nothing(capi):
    n, b = 19, 64
    with _hash_handle(capi, n, b, seed=3) as a, _hash_handle(capi, n, b, seed=3) as c:
        ia, ic = a.step(40), c.step(40)
        got = a.exhaustive_best(0, 50_000, k=500)
        assert len(got["index"]) == 500
        wa, wc = a.walkers(), c.walkers()
        for key in wa:
            assert np.array_equal(wa[key], wc[key]), key
        ga, gc = a.argmin(), c.argmin()
        assert ga["parents"].tolist() == gc["parents"].tolist() and ga["eval"] == gc["eval"]
        assert a.step(60) == c.step(60) and ia == ic
        assert a.argmin()["eval"] == c.argmin()["eval"]
        assert a.counters() == c.counters()


@pytest.mark.parametrize("n,b,steps", [(10, 32, 300), (19, 256, 300)])
def test_consistent_with_the_search(capi, n, b, steps):
    total = capi.free_tree_count(n)
    with _hash_handle(capi, n, b, seed=n) as h:
        h.step(steps)
        best = h.best_trees(50)
        ex = h.exhaustive_best(k=1)
        rows = h.free_trees(0, total)
        _, _, ev, _ = h.eval_costs(rows)
        codes = {tuple(int(x) for x in c): i for i, c in enumerate(h.tree_codes(rows))}
        assert len(codes) == total
        for code, e in zip(best["code"], best["eval"]):
            i = codes[tuple(int(x) for x in code)]
            assert ev[i].view(np.uint32) == np.float32(e).view(np.uint32)  # up to 22 vertices the cost is label-free
        assert h.argmin()["eval"] >= ex["eval"][0]
