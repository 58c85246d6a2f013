"""azb_certify_keys (include/azb.h) on the GPU: bit for bit the CPU restatement (certify_oracle.cpp) at the tree shapes
of every N from 5 to 64 and on 65 536 relabelled trees at N = 64; the refusals, NULL outputs, the read-only property and
the scratch being counted."""
import ctypes as C
import math

import numpy as np
import pytest

import certify_oracle as co
import tree_shapes as ts

pytestmark = pytest.mark.gpu


def _handle(capi, n, b=1, **kw):
    return capi.Handle(capi.default_config(n, b, **kw))


def _same(got, want, where):
    for name in ("lambda1_lo", "lambda1_hi"):
        assert np.array_equal(got[name].view(np.uint64), want[name].view(np.uint64)), f"{where}: {name}"
    assert np.array_equal(got["mu"], want["mu"]), f"{where}: mu"
    assert np.array_equal(got["verdict"], want["verdict"]), f"{where}: verdict"


@pytest.mark.parametrize("n", range(5, 65))
def test_equals_the_restatement(capi, n):
    parents = np.stack([p for _, p in ts.shape_batch(n)])
    with _handle(capi, n) as h:
        lam, mu, _, _ = h.eval_costs(parents)
        star = float(mu[0]) + float(lam[0])  # shape_batch starts with the star: its computed key, a bound >= 0
        for bound in (None, star, star + 0.5, math.nextafter(star, math.inf)):
            got = h.certify_keys(parents, bound)
            want = co.certify(parents, lam, -1.0 if bound is None else bound)
            _same(got, want, f"n {n} bound {bound!r}")
            assert np.array_equal(got["mu"], mu)  # the greedy matching is exact
        d = h.certify_keys(parents)
        assert d["verdict"][0] == 0  # the star ties sqrt(N - 1) + 1
        assert np.all(d["lambda1_lo"] < lam) and np.all(lam < d["lambda1_hi"])


def test_relabelled_trees_at_64(capi):
    n, m = 64, 65536
    rng = np.random.default_rng(64)
    base = [p for _, p in ts.shape_batch(n)]
    parents = np.stack([ts.relabel(base[i % len(base)], rng) for i in range(m)])
    with _handle(capi, n) as h:
        lam, _, _, _ = h.eval_costs(parents)
        got = h.certify_keys(parents)
        _same(got, co.certify(parents, lam), "relabelled")
        # the verdict is a function of the tree, whatever the labelling
        codes = h.tree_codes(parents)
        by_class = {}
        for c, v in zip(map(tuple, codes.tolist()), got["verdict"].tolist()):
            if v != 2:
                by_class.setdefault(c, set()).add(v)
        assert all(len(s) == 1 for s in by_class.values())


def test_refusals(capi):
    n = 12
    good = np.stack([ts.path(n), ts.star(n)])
    with _handle(capi, n) as h:
        with pytest.raises(capi.AzbError) as e:
            h.certify_keys(good, math.nan)
        assert e.value.code == capi.ERR_INVALID
        bad = good.copy()
        bad[1, 5] = 7
        with pytest.raises(capi.AzbError) as e:
            h.certify_keys(bad)
        assert e.value.code == capi.ERR_INVALID and "tree 1" in str(e.value)
        L = capi.lib()
        assert L.azb_certify_keys(h._h, good.ctypes.data_as(C.POINTER(C.c_uint8)), 0, -1.0, None, None, None, None, None) \
            == capi.ERR_INVALID
        assert L.azb_certify_keys(None, good.ctypes.data_as(C.POINTER(C.c_uint8)), 2, -1.0, None, None, None, None, None) \
            == capi.ERR_INVALID
        assert L.azb_certify_keys(h._h, None, 2, -1.0, None, None, None, None, None) == capi.ERR_INVALID


def test_null_outputs(capi):
    n = 20
    parents = np.stack([p for _, p in ts.shape_batch(n)])
    with _handle(capi, n) as h:
        full = h.certify_keys(parents)
        L = capi.lib()
        u8 = parents.ctypes.data_as(C.POINTER(C.c_uint8))
        assert L.azb_certify_keys(h._h, u8, len(parents), -1.0, None, None, None, None, None) == 0
        v = np.zeros(len(parents), dtype=np.int8)
        assert L.azb_certify_keys(h._h, u8, len(parents), -1.0, None, None, None, v.ctypes.data_as(C.POINTER(C.c_int8)),
                                  None) == 0
        assert np.array_equal(v, full["verdict"])


def test_read_only_and_scratch_counted(capi):
    n, b = 30, 64
    cfg = capi.default_config(n, b, prior_mode=capi.PRIOR_HASH, prior_seed=3, max_steps=400)
    with capi.Handle(cfg) as a, capi.Handle(cfg) as c:
        for x in (a, c):
            p, m = capi.generate_roots(3, 0, b, n)
            x.set_roots(p, m)
            x.init_trees()
        ia, ic = a.step(40), c.step(40)
        before = a.checkpoint_save().copy()
        m = 50000
        trees = capi.generate_roots(5, 0, m, n)[0]
        a.certify_keys(trees)
        # parents, lambda1, mu, c, lambda1_lo, lambda1_hi, mu, verdict of every tree
        assert a.device_bytes() - c.device_bytes() >= m * (n + 8 + 4 + 4 + 8 + 8 + 4 + 1)
        assert np.array_equal(a.checkpoint_save(), before)
        wa, wc = a.walkers(), c.walkers()
        for key in wa:
            assert np.array_equal(wa[key], wc[key]), key
        assert a.step(60) == c.step(60) and ia == ic
        assert a.argmin()["eval"] == c.argmin()["eval"] and a.counters() == c.counters()
