"""PUCT selection (include/azb.h, AZB_SELECT_PUCT) on the GPU: bit-exact against the PUCT oracle (tests/puct_oracle.cpp)
in the lock step, and
every other form of the search step (the one-launch hash mode, yielding launches, the asynchronous kernel) against
the lock step."""
import numpy as np
import pytest

from puct_oracle import PuctOptimizer

pytestmark = pytest.mark.gpu

PUCT = dict(selection=1, puct_c=1.0)


def _mk(capi, n, b, **kw):
    return capi.Handle(capi.default_config(n, b, **kw))


def _same_trees(da, db, where):
    for k in ("nodes", "keys", "preds", "arcs"):
        assert da[k].shape == db[k].shape and np.array_equal(da[k], db[k]), f"{where} {k}"


def _same_runs(ha, hb, b):
    for i in range(b):
        _same_trees(ha.dump_tree(i), hb.dump_tree(i), f"tree {i}")
    wa, wb = ha.walkers(), hb.walkers()
    for k in ("parents", "permitted", "path", "pos", "path_len"):
        assert np.array_equal(wa[k], wb[k]), k
    aa, ab = ha.argmin(), hb.argmin()
    assert aa["eval"] == ab["eval"] and np.array_equal(aa["parents"], ab["parents"])
    assert ha.counters() == hb.counters()


@pytest.mark.parametrize("n,b,steps,c_puct,seed", [(19, 256, 200, 1.0, 0), (19, 64, 120, 4.0, 1), (33, 16, 80, 0.5, 2),
                                                   (64, 4, 60, 1.0, 3)])
def test_lock_step_matches_oracle(capi, orc, n, b, steps, c_puct, seed):
    first = 1000 * seed
    a_dim = orc.action_dim(n)
    parents, masks = orc.generate_roots(seed, first, b, n)
    o = PuctOptimizer(n, b, c_puct=c_puct, lambda_method=orc.LAMBDA_MULTISECTION, n_threads=4)
    o.set_roots(parents, masks)
    o.init_trees(orc.hash_priors(seed, first, b, a_dim, 0))
    with _mk(capi, n, b, prior_mode=capi.PRIOR_HASH, prior_seed=seed, first_root=first, max_steps=steps,
             selection=capi.SELECT_PUCT, puct_c=c_puct) as h:
        h.set_roots(parents, masks)
        h.init_trees()
        imp_o, imp_g = [], []
        for s in range(steps):
            imp_o += o.steps_hash(seed, first, 1 + s, 1)
            n_imp, imps = h.step(1, cap=16)
            imp_g += [st for (st, _, _, _) in imps]
        for i in range(b):
            _same_trees(o.dump_tree(i), h.dump_tree(i), f"tree {i}")
        wo, wg = o.walkers(), h.walkers()
        for k in ("parents", "permitted", "path", "pos", "path_len"):
            assert np.array_equal(wo[k], wg[k]), k
        assert [s - 1 for s in imp_o] == imp_g
        assert h.counters() == o.counters()
        ao, ag = o.argmin(), h.argmin()
        assert ag["eval"] == ao["eval"] and ag["mu"] == ao["mu"] and np.array_equal(ag["parents"], ao["parents"])


@pytest.mark.parametrize("n,b,steps", [(19, 512, 120), (40, 64, 60), (64, 32, 40)])
def test_one_launch_hash_mode_and_yielding_launches_equal_lock_step(capi, n, b, steps):
    parents, masks = capi.generate_roots(4, 0, b, n)
    kw = dict(prior_mode=capi.PRIOR_HASH, prior_seed=4, max_steps=steps + 2, **PUCT)
    with _mk(capi, n, b, **kw) as lock, _mk(capi, n, b, **kw) as multi, _mk(capi, n, b, max_episodes=2, **kw) as yld, \
            _mk(capi, n, b, n_groups=2, **kw) as grp:
        for h in (lock, multi, yld, grp):
            h.set_roots(parents, masks)
            h.init_trees()
        for _ in range(steps):
            lock.step(1)
        multi.step(steps, cap=1024)
        yld.step(steps, cap=1024)
        grp.step(steps, cap=1024)
        for h in (multi, yld, grp):
            _same_runs(lock, h, b)


@pytest.mark.parametrize("steal", ["0", "1"])
def test_async_kernel_equals_lock_step_and_oracle(capi, orc, monkeypatch, steal):
    monkeypatch.setenv("AZB_ASYNC_STEAL", steal)
    n, b, steps = 19, 4096, 100
    parents, masks = capi.generate_roots(0, 0, b, n)
    kw = dict(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, max_steps=steps + 2, **PUCT)
    idx = list(range(0, b, b // 64))[:64]
    o = PuctOptimizer(n, len(idx), c_puct=1.0, lambda_method=orc.LAMBDA_MULTISECTION, n_threads=4)
    o.set_roots(parents[idx], masks[idx])
    with _mk(capi, n, b, **kw) as lock, _mk(capi, n, b, async_workers=capi.ASYNC_AUTO, **kw) as asy:
        for h in (lock, asy):
            h.mlp_init(1)
            h.set_roots(parents, masks)
            h.init_trees()
        o.init_trees(np.ascontiguousarray(lock.priors()[idx]))
        asy.step(steps, cap=1024)
        for _ in range(steps):  # the oracle follows the lock step on the priors its model produced
            lock.step(1)
            o.rollout()
            o.add_actions(np.ascontiguousarray(lock.priors()[idx]))
        _same_runs(lock, asy, b)
        for j, i in enumerate(idx):
            _same_trees(o.dump_tree(j), asy.dump_tree(i), f"tree {i}")
        k = asy.counters()
        assert k["n_live"] + k["n_noop"] == b * steps and k["n_cur"] == k["n_sel"]


@pytest.mark.parametrize("n,seed", [(7, 0), (9, 1), (12, 2)])
def test_quantised_prior_ties_match_oracle(capi, orc, n, seed):
    """Priors from {0.25, 0.5, 0.75} injected every step: equal scores, first maximum, at most selections."""
    b, steps = 32, 80
    a_dim = orc.action_dim(n)
    rng = np.random.default_rng(300 + seed)
    parents, masks = orc.generate_roots(seed, 0, b, n, k_min=min(5, a_dim // 2), k_max=a_dim // 2)
    vals = np.array([0.25, 0.5, 0.75], dtype=np.float32)
    o = PuctOptimizer(n, b, c_puct=1.0, lambda_method=orc.LAMBDA_MULTISECTION)
    o.set_roots(parents, masks)
    with _mk(capi, n, b, prior_mode=capi.PRIOR_INJECTED, max_steps=steps + 2, **PUCT) as h:
        h.set_roots(parents, masks)
        pri = rng.choice(vals, size=(b, a_dim)).astype(np.float32)
        h.set_priors(pri)
        h.init_trees()
        o.init_trees(pri)
        vecs = np.zeros((b, 2 * a_dim), dtype=np.float32)
        for s in range(steps):
            pri = rng.choice(vals, size=(b, a_dim)).astype(np.float32)
            h.rollout_host(vecs)
            h.add_actions_host(pri)
            o.rollout()
            o.add_actions(pri)
        for i in range(b):
            _same_trees(o.dump_tree(i), h.dump_tree(i), f"tree {i}")
        assert h.counters() == o.counters()


@pytest.mark.parametrize("selection,puct_c", [(2, 1.0), (7, 1.0), (1, 0.0), (1, -2.0), (1, float("inf")), (1, float("nan"))])
def test_create_rejects_bad_selection(capi, selection, puct_c):
    with pytest.raises(capi.AzbError) as e:
        _mk(capi, 19, 8, prior_mode=capi.PRIOR_HASH, selection=selection, puct_c=puct_c)
    assert e.value.code == capi.ERR_INVALID


def test_config_round_trip_and_default(capi):
    cfg = capi.default_config(19, 8)
    assert cfg.selection == capi.SELECT_REFERENCE and cfg.puct_c == 1.0
    with _mk(capi, 19, 8, prior_mode=capi.PRIOR_HASH, selection=capi.SELECT_PUCT, puct_c=2.5) as h:
        out = capi.Config()
        assert capi.lib().azb_get_config(h._h, capi.C.byref(out)) == 0
        assert out.selection == capi.SELECT_PUCT and out.puct_c == 2.5
    # the reference mode ignores puct_c: same trees as the default config
    parents, masks = capi.generate_roots(6, 0, 64, 19)
    with _mk(capi, 19, 64, prior_mode=capi.PRIOR_HASH, prior_seed=6) as a, \
            _mk(capi, 19, 64, prior_mode=capi.PRIOR_HASH, prior_seed=6, puct_c=0.3) as b:
        for h in (a, b):
            h.set_roots(parents, masks)
            h.init_trees()
            h.step(50)
        _same_runs(a, b, 64)
