"""The asynchronous search step (azb_config.async_workers > 0: ONE persistent cooperative kernel whose CTAs are tree
walkers or tensor-core model workers, azb_async.cuh) must give exactly what the lock step gives: trees are independent
and a row's forward pass does not depend on the tile it rides in.  Bit-exact trees, walkers, priors, improvement log,
argmin, counters.  The timed configurations themselves are covered in test_gpu_timed_configs.py."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _mk(capi, n, b, **kw):
    return capi.Handle(capi.default_config(n, b, **kw))


def _same(ha, hb, b):
    for i in range(b):
        da, db = ha.dump_tree(i), hb.dump_tree(i)
        for k in ("nodes", "keys", "preds", "arcs"):
            assert da[k].shape == db[k].shape and np.array_equal(da[k], db[k]), f"tree {i} {k}"
    wa, wb = ha.walkers(), hb.walkers()
    for k in ("parents", "permitted", "path", "pos", "path_len"):
        assert np.array_equal(wa[k], wb[k]), k
    live = wa["path_len"] > 0  # an exhausted root's prior row is never read again (and differs: the lock step keeps
    assert np.array_equal(ha.priors()[live], hb.priors()[live])  # its last live row, the async kernel an older one)
    aa, ab = ha.argmin(), hb.argmin()
    assert aa["eval"] == ab["eval"] and np.array_equal(aa["parents"], ab["parents"])
    assert ha.counters() == hb.counters()


@pytest.mark.parametrize("n,b,workers,mlp", [(19, 300, 4, "tc"), (19, 1024, 8, "tc"), (12, 77, 4, "tc"), (33, 160, 4, "tc"),
                                             (64, 96, 4, "tc"), (19, 200, 4, "tc3")])
def test_async_equals_lock_step(capi, n, b, workers, mlp):
    steps = 36
    parents, masks = capi.generate_roots(5, 0, b, n)
    kw = dict(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC3 if mlp == "tc3" else capi.MLP_TC, max_steps=2 * steps + 2)
    with _mk(capi, n, b, **kw) as lock, _mk(capi, n, b, async_workers=workers, **kw) as asy:
        for h in (lock, asy):
            h.mlp_init(3)
            h.set_roots(parents, masks)
            h.init_trees()
        n1, log1 = lock.step(steps, cap=256)
        n2, log2 = asy.step(steps, cap=256)
        assert n1 == n2 and [tuple(x) for x in log1] == [tuple(x) for x in log2]
        _same(lock, asy, b)
        # mixed calls: a single step (the CUDA-graph path) between two asynchronous runs
        for h in (lock, asy):
            h.step(1)
            h.step(steps)
        _same(lock, asy, b)


@pytest.mark.parametrize("env", [{"AZB_ASYNC_GROUP": "2"}, {"AZB_ASYNC_GROUP": "4"}, {"AZB_ASYNC_FLUSH_NS": "0"}])
@pytest.mark.parametrize("n,b,workers", [(19, 1024, 8), (12, 77, 4)])
def test_async_variants_equal_lock_step(capi, monkeypatch, env, n, b, workers):
    """Worker groups (G SMs per tile, N-split) and an eager flush of partial tiles: same results."""
    steps = 30
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    parents, masks = capi.generate_roots(6, 0, b, n)
    kw = dict(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, max_steps=2 * steps + 2)
    with _mk(capi, n, b, **kw) as lock, _mk(capi, n, b, async_workers=workers, **kw) as asy:
        for h in (lock, asy):
            h.mlp_init(4)
            h.set_roots(parents, masks)
            h.init_trees()
            h.step(steps)
            h.step(steps)
        _same(lock, asy, b)


@pytest.mark.parametrize("steal", ["0", "1"])
@pytest.mark.parametrize("n,b,workers", [(19, 300, 4), (19, 5000, 20), (12, 77, 4), (33, 160, 4), (64, 96, 4)])
def test_tree_scheduling_forms_equal_lock_step(capi, monkeypatch, steal, n, b, workers):
    """Inside a tree CTA either every warp advances only its own trees (AZB_ASYNC_STEAL=0: bookkeeping in registers, the
    default while there is a warp for every tree) or any free warp takes over any runnable tree of the CTA through the
    scheduling table in shared memory (1: the default beyond that).  Who advances a tree does not change the tree."""
    steps = 30
    monkeypatch.setenv("AZB_ASYNC_STEAL", steal)
    parents, masks = capi.generate_roots(12, 0, b, n)
    kw = dict(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, max_steps=2 * steps + 2)
    with _mk(capi, n, b, **kw) as lock, _mk(capi, n, b, async_workers=workers, **kw) as asy:
        for h in (lock, asy):
            h.mlp_init(7)
            h.set_roots(parents, masks)
            h.init_trees()
        n1, log1 = lock.step(steps, cap=256)
        n2, log2 = asy.step(steps, cap=256)
        assert n1 == n2 and [tuple(x) for x in log1] == [tuple(x) for x in log2]
        _same(lock, asy, b)
        for h in (lock, asy):
            h.step(1)
            h.step(steps)
        _same(lock, asy, b)


def test_async_then_training_and_reset(capi):
    """An epoch on the asynchronous kernel followed by the epoch boundary (update_model, reset_trees) and a second
    epoch: identical to the lock step all the way."""
    n, b, steps = 19, 200, 30
    parents, masks = capi.generate_roots(8, 0, b, n)
    kw = dict(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, max_steps=steps)
    with _mk(capi, n, b, **kw) as lock, _mk(capi, n, b, async_workers=4, **kw) as asy:
        out = []
        for h in (lock, asy):
            h.mlp_init(1)
            h.set_roots(parents, masks)
            h.init_trees()
            h.step(steps)
            loss = h.update_model(3)
            h.reset_trees(17)
            h.step(steps)
            out.append(loss)
        assert out[0] == out[1]
        assert np.array_equal(lock.mlp_get_params(), asy.mlp_get_params())
        _same(lock, asy, b)


@pytest.mark.parametrize("b", [1, 129])
def test_async_ragged_batch_sizes(capi, b):
    """One root, and one more than a tile: partial tiles are flushed with dummy rows, nothing hangs, same trees."""
    n, steps = 19, 25
    parents, masks = capi.generate_roots(2, 0, b, n)
    kw = dict(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, max_steps=steps)
    with _mk(capi, n, b, **kw) as lock, _mk(capi, n, b, async_workers=2, **kw) as asy:
        for h in (lock, asy):
            h.mlp_init(9)
            h.set_roots(parents, masks)
            h.init_trees()
            h.step(steps)
        _same(lock, asy, b)


def test_async_reports_capacity_overflow_instead_of_hanging(capi):
    """A tree that overflows its arena inside the persistent kernel raises the abort flag: every spin loop drains and
    the call returns AZB_ERR_CAPACITY (the lock step reports the same error)."""
    n, b = 19, 200
    parents, masks = capi.generate_roots(3, 0, b, n)
    for workers in (0, 4):
        with _mk(capi, n, b, prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, max_steps=200, cap_nodes=24,
                 async_workers=workers) as h:
            h.mlp_init(1)
            h.set_roots(parents, masks)
            h.init_trees()
            with pytest.raises(capi.AzbError) as e:
                h.step(150)
            assert e.value.code == capi.ERR_CAPACITY


def test_async_needs_the_tensor_core_model(capi):
    n, b = 19, 64
    parents, masks = capi.generate_roots(3, 0, b, n)
    with _mk(capi, n, b, prior_mode=capi.PRIOR_HASH, async_workers=4, max_steps=20) as h:
        h.set_roots(parents, masks)
        h.init_trees()
        with pytest.raises(capi.AzbError) as e:
            h.step(10)
        assert e.value.code == capi.ERR_INVALID


@pytest.mark.parametrize("workers", [0, 4])
def test_step_poll_reports_each_step_while_later_steps_run(capi, workers):
    """azb_step_enqueue + one azb_step_poll per step: the per-step ArgminImprovement of par_roll_out_episodes, read while
    the trees run ahead.  The polled improvements are exactly the log azb_step(h, 0) then returns, and exactly what one
    blocking azb_step(K) gives."""
    n, b, steps = 19, 300, 40
    parents, masks = capi.generate_roots(11, 0, b, n)
    kw = dict(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, max_steps=2 * steps, async_workers=workers)
    with _mk(capi, n, b, **kw) as ref, _mk(capi, n, b, **kw) as h:
        for x in (ref, h):
            x.mlp_init(5)
            x.set_roots(parents, masks)
            x.init_trees()
        with pytest.raises(capi.AzbError) as e:
            h.step_poll()
        assert e.value.code == capi.ERR_STATE
        for rnd in range(2):  # two batches: the running best carries over
            n_ref, log_ref = ref.step(steps, cap=256)
            h.step_enqueue(steps)
            polled = []
            for s in range(steps):
                improved, rec = h.step_poll()
                assert rec[0] == rnd * steps + s
                if improved:
                    polled.append(tuple(rec))
            with pytest.raises(capi.AzbError):
                h.step_poll()  # nothing left
            n_end, log_end = h.step(0, cap=256)
            assert n_end == n_ref == len(polled)
            assert [tuple(x) for x in log_end] == polled == [tuple(x) for x in log_ref]
        _same(ref, h, b)


def test_async_watchdog_ends_a_stuck_launch_within_seconds(capi, monkeypatch):
    """Every spin loop of the persistent kernel watches %globaltimer.  With the floor set to 1 ms and no per-step
    allowance left to speak of, a launch that cannot finish in time must drain and return AZB_ERR_CUDA ("watchdog")
    instead of hanging, and the handle must be usable afterwards."""
    import time

    n, b = 19, 2048
    monkeypatch.setenv("AZB_ASYNC_TIMEOUT_MS", "0")
    parents, masks = capi.generate_roots(3, 0, b, n)
    with _mk(capi, n, b, prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, max_steps=4000, async_workers=8) as h:
        h.mlp_init(1)
        h.set_roots(parents, masks)
        h.init_trees()
        t0 = time.time()
        try:
            h.step(2)  # allowance: 2 x 20 ms — enough for two steps; must succeed or report, never hang
        except capi.AzbError as e:
            assert e.code == capi.ERR_CUDA and "watchdog" in str(e)
        assert time.time() - t0 < 20.0


@pytest.mark.parametrize("env", [{}, {"AZB_ASYNC_GROUP": "4"}, {"AZB_ASYNC_GROUP": "16"}, {"AZB_ASYNC_FLUSH_NS": "0"}])
@pytest.mark.parametrize("n,b,mlp", [(19, 1024, "tc"), (19, 300, "tc"), (12, 77, "tc"), (33, 160, "tc"), (19, 200, "tc3")])
def test_shared_sm_form_equals_lock_step(capi, monkeypatch, env, n, b, mlp):
    """AZB_ASYNC_SHARED: every SM walks trees with 28 warps and its last warpgroup is one of G members of a model group
    (column slices of every layer, layer barriers through the group's counter line).  Same results as the lock step."""
    steps = 30
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    parents, masks = capi.generate_roots(9, 0, b, n)
    kw = dict(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC3 if mlp == "tc3" else capi.MLP_TC, max_steps=2 * steps + 2)
    with _mk(capi, n, b, **kw) as lock, _mk(capi, n, b, async_workers=capi.ASYNC_SHARED, **kw) as asy:
        for h in (lock, asy):
            h.mlp_init(4)
            h.set_roots(parents, masks)
            h.init_trees()
        n1, log1 = lock.step(steps, cap=256)
        n2, log2 = asy.step(steps, cap=256)
        assert n1 == n2 and [tuple(x) for x in log1] == [tuple(x) for x in log2]
        _same(lock, asy, b)
        for h in (lock, asy):
            h.step(1)
            h.step(steps)
        _same(lock, asy, b)
