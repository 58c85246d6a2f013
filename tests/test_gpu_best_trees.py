"""azb_tree_codes and azb_best_trees (include/azb.h) on the GPU: the code kernel against observe.tree_code, the k best
isomorphism classes against a host expectation built from tree dumps, and the call's invariances (prefixes, repeat
calls, the asynchronous kernel, sharding, widening rounds, enqueued steps, read-only)."""
import ctypes as C

import networkx as nx
import numpy as np
import pytest

from azdopt_b200 import observe
from best_trees_util import expected_best, parents_of, random_parents

pytestmark = pytest.mark.gpu


def _hash_handle(capi, n, b, steps, seed=0, first=0, roots=None, **kw):
    h = capi.Handle(capi.default_config(n, b, prior_mode=capi.PRIOR_HASH, prior_seed=seed, first_root=first,
                                        max_steps=max(steps, 1), **kw))
    p, m = roots if roots is not None else capi.generate_roots(seed, first, b, n)
    h.set_roots(p, m)
    h.init_trees()
    if steps:
        h.step(steps)
    return h


def _codes(rows):
    return [observe.tree_code(p) for p in rows]


def _fast_relabel(rng, p):
    """An isomorphic copy of the tree in parents[v] < v form: BFS from a random vertex with shuffled neighbours."""
    n = len(p)
    adj = [[] for _ in range(n)]
    for v in range(1, n):
        adj[v].append(int(p[v]))
        adj[int(p[v])].append(v)
    root = int(rng.integers(0, n))
    idx = {root: 0}
    order = [root]
    out = np.zeros(n, dtype=np.uint8)
    for v in order:
        nb = adj[v][:]
        rng.shuffle(nb)
        for u in nb:
            if u not in idx:
                idx[u] = len(order)
                order.append(u)
                out[idx[u]] = idx[v]
    return out


@pytest.mark.parametrize("n", range(5, 13))
def test_tree_codes_of_every_small_tree(capi, n):
    rows = np.stack([parents_of(T) for T in nx.nonisomorphic_trees(n)])
    with capi.Handle(capi.default_config(n, 1)) as h:
        got = h.tree_codes(rows)
    assert [tuple(int(x) for x in r) for r in got] == _codes(rows)


@pytest.mark.parametrize("n", [19, 33, 47, 64])
def test_tree_codes_of_random_trees(capi, n):
    rng = np.random.default_rng(n)
    rows = np.stack([random_parents(rng, n) for _ in range(300)] + [np.zeros(n, np.uint8), np.arange(-1, n - 1).clip(0).astype(np.uint8)])
    with capi.Handle(capi.default_config(n, 1)) as h:
        got = h.tree_codes(rows)
    assert [tuple(int(x) for x in r) for r in got] == _codes(rows)


def test_tree_codes_65536_relabelled_trees(capi):
    n, m = 64, 65536
    rng = np.random.default_rng(7)
    rows = np.stack([random_parents(rng, n) for _ in range(m)])
    copies = np.stack([_fast_relabel(rng, p) for p in rows])
    with capi.Handle(capi.default_config(n, 1)) as h:
        a, b = h.tree_codes(rows), h.tree_codes(copies)
    assert np.array_equal(a, b)
    sub = rng.choice(m, 256, replace=False)
    assert [tuple(int(x) for x in a[i]) for i in sub] == _codes(rows[sub])
    assert len({tuple(r) for r in a.tolist()}) > m // 2  # random trees at 64 vertices are almost never isomorphic


def test_tree_codes_rejects_and_accepts_null_outputs(capi):
    n = 19
    rng = np.random.default_rng(5)
    rows = np.stack([random_parents(rng, n) for _ in range(8)])
    bad = rows.copy()
    bad[3, 7] = 7
    bad[5, 2] = 9
    with capi.Handle(capi.default_config(n, 1)) as h:
        with pytest.raises(capi.AzbError) as e:
            h.tree_codes(bad)
        assert e.value.code == capi.ERR_INVALID and "tree 3" in str(e.value)
        assert [tuple(int(x) for x in r) for r in h.tree_codes(rows)] == _codes(rows)
        rc = capi.lib().azb_tree_codes(h._h, rows.ctypes.data_as(C.POINTER(C.c_uint8)), 8, None, None)
        assert rc == capi.OK


def _check_against_expectation(capi, h, k):
    got = h.best_trees(k)
    want = expected_best(h, k)
    assert len(got["eval"]) == len(want) == min(k, len(want))
    for i, (cbits, code, t, node, p, m) in enumerate(want):
        assert int(got["eval"][i:i + 1].view(np.uint32)[0]) == cbits, i
        assert (int(got["code"][i, 0]), int(got["code"][i, 1])) == code, i
        assert (int(got["tree"][i]), int(got["node"][i])) == (t, node), i
        assert np.array_equal(got["parents"][i], p) and np.array_equal(got["permitted"][i], m), i
    for i in range(min(len(want), 5)):
        sp, sm = h.node_state(int(got["tree"][i]), int(got["node"][i]))
        assert np.array_equal(sp, got["parents"][i]) and np.array_equal(sm, got["permitted"][i])
    if len(want):
        lam, mu, c, _ = h.eval_costs(got["parents"])
        assert np.array_equal(lam, got["lambda1"]) and np.array_equal(mu, got["mu"])
    return got, want


@pytest.mark.parametrize("n,b,steps", [(19, 64, 200), (33, 16, 60), (64, 4, 30)])
def test_best_trees_match_the_host_expectation(capi, n, b, steps):
    with _hash_handle(capi, n, b, steps, seed=n) as h:
        n_cls = len(expected_best(h, 1 << 30))
        for k in (1, 10, n_cls + 5):
            got, want = _check_against_expectation(capi, h, k)
        assert len(got["eval"]) == n_cls


def test_timed_shape_consistency(capi):
    n, b, steps = 19, 4096, 800
    with _hash_handle(capi, n, b, steps, seed=3) as h:
        a100, a1000, again = h.best_trees(100), h.best_trees(1000), h.best_trees(1000)
        for key in a1000:
            assert np.array_equal(a1000[key][:100], a100[key]), key
            assert np.array_equal(a1000[key], again[key]), key
        assert a1000["eval"][0] == h.argmin()["eval"]  # a first epoch: the argmin is the best class's value
        assert np.all(np.diff(a1000["eval"]) >= 0)


def test_async_kernel_and_lock_step_agree(capi):
    n, b, steps = 19, 1024, 100
    res = []
    for workers in (capi.ASYNC_AUTO, 0):
        cfg = capi.default_config(n, b, prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, max_steps=steps, async_workers=workers)
        with capi.Handle(cfg) as h:
            h.mlp_init(5)
            h.set_roots(*capi.generate_roots(4, 0, b, n))
            h.init_trees()
            h.step(steps)
            res.append(h.best_trees(200))
    for key in res[0]:
        assert np.array_equal(res[0][key], res[1][key]), key


def _records(h, res, first):
    from azdopt_b200.nabla import BestTree

    return [BestTree(res["eval"][i], float(res["lambda1"][i]), int(res["mu"][i]), res["parents"][i], res["permitted"][i],
                     (int(res["code"][i, 0]), int(res["code"][i, 1])), first + int(res["tree"][i]), int(res["node"][i]))
            for i in range(len(res["eval"]))]


def test_two_shards_merge_to_one_handle(capi):
    from azdopt_b200.nabla import BestTrees

    n, b, steps, k = 19, 256, 150, 300
    with _hash_handle(capi, n, b, steps, seed=9) as one:
        whole = _records(one, one.best_trees(k), 0)
    acc = BestTrees(k)
    for first in (0, b // 2):
        with _hash_handle(capi, n, b // 2, steps, seed=9, first=first) as h:
            acc.add(_records(h, h.best_trees(k), first))
    key = lambda ts: [(float(t.eval), t.code, t.root, t.node, t.parents.tobytes(), t.lambda_1, t.mu) for t in ts]
    assert key(acc.result()) == key(whole)


def test_widening_rounds_give_the_default_result(capi, monkeypatch):
    n, b, steps, k = 19, 128, 120, 25
    p, m = capi.generate_roots(2, 0, 1, n)
    roots = (np.repeat(p, b, axis=0), np.repeat(m, b, axis=0))  # every root the same tree: the cheapest nodes repeat
    with _hash_handle(capi, n, b, steps, seed=2, roots=roots) as h:
        want = h.best_trees(k)
    for cap in ("1", "7"):
        monkeypatch.setenv("AZB_TEST_BEST_CAP", cap)
        with _hash_handle(capi, n, b, steps, seed=2, roots=roots) as h:
            got = h.best_trees(k)
        for key in want:
            assert np.array_equal(got[key], want[key]), (cap, key)
    assert len(want["eval"]) == k


def test_enqueued_steps_errors_and_read_only(capi):
    n, b = 19, 128
    with capi.Handle(capi.default_config(n, b, prior_mode=capi.PRIOR_HASH, max_steps=200)) as h:
        with pytest.raises(capi.AzbError) as e:
            h.best_trees(1)
        assert e.value.code == capi.ERR_STATE
        h.set_roots(*capi.generate_roots(1, 0, b, n))
        h.init_trees()
        h.step(40)
        for k in (0, 65537):
            with pytest.raises(capi.AzbError) as e:
                h.best_trees(k)
            assert e.value.code == capi.ERR_INVALID
        h.step_enqueue(60)
        during = h.best_trees(50)
        h.step(0)
        after = h.best_trees(50)
        for key in during:
            assert np.array_equal(during[key], after[key]), key
        before = ([h.dump_tree(i) for i in range(b)], h.counters(), h.argmin(), h.walkers())
        assert len(h.best_trees(65536)["eval"]) > 50
        now = ([h.dump_tree(i) for i in range(b)], h.counters(), h.argmin(), h.walkers())
        for da, db in zip(before[0], now[0]):
            for key in da:
                assert np.array_equal(da[key], db[key])
        assert before[1] == now[1]
        assert before[2]["eval"] == now[2]["eval"] and np.array_equal(before[2]["parents"], now[2]["parents"])
        for key in before[3]:
            assert np.array_equal(before[3][key], now[3][key])
