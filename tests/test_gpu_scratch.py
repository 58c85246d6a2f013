"""The device scratch of the calls outside the search step (one grow-only slab on the handle) on the GPU: azb_device_bytes
counts it, a grow replaces the old slab in the count instead of adding to it, and calls that share the slab in any
order return what each returns on a fresh handle in the same state."""
import numpy as np
import pytest

from azdopt_b200 import checkpoint
from graphs64_util import random_connected_graph64

pytestmark = pytest.mark.gpu

N, B, STEPS = 19, 256, 40


def _trees(rng, m, n=N):
    """m uniform-attachment random trees: parents[v] uniform in 0..v-1."""
    return (rng.random((m, n)) * np.arange(n)).astype(np.uint8)


def test_graph_costs_are_counted(capi):
    m, n = 2048, 40
    rng = np.random.default_rng(1)
    nbr = np.stack([random_connected_graph64(rng, n, 0.05) for _ in range(m)])
    with capi.Handle(capi.default_config(6, 2, prior_mode=capi.PRIOR_HASH)) as h:
        before = h.device_bytes()
        h.eval_graph_costs64(nbr)
        assert h.device_bytes() - before >= m * n * 8


def test_growing_batches_count_the_largest(capi):
    rng = np.random.default_rng(2)
    need = 65536 * (N + 8 + 4 + 4) + 4  # parents, lambda_1, mu, eval, the error word
    with capi.Handle(capi.default_config(N, 1)) as h:
        before = h.device_bytes()
        for m in (1024, 4096, 16384, 65536):
            h.eval_costs(_trees(rng, m))
        grown = h.device_bytes() - before
    assert need <= grown < 1.2 * need


def _stepped(capi):
    h = capi.Handle(capi.default_config(N, B, prior_mode=capi.PRIOR_HASH, prior_seed=5, max_steps=STEPS))
    h.set_roots(*capi.generate_roots(5, 0, B, N))
    h.init_trees()
    h.step(STEPS)
    h.walkers()  # runs the deferred add_actions, so every call below only reads
    return h


def _calls():
    rng = np.random.default_rng(3)
    parents, codes_in = _trees(rng, 2048), _trees(rng, 256)
    nbr = np.stack([random_connected_graph64(rng, 40, 0.05) for _ in range(2048)])
    return {
        "argmin": lambda h: h.argmin(),
        "tree_codes": lambda h: h.tree_codes(codes_in),
        "eval_costs": lambda h: h.eval_costs(parents)[:3],
        "best_trees": lambda h: h.best_trees(1000),
        "graph_costs64": lambda h: h.eval_graph_costs64(nbr)[:3],
        "checkpoint_save": lambda h: h.checkpoint_save(),
        "trees_within": lambda h: _no_ms(h.trees_within(k=100)),
        "exhaustive_best": lambda h: _no_ms(h.exhaustive_best(k=100)),
    }


def _no_ms(res):
    return {k: v for k, v in res.items() if k != "ms"}


def _same(a, b):
    if isinstance(a, dict):
        assert a.keys() == b.keys()
        for k in a:
            _same(a[k], b[k])
    elif isinstance(a, tuple):
        assert len(a) == len(b)
        for x, y in zip(a, b):
            _same(x, y)
    else:
        assert np.array_equal(a, b)


def _check(name, got, want):
    if name == "checkpoint_save":
        # a tree record keeps the bytes of its reserved arc slots as the handle's arena held them (include/azb.h), so
        # another handle agrees on the header, the model and the offset table
        end = checkpoint.read_header(got).trees[0]
        got, want = got[:end], want[:end]
    _same(got, want)


def test_interleaved_calls_share_nothing(capi):
    calls = _calls()
    # each call alone on a fresh handle: its result, and the scratch it needs
    alone, need = {}, {}
    for name, call in calls.items():
        with _stepped(capi) as h:
            before = h.device_bytes()
            alone[name] = call(h)
            need[name] = h.device_bytes() - before
    order = sorted(calls, key=need.get)
    assert len(set(need.values())) == len(need), need
    saves = []
    with _stepped(capi) as h:
        # ascending need: the slab grows before every call
        for name in order:
            before = h.device_bytes()
            got = calls[name](h)
            assert h.device_bytes() > before, name
            _check(name, got, alone[name])
            if name == "checkpoint_save":
                saves.append(got)
        # descending: the slab no longer grows, and each call finds the bytes the larger ones left behind
        top = h.device_bytes()
        for name in reversed(order):
            got = calls[name](h)
            _check(name, got, alone[name])
            if name == "checkpoint_save":
                saves.append(got)
        assert h.device_bytes() == top
    assert np.array_equal(saves[0], saves[1])  # two saves of one handle write the same bytes
