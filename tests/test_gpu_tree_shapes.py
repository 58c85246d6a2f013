"""The c21 cost on the GPU at the tree shapes that fill the section method's stack (tree_shapes.py), for every N from 5
to 64, against the exact lambda_1 and mu: azb_eval_costs, the search step's root evaluation (lock step and the
asynchronous kernel), the bitset-graph entries and the canonical code.

lambda_1 is held to 4 ulp of the exact value.  The oracle's mirror of the kernel is never more than 2.3 ulp off on these
inputs (test_tree_shapes_ref.py); the 1e-12 check against LAPACK elsewhere would let an error three orders of magnitude
larger through."""
import networkx as nx
import numpy as np
import pytest
from networkx.algorithms.isomorphism import tree_isomorphism

import pyref
import tree_shapes as ts
from azdopt_b200 import observe
from test_gpu_parity import _cmp_trees, _cmp_walkers

pytestmark = pytest.mark.gpu

ULP = 4.0
# The graph entries solve a general symmetric eigenproblem, so they are held to their oracles' accuracy on these trees:
# worst 1.1e-14 relative for the B32 oracle, 2.3e-14 for the B64 oracle (tests/graph64_oracle.py, the dumbbell on 62
# vertices).  The B200 measured 6.7e-16 for both entries.
B32_REL = 2e-14
B64_REL = 5e-14


def _mk(capi, n, b=4, **kw):
    return capi.Handle(capi.default_config(n, b, **kw))


def _bits(x):
    return int(np.float32(x).view(np.uint32))


@pytest.mark.parametrize("n", range(5, 65))
def test_eval_costs_exact(capi, orc, n):
    batch = ts.shape_batch(n)
    parents = np.stack([p for _, p in batch])
    if n in (22, 23, 46, 47, 64):  # the inputs reach the deepest stack level the kernel allows
        assert max(ts.slots(p) for p in parents) == ts.stack_depth(n)
    if n == 64:
        assert max(ts.program_length(p) for p in parents) == 94
    with _mk(capi, n, prior_mode=capi.PRIOR_HASH) as h:
        lam, mu, c, _ = h.eval_costs(parents)
    near, by_name = 0, {}
    for i, (name, p) in enumerate(batch):
        lo, mo, co, rc = orc.cost(p, method=orc.LAMBDA_MULTISECTION)
        assert rc == 0 and lam[i] == lo, f"{name} row {i}: lambda_1 not bit-identical to the oracle's mirror"
        u = ts.ulps(lam[i], p)
        assert u <= ULP, f"{name} row {i}: lambda_1 {lam[i]!r} is {u:.2f} ulp from the exact {ts.exact_lambda1(p)[0]!r}"
        mu_x = ts.exact_mu(p)
        assert mu[i] == mu_x, f"{name} row {i}: mu {mu[i]} != {mu_x}"
        assert _bits(c[i]) == _bits(pyref.evaluate(n, mu[i], lam[i])) == _bits(co)
        if ts.near_f32_boundary(p, ULP):
            near += 1
        else:
            assert _bits(c[i]) == _bits(pyref.evaluate(n, mu_x, ts.exact_lambda1(p)[0])), f"{name} row {i}: c"
        by_name.setdefault(name, []).append(lam[i])
    assert near == 0
    for name, vals in by_name.items():  # relabelled copies of one tree
        r = ts.exact_lambda1(next(p for q, p in batch if q == name))[0]
        assert max(vals) - min(vals) <= ULP * np.spacing(r), f"{name}: relabellings differ by more than {ULP} ulp"


def _search_roots(n, copies):
    rng = np.random.default_rng(7 * n)
    rows = []
    for f in (ts.stack_extremal, ts.longest_program):
        p = f(n)
        rows += [p] + [ts.relabel(p, rng) for _ in range(copies)]
    return np.stack(rows)


@pytest.mark.parametrize("n", [22, 23, 46, 47, 64])
def test_search_step_on_stack_extremal_roots(capi, orc, n):
    """Every root is evaluated by the init path of the search kernel; the steps then evaluate their neighbours.  Trees,
    walkers, counters and argmin are bit-exact with the oracle, and each root node's c is the exact lambda_1's."""
    parents = _search_roots(n, 3)
    b, steps, seed, first = len(parents), 60, 40 + n, 100 * n
    assert max(ts.slots(p) for p in parents) == ts.stack_depth(n)
    a_dim = orc.action_dim(n)
    masks = orc.generate_roots(seed, first, b, n, k_min=5, k_max=a_dim // 2)[1]
    o = orc.Optimizer(n, b, lambda_method=orc.LAMBDA_MULTISECTION, n_threads=4)
    o.set_roots(parents, masks)
    o.init_trees(orc.hash_priors(seed, first, b, a_dim, 0))
    with _mk(capi, n, b, prior_mode=capi.PRIOR_HASH, prior_seed=seed, first_root=first, max_steps=steps) as h:
        h.set_roots(parents, masks)
        h.init_trees()
        for i in range(b):
            want = pyref.evaluate(n, ts.exact_mu(parents[i]), ts.exact_lambda1(parents[i])[0])
            assert int(h.dump_tree(i)["nodes"][0, 0]) == _bits(want), f"root {i}: c"
        _cmp_trees(o, h, b)
        done, imp_o, imp_g = 0, [], []
        for chunk in (1, 2, steps // 3, steps):
            k = min(chunk, steps - done)
            if k <= 0:
                break
            imp_o += o.steps_hash(seed, first, 1 + done, k)
            imp_g += [s for (s, _, _, _) in h.step(k, cap=1024)[1]]
            done += k
            _cmp_trees(o, h, b)
            _cmp_walkers(o, h)
        assert [s - 1 for s in imp_o] == imp_g
        assert h.counters() == o.counters()
        ao, ag = o.argmin(), h.argmin()
        assert ag["eval"] == ao["eval"] and ag["mu"] == ao["mu"] and ag["lambda1"] == ao["lambda1"]
        assert np.array_equal(ag["parents"], ao["parents"])


@pytest.mark.parametrize("n", [47, 64])
def test_async_kernel_on_stack_extremal_roots(capi, n):
    """The asynchronous kernel (its DEPTH-5 form from 47 vertices) equals the lock step on these roots."""
    from test_gpu_async import _same

    parents = _search_roots(n, 23)
    b, steps = len(parents), 30
    masks = capi.generate_roots(5, 0, b, n)[1]
    kw = dict(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, max_steps=steps + 2)
    with _mk(capi, n, b, **kw) as lock, _mk(capi, n, b, async_workers=4, **kw) as asy:
        for h in (lock, asy):
            h.mlp_init(3)
            h.set_roots(parents, masks)
            h.init_trees()
        n1, log1 = lock.step(steps, cap=256)
        n2, log2 = asy.step(steps, cap=256)
        assert n1 == n2 and [tuple(x) for x in log1] == [tuple(x) for x in log2]
        _same(lock, asy, b)
        for i in range(b):
            want = pyref.evaluate(n, ts.exact_mu(parents[i]), ts.exact_lambda1(parents[i])[0])
            assert int(asy.dump_tree(i)["nodes"][0, 0]) == _bits(want), f"root {i}: c"


def test_graph_entries_on_tree_shapes(capi):
    """The same trees as bitset graphs: mu exact, lambda_1 of A + 1e-4 I against the exact lambda_1 + 1e-4."""
    with _mk(capi, 6, 2, prior_mode=capi.PRIOR_HASH) as h:
        for n in range(5, 65):
            batch = ts.shape_batch(n)
            g = np.zeros((len(batch), n), dtype=np.uint64)
            for i, (_, p) in enumerate(batch):
                for v, u in ts.edges_of(p):
                    g[i, v] |= np.uint64(1 << u)
                    g[i, u] |= np.uint64(1 << v)
            entries = [("B64", h.eval_graph_costs64(g), B64_REL)]
            if n <= 32:
                entries.append(("B32", h.eval_graph_costs(g.astype(np.uint32)), B32_REL))
            for what, (lam, mu, _, _), rel in entries:
                for i, (name, p) in enumerate(batch):
                    want = ts.exact_lambda1(p)[0] + 1e-4
                    assert mu[i] == ts.exact_mu(p), f"{what} n={n} {name} row {i}: mu"
                    assert abs(lam[i] - want) <= rel * want, f"{what} n={n} {name} row {i}: {lam[i]!r} vs {want!r}"


def _shapes(batch):
    """Shape index of every row: rows of one family share it, isomorphic trees of different names are merged."""
    firsts, shape_of_name, out = [], {}, []
    for name, p in batch:
        if name not in shape_of_name:
            t = nx.Graph(ts.edges_of(p))
            deg = sorted(d for _, d in t.degree())
            same = [k for k, (dq, tq) in enumerate(firsts) if dq == deg and tree_isomorphism(t, tq)]
            shape_of_name[name] = same[0] if same else len(firsts)
            if not same:
                firsts.append((deg, t))
        out.append(shape_of_name[name])
    return out, len(firsts)


@pytest.mark.parametrize("n", range(5, 65))
def test_tree_codes_on_tree_shapes(capi, n):
    batch = ts.shape_batch(n)
    parents = np.stack([p for _, p in batch])
    with _mk(capi, n, prior_mode=capi.PRIOR_HASH) as h:
        codes = h.tree_codes(parents)
    got = [(int(a), int(b)) for a, b in codes]
    assert got == [observe.tree_code(p) for p in parents]
    shape, n_shapes = _shapes(batch)
    code_of = {}
    for s, c in zip(shape, got):
        assert code_of.setdefault(s, c) == c, "one shape, two codes"
    assert len(set(code_of.values())) == n_shapes
    if n == 64:  # the path's code fills all 128 bits: 1, 32 ones, 32 zeros, 31 ones, 31 zeros, 0
        s = "1" + "1" * 32 + "0" * 32 + "1" * 31 + "0" * 31 + "0"
        assert got[[name for name, _ in batch].index("path")] == (int(s[:64], 2), int(s[64:], 2))
