"""azb_eval_graph_costs64 on the GPU: the cost row and action kinds of ConnectedBitsetGraph<N, B64> (N <= 64) through
the C ABI.  Action kinds bit-exact against the oracle, lambda_1 within 1e-12 relative of the oracle's.  The matching
number is checked against networkx (max_weight_matching with maxcardinality) on random graphs: the oracle's
restatement of the reference's branch and bound takes seconds per graph on sparse graphs of 48 and more vertices."""
import ctypes as C

import networkx as nx
import numpy as np
import pytest

import graph64_oracle as g64
from graphs64_util import lambda1_lapack, named_graphs64, random_connected_graph64
from graphs_util import edges_of, named_graphs, random_connected_graph

pytestmark = pytest.mark.gpu


def _mk(capi):
    return capi.Handle(capi.default_config(6, 2, prior_mode=capi.PRIOR_HASH))


def _mu_nx(g):
    return len(nx.max_weight_matching(nx.Graph(edges_of(g)), maxcardinality=True))


def _relabel(g, perm):
    """Vertex v -> perm[v] on u64 neighbourhood masks."""
    n = len(g)
    bits = (g[:, None] >> np.arange(n, dtype=np.uint64)[None, :]) & np.uint64(1)
    pb = np.zeros_like(bits)
    pb[np.ix_(perm, perm)] = bits
    return (pb << np.arange(n, dtype=np.uint64)[None, :]).sum(axis=1, dtype=np.uint64)


def test_named_graphs_closed_forms(capi, orc):
    with _mk(capi) as h:
        for name, n, edges, lam, mu in named_graphs() + named_graphs64():
            if lam is None:
                lam = lambda1_lapack(n, edges)
            g = g64.graph64_from_edges(n, edges)
            if lam + 1e-4 <= 1.4:  # connected_bitset_graph/mod.rs:333 asserts
                with pytest.raises(capi.AzbError) as e:
                    h.eval_graph_costs64(g[None, :])
                assert e.value.code == capi.ERR_LAMBDA, name
                continue
            l1, m, kinds, _ = h.eval_graph_costs64(g[None, :])
            assert m[0] == mu, name
            assert abs(l1[0] - (lam + 1e-4)) <= 1e-12 * max(1.0, lam), name
            assert np.array_equal(kinds[0], g64.graph64_action_kinds(g)), name


# n = 2 is K2 alone, whose lambda_1 is below 1.4: test_named_graphs_closed_forms covers it (ERR_LAMBDA)
@pytest.mark.parametrize("n,p,m", [(3, 0.0, 50), (5, 0.3, 200), (19, 0.12, 300), (32, 0.06, 300), (33, 0.0, 200),
                                   (33, 0.3, 200), (47, 0.05, 200), (48, 0.0, 200), (48, 0.5, 150), (63, 0.02, 150),
                                   (64, 0.0, 150), (64, 0.06, 150), (64, 0.3, 100), (64, 0.95, 60)])
def test_random_graphs_match_oracle(capi, orc, n, p, m):
    rng = np.random.default_rng(91 * n + int(1000 * p))
    graphs = np.stack([random_connected_graph64(rng, n, p) for _ in range(m)])
    with _mk(capi) as h:
        l1, mu, kinds, _ = h.eval_graph_costs64(graphs)
    for i in range(m):
        lo = g64.graph64_lambda1(graphs[i])
        assert mu[i] == _mu_nx(graphs[i]), f"graph {i}: mu"
        assert abs(l1[i] - lo) <= 1e-12 * lo, f"graph {i}: lambda_1 {l1[i]!r} vs oracle {lo!r}"
        assert np.array_equal(kinds[i], g64.graph64_action_kinds(graphs[i])), f"graph {i}: action kinds"


@pytest.mark.parametrize("n,p", [(3, 0.5), (5, 0.3), (19, 0.0), (19, 0.2), (32, 0.04), (32, 0.9)])
def test_up_to_32_vertices_equals_the_b32_entry(capi, n, p):
    rng = np.random.default_rng(7 * n + int(100 * p))
    graphs = np.stack([random_connected_graph(rng, n, p) for _ in range(400)])
    with _mk(capi) as h:
        l1, mu, kinds, _ = h.eval_graph_costs(graphs)
        l64, mu64, kinds64, _ = h.eval_graph_costs64(graphs.astype(np.uint64))
    assert np.array_equal(mu, mu64) and np.array_equal(kinds, kinds64)
    assert np.all(np.abs(l1 - l64) <= 1e-12 * l1)


def test_invalid_graphs_are_rejected(capi, orc):
    with _mk(capi) as h:
        two_parts = g64.graph64_from_edges(40, [(i, i + 1) for i in range(19)] + [(i, i + 1) for i in range(20, 39)])
        one_way = g64.graph64_from_edges(36, [(i, i + 1) for i in range(35)])
        one_way[35] ^= np.uint64(1 << 34)
        loop = g64.graph64_from_edges(3, [(0, 1), (1, 2)])
        loop[1] |= np.uint64(1 << 1)
        high40 = g64.graph64_from_edges(40, [(i, i + 1) for i in range(39)])
        high40[7] |= np.uint64(1 << 63)  # a neighbour >= n
        high20 = g64.graph64_from_edges(20, [(i, i + 1) for i in range(19)])
        high20[3] |= np.uint64(1 << 40)  # bits 32..63 when n <= 32
        for bad in (two_parts, one_way, loop, high40, high20, np.zeros(65, dtype=np.uint64), np.zeros(1, dtype=np.uint64)):
            with pytest.raises(capi.AzbError) as e:
                h.eval_graph_costs64(bad[None, :])
            assert e.value.code == capi.ERR_INVALID


def test_one_bad_graph_in_a_batch_is_named(capi, orc):
    rng = np.random.default_rng(3)
    graphs = np.stack([random_connected_graph64(rng, 50, 0.1) for _ in range(64)])
    graphs[37, 4] ^= np.uint64(1 << 45)  # one direction of an edge only
    with _mk(capi) as h:
        with pytest.raises(capi.AzbError) as e:
            h.eval_graph_costs64(graphs)
        assert e.value.code == capi.ERR_INVALID and "graph 37" in str(e.value)
        graphs[37, 4] ^= np.uint64(1 << 45)
        l1, mu, kinds, _ = h.eval_graph_costs64(graphs)  # the handle stays usable
        assert mu[37] == _mu_nx(graphs[37])
        assert np.array_equal(kinds[37], g64.graph64_action_kinds(graphs[37]))


def test_null_outputs_are_accepted(capi):
    rng = np.random.default_rng(4)
    graphs = np.ascontiguousarray(np.stack([random_connected_graph64(rng, 64, 0.1) for _ in range(16)]))
    with _mk(capi) as h:
        rc = h._L.azb_eval_graph_costs64(h._h, graphs.ctypes.data_as(C.POINTER(C.c_uint64)), 16, 64, None, None, None, None)
        assert rc == 0
        l1, mu, kinds, ms = h.eval_graph_costs64(graphs)
        assert ms > 0.0 and np.all(l1 > 1.4)


def test_full_size_properties(capi, orc):
    """65 536 graphs on 64 vertices: relabelling invariance (the cost is a graph invariant, the kinds permute with the
    vertices, so their counts do not change), counts of the kind masks, and the oracle (networkx for mu) on a sample."""
    n, m = 64, 65536
    rng = np.random.default_rng(5)
    base = np.stack([random_connected_graph64(rng, n, 0.06) for _ in range(512)])
    graphs = np.empty((m, n), dtype=np.uint64)
    for i in range(m):
        graphs[i] = base[i % 512] if i < 512 else _relabel(base[i % 512], rng.permutation(n))
    with _mk(capi) as h:
        l1, mu, kinds, ms = h.eval_graph_costs64(graphs)
    e2 = n * (n - 1) // 2
    n_edges = np.array([sum(bin(int(x)).count("1") for x in g) // 2 for g in base])
    b = np.arange(m) % 512
    assert np.array_equal(mu, mu[b])
    assert np.all(np.abs(l1 - l1[b]) <= 1e-12 * l1[b])
    bits = np.unpackbits(kinds.view(np.uint8), axis=1, bitorder="little")
    adds, dels = bits[:, :e2].sum(axis=1), bits[:, e2:2 * e2].sum(axis=1)
    assert bits.sum(axis=1).tolist() == (adds + dels).tolist()
    assert np.array_equal(adds, e2 - n_edges[b])
    assert np.array_equal(dels, dels[b]) and np.all(dels <= n_edges[b])
    for i in range(0, 512, 8):
        assert mu[i] == _mu_nx(graphs[i])
        lo = g64.graph64_lambda1(graphs[i])
        assert abs(l1[i] - lo) <= 1e-12 * lo
        assert np.array_equal(kinds[i], g64.graph64_action_kinds(graphs[i]))
    j = 4096 + 17  # a relabelled copy: its kinds are the base's, permuted
    assert np.array_equal(kinds[j], g64.graph64_action_kinds(graphs[j]))
