"""The B64 restatement of ConnectedBitsetGraph's cost and action kinds (tests/graph64_oracle.cpp, N <= 64) against
networkx / LAPACK, closed forms, and the oracle's B32 functions on zero-extended words.  CPU only."""
import networkx as nx
import numpy as np
import pytest

import graph64_oracle as g64
from graphs64_util import lambda1_lapack, named_graphs64, random_connected_graph64
from graphs_util import edges_of, random_connected_graph


def _bit(kinds, i):
    return int(kinds[i >> 5]) >> (i & 31) & 1


def test_named_graphs_closed_forms(orc):
    """Includes K(5,40), on which the branch and bound takes about ten seconds (its bound popcount(unvisited) / 2 is far
    above the matching number 5)."""
    for name, n, edges, lam, mu in named_graphs64():
        if lam is None:
            lam = lambda1_lapack(n, edges)
        g = g64.graph64_from_edges(n, edges)
        l1, m, rc = g64.graph64_cost(g)
        assert m == mu, name
        assert abs(l1 - (lam + 1e-4)) <= 1e-12 * max(1.0, lam), name
        assert rc == 0, name


@pytest.mark.parametrize("n", [33, 40, 48, 63, 64])
@pytest.mark.parametrize("p", [0.0, 0.03, 0.1, 0.3, 0.9])
def test_random_graphs_against_networkx_and_lapack(orc, n, p):
    """The matching number is compared only where the branch and bound finishes in milliseconds: up to 40 vertices at
    any density, and from a density of 0.3 up.  On sparse graphs of 48 and more vertices it takes seconds each."""
    rng = np.random.default_rng(1000 * n + int(100 * p))
    for _ in range(6):
        g = random_connected_graph64(rng, n, p)
        edges = edges_of(g)
        G = nx.Graph(edges)
        if n <= 40 or p >= 0.3:
            assert g64.graph64_matching_number(g) == len(nx.max_weight_matching(G, maxcardinality=True))
        l1 = g64.graph64_lambda1(g)
        assert abs(l1 - (lambda1_lapack(n, edges) + 1e-4)) <= 1e-12 * l1
        bridges = {(max(e), min(e)) for e in nx.bridges(G)}
        kinds = g64.graph64_action_kinds(g)
        e2 = n * (n - 1) // 2
        edge_set = set(edges)
        for v in range(n):
            for u in range(v):
                pos = orc.colex_position(v, u)
                is_edge = (v, u) in edge_set
                assert _bit(kinds, pos) == (0 if is_edge else 1)
                assert _bit(kinds, e2 + pos) == (1 if is_edge and (v, u) not in bridges else 0)
                if is_edge:
                    assert g64.graph64_is_cut_edge(g, v, u) == ((v, u) in bridges)


def test_zero_extended_words_equal_the_b32_oracle(orc):
    rng = np.random.default_rng(12)
    for n in range(2, 33):
        for _ in range(4):
            g = random_connected_graph(rng, n, float(rng.random()) * 0.6)
            w = g.astype(np.uint64)
            assert g64.graph64_cost(w) == orc.graph_cost(g)
            assert np.array_equal(g64.graph64_action_kinds(w), orc.graph_action_kinds(g))
            for v, u in edges_of(g):
                assert g64.graph64_is_cut_edge(w, v, u) == orc.graph_is_cut_edge(g, v, u)


@pytest.mark.parametrize("n,p", [(40, 0.05), (64, 0.3), (64, 0.6)])
def test_relabelling(orc, n, p):
    """lambda_1 and mu are graph invariants; the kinds permute with the vertices."""
    rng = np.random.default_rng(n + int(10 * p))
    for _ in range(4):
        g = random_connected_graph64(rng, n, p)
        edges = edges_of(g)
        perm = rng.permutation(n)
        g2 = g64.graph64_from_edges(n, [(int(perm[a]), int(perm[b])) for a, b in edges])
        l1, mu, _ = g64.graph64_cost(g)
        l2, mu2, _ = g64.graph64_cost(g2)
        assert mu == mu2 and abs(l1 - l2) <= 1e-12 * l1
        k1, k2 = g64.graph64_action_kinds(g), g64.graph64_action_kinds(g2)
        e2 = n * (n - 1) // 2
        for v in range(n):
            for u in range(v):
                p1, p2 = orc.colex_position(v, u), orc.colex_position(int(perm[v]), int(perm[u]))
                for off in (0, e2):
                    assert _bit(k1, off + p1) == _bit(k2, off + p2)
