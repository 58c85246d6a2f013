"""Connected graphs on up to 64 vertices as u64 neighbourhood masks (test helper; shared by the CPU and GPU tests of
azb_eval_graph_costs64 and by tools/graph64_probe.py)."""
import math

import numpy as np


def random_connected_graph64(rng, n, p):
    """A random spanning tree plus G(n, p) edges: u64[n] neighbourhood masks (n <= 64)."""
    nbr = np.zeros(n, dtype=np.uint64)
    order = rng.permutation(n)
    for i in range(1, n):
        a, b = int(order[i]), int(order[rng.integers(0, i)])
        nbr[a] |= np.uint64(1 << b)
        nbr[b] |= np.uint64(1 << a)
    extra = np.triu(rng.random((n, n)) < p, 1)
    for a, b in zip(*np.nonzero(extra)):
        nbr[a] |= np.uint64(1 << int(b))
        nbr[b] |= np.uint64(1 << int(a))
    return nbr


def named_graphs64():
    """(name, n, edges, lambda_1 of A or None, mu) on 33..64 vertices; None: no closed form, compare with LAPACK."""
    out = []
    for n in (33, 48, 64):
        out.append((f"path{n}", n, [(i, i + 1) for i in range(n - 1)], 2 * math.cos(math.pi / (n + 1)), n // 2))
        out.append((f"star{n}", n, [(0, i) for i in range(1, n)], math.sqrt(n - 1), 1))
        out.append((f"complete{n}", n, [(i, j) for i in range(n) for j in range(i)], float(n - 1), n // 2))
        out.append((f"cycle{n}", n, [(i, (i + 1) % n) for i in range(n)], 2.0, n // 2))
    for a, b in ((1, 63), (32, 32), (5, 40)):
        out.append((f"K{a},{b}", a + b, [(i, a + j) for i in range(a) for j in range(b)], math.sqrt(a * b), min(a, b)))
    # Petersen graph (vertices 0..9) with a path 9-10-...-63 hung on vertex 9: mu = 5 + 27 (the Petersen graph's perfect
    # matching and every second path edge)
    pet = [(i, (i + 1) % 5) for i in range(5)] + [(i, i + 5) for i in range(5)] + [(5 + i, 5 + (i + 2) % 5) for i in range(5)]
    out.append(("petersen+path64", 64, pet + [(i, i + 1) for i in range(9, 63)], None, 32))
    return out


def lambda1_lapack(n, edges):
    """Largest eigenvalue of the adjacency matrix (numpy.linalg.eigvalsh)."""
    a = np.zeros((n, n))
    for v, u in edges:
        a[v, u] = a[u, v] = 1.0
    return float(np.linalg.eigvalsh(a)[-1])
