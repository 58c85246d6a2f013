"""Helpers of the canonical-code and best-trees tests: BFS relabelling of networkx trees into parent arrays with
parents[v] < v, random trees, and the host expectation of azb_best_trees built from tree dumps."""
import numpy as np


def parents_of(T, root=0):
    """Parent array (parents[v] < v) of a networkx tree, vertices renumbered in breadth-first order from `root`."""
    import networkx as nx

    order = [root] + [v for _, v in nx.bfs_edges(T, root)]
    idx = {v: i for i, v in enumerate(order)}
    p = np.zeros(len(order), dtype=np.uint8)
    for v in order[1:]:
        p[idx[v]] = min(idx[u] for u in T[v])
    return p


def random_parents(rng, n):
    """A uniform-attachment random tree: parents[v] uniform in 0..v-1."""
    p = np.zeros(n, dtype=np.uint8)
    for v in range(1, n):
        p[v] = rng.integers(0, v)
    return p


def relabel(rng, parents):
    """The same tree under a random labelling, back in parents[v] < v form (BFS from a random vertex)."""
    import networkx as nx

    n = len(parents)
    perm = rng.permutation(n)
    T = nx.Graph([(int(perm[v]), int(perm[parents[v]])) for v in range(1, n)])
    return parents_of(T, int(rng.integers(0, n)))


def replay(root_parents, root_permitted, key, n):
    """azb_get_node_state's rule on the host: the root with the key's actions replayed in ascending order."""
    p = np.array(root_parents, dtype=np.uint8).copy()
    m = np.array(root_permitted, dtype=np.uint32).copy()
    for w, word in enumerate(key):
        word = int(word)
        while word:
            b = (word & -word).bit_length() - 1
            word &= word - 1
            a = 32 * w + b
            child = 2
            while (child + 1) * child // 2 <= a + 1:
                child += 1
            first = child * (child - 1) // 2 - 1
            p[child] = a - first
            for q in range(first, first + child):
                m[q >> 5] &= np.uint32(~(1 << (q & 31)) & 0xFFFFFFFF)
    return p, m


def expected_best(h, k, first_root=0):
    """The azb_best_trees result from dumps of every tree, host replay and observe.tree_code: a list of
    (eval bits, code, tree, node, parents, permitted) ascending by (value, code)."""
    from azdopt_b200 import observe

    roots_p, roots_m = h.get_roots()
    best = {}
    for t in range(h.b):
        d = h.dump_tree(t)
        cbits = d["nodes"][:, 0]
        for i in range(len(cbits)):
            p, m = replay(roots_p[t], roots_m[t], d["keys"][i], h.n)
            code = observe.tree_code(p)
            c = float(np.uint32(cbits[i]).view(np.float32))
            key = (c, first_root + t, i)
            if code not in best or key < best[code][0]:
                best[code] = (key, int(cbits[i]), t, i, p, m)
    rows = sorted(best.items(), key=lambda kv: (kv[1][0][0], kv[0]))[:k]
    return [(v[1], code, v[2], v[3], v[4], v[5]) for code, v in rows]
