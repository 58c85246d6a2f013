"""A plain restatement of azb_trees_within (include/azb.h), written from the definition (not from the CUDA code): the
classes on s + 1 vertices are grown from those on s vertices by one leaf, starting from the two trees on 4 vertices;
each child is identified by observe.tree_code, evaluated on the canonical labelling decoded from its code, and kept
when its key (double)mu + lambda1 is <= bound + EPS below N and <= bound at N.  `cost(parents) -> (lambda1, mu)` is
the cost function (the tests pass the oracle's)."""
from __future__ import annotations

import numpy as np

from azdopt_b200 import observe

EPS = 1e-9
SEED = ((0, 0, 1, 0), (0, 0, 0, 0))  # the path and the star on 4 vertices


def decode(code, n: int) -> np.ndarray:
    """The canonical parent array u8[n] of a code: a 1 opens the next vertex under the current one, a 0 returns to the
    current vertex's parent; the first 1 is vertex 0."""
    bits = (int(code[0]) << 64) | int(code[1])
    par = np.zeros(n, dtype=np.uint8)
    cur, nxt = 0, 1
    for i in range(1, 2 * n - 1):
        if (bits >> (127 - i)) & 1:
            par[nxt] = cur
            cur, nxt = nxt, nxt + 1
        else:
            cur = int(par[cur])
    return par


def key_of(cost, parents) -> float:
    lam, mu = cost(parents)
    return float(mu) + float(lam)


def star_key(cost, n: int) -> float:
    return key_of(cost, np.zeros(n, dtype=np.uint8))


def trees_within(n: int, bound: float, cost):
    """(classes, sizes, evaluated): classes = [(key, code)] on n vertices with key <= bound, ascending; sizes = the level
    sizes for 5 .. n vertices; evaluated = the number of distinct children costed."""
    level = {observe.tree_code(p) for p in SEED}
    sizes, evaluated = [], 0
    for s in range(4, n):
        thr = bound if s + 1 == n else bound + EPS
        children = set()
        for code in level:
            par = [int(x) for x in decode(code, s)]
            for v in range(s):
                children.add(observe.tree_code(par + [v]))
        kept = {}
        for code in children:
            k = key_of(cost, decode(code, s + 1))
            evaluated += 1
            if k <= thr:
                kept[code] = k
        level = kept
        sizes.append(len(level))
        if not level:  # no tree on more vertices is within the bound either
            break
    return sorted((k, c) for c, k in level.items()), sizes, evaluated
