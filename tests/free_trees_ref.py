"""A plain restatement of the free-tree enumeration defined in include/azb.h, written from the definition (not from the
CUDA code): rooted trees by global id (size first, then their non-increasing child-id sequences in lexicographic order),
free trees rooted at their centroid (unicentroidal sequences first, then for even n the pairs i >= j of rooted trees of
size n / 2), preorder labels with children in sequence order."""
from __future__ import annotations

import bisect
import functools
import math

import numpy as np

NMAX = 32
SMAX = NMAX // 2


@functools.lru_cache(maxsize=None)
def _tables():
    """(starts, P): starts[s - 1] = first global id of size s for s = 1..SMAX + 1; P[r, g] (r < NMAX, g over the ids of
    size <= (NMAX - 1) // 2) = the number of non-increasing sequences of ids <= g whose sizes sum to r."""
    starts = [0]
    last = np.zeros(NMAX, dtype=np.int64)  # P[:, g - 1]; P[r, -1] = 1 for the empty sequence (r = 0)
    last[0] = 1
    blocks = []
    for s in range(1, SMAX + 1):
        count = int(last[s - 1])  # A000081(s): sequences of sum s - 1, every id of size < s already counted
        starts.append(starts[-1] + count)
        if s > (NMAX - 1) // 2:
            break
        blk = np.empty((NMAX, count), dtype=np.int64)
        for r in range(NMAX):  # P[r, g] = P[r, g - 1] + P[r - s, g], g running over the ids of size s
            blk[r] = last[r] + (np.cumsum(blk[r - s]) if r >= s else 0)
        blocks.append(blk)
        last = blk[:, -1].copy()
    return starts, np.concatenate(blocks, axis=1)


def size_of(g: int) -> int:
    starts, _ = _tables()
    return bisect.bisect_right(starts, g)


def rooted_count(s: int) -> int:
    starts, _ = _tables()
    return starts[s] - starts[s - 1]


def _sequence(r: int, x: int, bound: int):
    """The x-th (0-based) non-increasing sequence of ids <= bound with size sum r, in lexicographic order."""
    _, P = _tables()
    out = []
    while r > 0:
        row = P[r]
        g = int(np.searchsorted(row[:bound + 1], x, side="right"))  # first g with P[r, g] > x
        if g:
            x -= int(row[g - 1])
        out.append(g)
        r -= size_of(g)
        bound = g
    return out


def _attach(par: list, sub) -> None:
    base = len(par)
    par.append(0)
    par.extend(base + p for p in sub[1:])


@functools.lru_cache(maxsize=None)
def rooted(g: int) -> tuple:
    """Preorder parent array of the rooted tree with global id g."""
    starts, _ = _tables()
    s = size_of(g)
    par = [0]
    if s > 1:
        for c in _sequence(s - 1, g - starts[s - 1], starts[s - 1] - 1):
            _attach(par, rooted(c))
    return tuple(par)


def unicentroidal_count(n: int) -> int:
    starts, P = _tables()
    return int(P[n - 1, starts[(n - 1) // 2] - 1])


def free_tree_count(n: int) -> int:
    t = rooted_count(n // 2) if n % 2 == 0 else 0
    return unicentroidal_count(n) + t * (t + 1) // 2


def free_tree(n: int, idx: int) -> np.ndarray:
    """Parent array u8[n] of the free tree with index idx."""
    starts, _ = _tables()
    u = unicentroidal_count(n)
    if not 0 <= idx < free_tree_count(n):
        raise IndexError(idx)
    if idx < u:
        par = [0]
        for c in _sequence(n - 1, idx, starts[(n - 1) // 2] - 1):
            _attach(par, rooted(c))
    else:
        rem = idx - u
        i = (math.isqrt(8 * rem + 1) - 1) // 2
        j = rem - i * (i + 1) // 2
        h = n // 2
        ti, tj = rooted(starts[h - 1] + i), rooted(starts[h - 1] + j)
        par = [0]
        _attach(par, tj)
        par.extend(0 if p == 0 else h + p for p in ti[1:])
    return np.array(par, dtype=np.uint8)


def free_trees(n: int, start: int, m: int) -> np.ndarray:
    return np.stack([free_tree(n, i) for i in range(start, start + m)]) if m else np.zeros((0, n), np.uint8)
