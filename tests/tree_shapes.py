"""Tree shapes that drive the c21 cost kernel to its limits, and an exact reference for lambda_1 and mu (plain Python,
no GPU).  TEST INFRASTRUCTURE ONLY.

Every family gives, for any n >= 5, a parent array with parents[v] < v.  Two of them are built for the section method's
stack program (azb_cost.cuh, azb_cost_prepare): the stack-extremal trees fill all the stack levels the kernel allows at
n = 22, 23, 46, 47 and 64, and the comb of cherries has the longest program (94 ops at n = 64).

The exact lambda_1 counts eigenvalues by Sylvester's law of inertia (Jacobs and Trevisan, "Locating the eigenvalues of
trees", 2011) in exact integer arithmetic and bisects, so it shares neither the kernel's floating point nor its
Laguerre or sectioning steps, and stays right where lambda_1 and lambda_2 are closer than f64 can tell.
"""
from __future__ import annotations

import math
from fractions import Fraction

import numpy as np

from azdopt_b200 import observe


# ---- shape families ---------------------------------------------------------------------------------------------------
def star(n):
    return np.zeros(n, dtype=np.uint8)


def path(n):
    return np.maximum(np.arange(n) - 1, 0).astype(np.uint8)


def double_star(n):
    """Two adjacent centres 0 and 1, the other vertices split between them as leaves."""
    p = np.zeros(n, dtype=np.uint8)
    p[2 + (n - 2 + 1) // 2:] = 1
    return p


def broom(n):
    """A path on n // 2 vertices with the other vertices as leaves on its far end."""
    h = n // 2
    p = path(n)
    p[h:] = h - 1
    return p


def caterpillar(n):
    """A spine on n // 3 vertices; the other vertices hang on the spine in turn."""
    s = n // 3
    p = path(n)
    p[s:] = (np.arange(s, n) - s) % s
    return p


def spider(n):
    """Legs of 3 vertices on centre 0 (plus (n - 1) % 3 single leaves): the legs' codes tie."""
    p = np.zeros(n, dtype=np.uint8)
    legs = (n - 1) // 3
    for j in range(legs):
        a = 1 + 3 * j
        p[a], p[a + 1], p[a + 2] = 0, a, a + 1
    return p


def dumbbell(n):
    """Two stars with max(1, n // 4) leaves each, their centres joined by a path: lambda_1 and lambda_2 nearly equal."""
    k = max(1, n // 4)
    length = n - 2 * k  # path vertices 0 .. length-1, both ends are the stars' centres
    p = path(n)
    p[length:length + k] = 0
    p[length + k:] = length - 1
    return p


def binary(n):
    """The complete binary tree in heap order."""
    return np.maximum((np.arange(n) - 1) // 2, 0).astype(np.uint8)


def t_k(k):
    """Stack-extremal T(k) in preorder: T(1) is a vertex with one leaf, T(k) a root with two T(k-1).  It has
    3 * 2^(k-1) - 1 vertices (2, 5, 11, 23, 47) and its stack program needs exactly k slots."""
    if k == 1:
        return [0, 0]
    sub = t_k(k - 1)
    out = [0]
    for _ in range(2):
        off = len(out)
        out += [0 if v == 0 else off + q for v, q in enumerate(sub)]
    return out


def stack_extremal(n):
    """The largest T(k) with at most n vertices, padded with leaves on its root: 3 slots at n = 22, 4 at n = 23 and 46,
    5 at n = 47 to 64."""
    k = 1
    while 3 * 2 ** k - 1 <= n:
        k += 1
    t = t_k(k)
    return np.array(t + [0] * (n - len(t)), dtype=np.uint8)


def longest_program(n):
    """A root with a comb of cherries (a vertex and its leaf), plus one leaf when n is even:
    n + (n - 1) // 2 - 1 ops, 94 at n = 64."""
    p = np.zeros(n, dtype=np.uint8)
    for a in range(1, n - 1, 2):
        p[a + 1] = a
    return p


FAMILIES = {f.__name__: f for f in (star, path, double_star, broom, caterpillar, spider, dumbbell, binary,
                                     stack_extremal, longest_program)}


# ---- the stack program (restated from the comments in azb_cost_prepare) ------------------------------------------------
def _children(parents):
    ch = [[] for _ in range(len(parents))]
    for v in range(1, len(parents)):
        ch[int(parents[v])].append(v)
    return ch


def slots(parents):
    """Slots the stack program needs (the Sethi-Ullman number of the root): an internal vertex needs
    max(s1, 1 + s2), s1 >= s2 the two largest needs of its internal children (0 where there are none)."""
    ch = _children(parents)
    su = [0] * len(parents)
    for v in range(len(parents) - 1, -1, -1):
        need = sorted((su[c] for c in ch[v] if ch[c]), reverse=True) + [0, 0]
        su[v] = max(need[0], 1 + need[1])
    return su[0]


def program_length(parents):
    """Ops of the program, OP_END included: a leaf child is one op, the heaviest internal child its own ops and OP_T,
    every other internal child its ops between PUSH and POPF."""
    ch = _children(parents)
    ln = [0] * len(parents)
    for v in range(len(parents) - 1, -1, -1):
        internal = [c for c in ch[v] if ch[c]]
        ln[v] = (len(ch[v]) - len(internal)) + sum(ln[c] + 2 for c in internal) - (1 if internal else 0)
    return ln[0] + 1


def stack_depth(n):
    """Stack levels the kernel allows at n vertices (azb_stack_depth)."""
    return 3 if n <= 22 else (4 if n <= 46 else 5)


# ---- random trees and labellings --------------------------------------------------------------------------------------
def _from_edges(n, edges, rng=None, root=0):
    """Parent array of the tree with these edges: labels in a parent-before-child order from `root`; with `rng` the
    next vertex is drawn from all vertices whose parent is labelled, otherwise breadth first."""
    adj = [[] for _ in range(n)]
    for u, v in edges:
        adj[u].append(v)
        adj[v].append(u)
    label = {root: 0}
    up = {root: root}
    frontier = [u for u in adj[root]]
    for u in frontier:
        up[u] = root
    p = np.zeros(n, dtype=np.uint8)
    while frontier:
        u = frontier.pop(int(rng.integers(0, len(frontier))) if rng is not None else 0)
        label[u] = len(label)
        p[label[u]] = label[up[u]]
        for w in adj[u]:
            if w not in label and w not in up:
                up[w] = u
                frontier.append(w)
    assert len(label) == n, "not a tree"
    return p


def edges_of(parents):
    return [(v, int(parents[v])) for v in range(1, len(parents))]


def random_tree(n, rng):
    """A uniform labelled tree on n vertices (Pruefer decoding), as a parent array."""
    seq = [int(x) for x in rng.integers(0, n, size=n - 2)]
    deg = [1] * n
    for x in seq:
        deg[x] += 1
    edges = []
    for x in seq:
        leaf = min(v for v in range(n) if deg[v] == 1)
        edges.append((leaf, x))
        deg[leaf] -= 1
        deg[x] -= 1
    u, v = (w for w in range(n) if deg[w] == 1)
    edges.append((u, v))
    return _from_edges(n, edges)


def relabel(parents, rng):
    """The same tree from a random root in a random parent-before-child order: another op program, other heavy-child
    ties and another vertex order in the kernel's passes."""
    n = len(parents)
    return _from_edges(n, edges_of(parents), rng=rng, root=int(rng.integers(0, n)))


# ---- exact lambda_1 ---------------------------------------------------------------------------------------------------
SCALE = 120  # x = X / 2^SCALE: every point the bisection visits is exact


def eigen_count_above(parents, X):
    """Number of eigenvalues of the adjacency matrix greater than x = X / 2^SCALE, exactly.

    Jacobs-Trevisan Diagonalize(T, -x): leaves first, a(v) = -x - sum over children of 1 / a(c); where a child has
    a(c) = 0, a(v) = -1/2, a(c) = 2 and v is cut from its parent.  The diagonal is congruent to A - x I, so its
    positive entries count the eigenvalues above x.  a(v) is kept as an unreduced integer fraction."""
    ch = _children(parents)
    n = len(parents)
    num, den = [0] * n, [0] * n
    cut = [False] * n
    for v in range(n - 1, -1, -1):  # parents[v] < v: every child is final before its parent
        zero = next((c for c in ch[v] if num[c] == 0), None)
        if zero is not None:
            num[zero], den[zero] = 2, 1
            num[v], den[v] = -1, 2
            cut[v] = True
            continue
        a, b = -X, 1 << SCALE
        for c in ch[v]:
            if not cut[c]:
                a, b = a * num[c] - b * den[c], b * num[c]
        num[v], den[v] = a, b
    return sum(1 for v in range(n) if (num[v] > 0) == (den[v] > 0) and num[v] != 0)


def lambda1_dense(parents):
    n = len(parents)
    a = np.zeros((n, n))
    for v, u in edges_of(parents):
        a[v, u] = a[u, v] = 1.0
    return float(np.linalg.eigvalsh(a)[-1])


_CACHE = {}


def exact_lambda1(parents):
    """(lambda_1 correctly rounded to f64, lo, hi): lo < lambda_1 <= hi are exact Fractions less than 2^-92 apart.
    Cached by canonical code: lambda_1 does not depend on the labelling."""
    key = observe.tree_code(parents)
    if key in _CACHE:
        return _CACHE[key]
    guess = lambda1_dense(parents)
    lo = int(Fraction(guess * (1 - 1e-12)) * 2 ** SCALE)
    hi = int(Fraction(guess * (1 + 1e-12)) * 2 ** SCALE) + 1
    if eigen_count_above(parents, hi) != 0 or eigen_count_above(parents, lo) < 1:
        raise AssertionError(f"lambda_1 is not within 1e-12 of eigvalsh's {guess!r}")
    # lambda_1 is in (lo, hi]: bisect to 2^-92, then on until both ends round to the same double
    while hi - lo > 1 << (SCALE - 92) or lo / 2 ** SCALE != hi / 2 ** SCALE:
        if hi - lo < 2:
            raise AssertionError("lambda_1 is a rounding tie")  # only integers are rational eigenvalues here
        mid = (lo + hi) // 2
        if eigen_count_above(parents, mid) == 0:
            hi = mid
        else:
            lo = mid
    out = (hi / 2 ** SCALE, Fraction(lo, 2 ** SCALE), Fraction(hi, 2 ** SCALE))
    _CACHE[key] = out
    return out


def ulps(value, parents):
    """|value - lambda_1| in units in the last place of the correctly rounded lambda_1."""
    r, lo, hi = exact_lambda1(parents)
    return float(abs(Fraction(value) - (lo + hi) / 2) / Fraction(math.ulp(r)))


def near_f32_boundary(parents, k=4):
    """True if lambda_1 lies within k f64 ulps of a point where the rounding to f32 changes."""
    r, lo, hi = exact_lambda1(parents)
    u = Fraction(math.ulp(r)) * k
    return np.float32(float(lo - u)) != np.float32(float(hi + u))


# ---- exact mu ---------------------------------------------------------------------------------------------------------
def _pmul(a, b):
    out = [0] * (len(a) + len(b) - 1)
    for i, x in enumerate(a):
        if x:
            for j, y in enumerate(b):
                out[i + j] += x * y
    return out


def _padd(a, b):
    if len(a) < len(b):
        a, b = b, a
    return [x + (b[i] if i < len(b) else 0) for i, x in enumerate(a)]


def exact_mu(parents):
    """The matching number: the degree of the matching polynomial.  Leaves first, a_v counts the matchings of the
    subtree of v and b_v those that leave v free, by size; folding a child c: b <- b a_c, a <- a a_c + x b b_c."""
    ch = _children(parents)
    n = len(parents)
    a, b = [None] * n, [None] * n
    for v in range(n - 1, -1, -1):
        av, bv = [1], [1]
        for c in ch[v]:
            av, bv = _padd(_pmul(av, a[c]), [0] + _pmul(bv, b[c])), _pmul(bv, a[c])
        a[v], b[v] = av, bv
    return max(k for k, m in enumerate(a[0]) if m > 0)


# ---- the inputs of the tests ------------------------------------------------------------------------------------------
BOUNDARY_N = (5, 21, 22, 23, 24, 32, 33, 45, 46, 47, 48, 63, 64)


def shape_batch(n, relabellings=3, pruefer=20, seed=0):
    """[(name, parents)] at n: every family and `relabellings` relabellings of each, and `pruefer` uniform trees when
    n is a boundary of the kernel (BOUNDARY_N).  A relabelled copy keeps its family's name."""
    rng = np.random.default_rng(1000 * seed + n)
    out = []
    for name, f in FAMILIES.items():
        p = f(n)
        out.append((name, p))
        out += [(name, relabel(p, rng)) for _ in range(relabellings)]
    if n in BOUNDARY_N:
        out += [(f"pruefer{i}", random_tree(n, rng)) for i in range(pruefer)]
    return out
