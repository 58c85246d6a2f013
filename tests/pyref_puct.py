"""Independent pure-Python restatement of the PUCT selection mode (include/azb.h, AZB_SELECT_PUCT), for SMALL cases.

The rule is this project's own: the reference has no PUCT, so there is nothing upstream to restate.  It is written
here from the rule's text (not from oracle/azb_oracle.cpp) in numpy float32 scalars, one rounding per operation, on
top of tests/pyref.py's search DAG: only next_action changes, everything after the choice is pyref's.
"""
from __future__ import annotations

import numpy as np

import pyref

F = np.float32


def butterfly_sum(chunk):
    """Sum of at most 32 values as a warp's xor butterfly forms it: lane i holds chunk[i] (+0 beyond its end); for
    m = 16, 8, 4, 2, 1 every lane adds the value of lane i ^ m at once; lane 0's value is the sum."""
    x = [F(v) for v in chunk] + [F(0)] * (32 - len(chunk))
    for m in (16, 8, 4, 2, 1):
        x = [F(x[i] + x[i ^ m]) for i in range(32)]
    return x[0]


def prior_sum(w):
    """Z: butterfly sums of the 32-value chunks, folded left to right from chunk 0's."""
    z = None
    for base in range(0, len(w), 32):
        s = butterfly_sum(w[base:base + 32])
        z = s if z is None else F(z + s)
    return z


class PuctError(Exception):
    def __init__(self, code):
        super().__init__(code)
        self.code = code  # 3: N_s reached 2^24, 4: NaN score, 6: no candidate at an active node


class PuctTree(pyref.Tree):
    c_puct = F(1)

    def __init__(self):
        super().__init__()
        self.k = dict(n_sel=0, d_sel=0, n_cur=0, n_cand=0)

    def next_action(self, pos, tol):  # tol (n_as_tol) is not consulted
        node = self.nodes[pos]
        if not node.active():
            return None
        kids = [self.arcs[e][1] for e in node.out]
        cnt = node.hi - node.lo
        self.k["n_sel"] += 1
        self.k["d_sel"] += len(kids)
        self.k["n_cur"] += 1
        self.k["n_cand"] += cnt
        n_s = 1 + sum(self.nodes[d].nt + 1 for d in kids)
        if n_s >= 1 << 24:
            raise PuctError(3)
        sq = F(np.sqrt(F(n_s)))
        c_s = node.c
        w = []
        for j in range(node.lo, node.hi):
            x = F(F(F(1) - c_s) + self.preds[j][1])
            w.append(F(0) if x < 0 else x)
        z = prior_sum(w)
        best = None
        for i, j in enumerate(range(node.lo, node.hi)):
            a, g, arc = self.preds[j]
            p = F(F(1) / F(cnt)) if z == 0 else F(w[i] / z)
            if arc is None:
                n, q = 0, g
            else:
                kid = self.nodes[self.arcs[arc][1]]
                assert self.preds[self.arcs[arc][2]][0] == a
                if not kid.active():
                    continue
                n, q = kid.nt + 1, F(c_s - kid.cstar)
            score = F(q + F(F(F(self.c_puct * p) * sq) / F(1 + n)))
            if np.isnan(score):
                raise PuctError(4)
            if best is None or score > best[0]:  # first maximum
                best = (score, j, arc)
        if best is None:
            raise PuctError(6)
        return ("V", best[2]) if best[2] is not None else ("U", best[1])


class Optimizer(pyref.Optimizer):
    """pyref.Optimizer with PUCT selection."""

    def __init__(self, n, parents, permitted_lists, c_puct=1.0):
        super().__init__(n, parents, permitted_lists)
        self.c_puct = F(c_puct)

    def init_trees(self, priors):
        super().init_trees(priors)
        for t in self.trees:  # pyref builds plain Trees; only their selection changes
            t.__class__ = PuctTree
            t.c_puct = self.c_puct
            t.k = dict(n_sel=0, d_sel=0, n_cur=0, n_cand=0)

    def counters(self):
        out = dict(n_sel=0, d_sel=0, n_cur=0, n_cand=0)
        for t in self.trees:
            for key in out:
                out[key] += t.k[key]
        return out
