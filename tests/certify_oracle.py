"""ctypes binding of the CPU restatement of the c21 key certificates (tests/certify_oracle.cpp): bit-identical to
azb_certify_keys.  TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a cache directory outside the source tree ($AZB_CERTIFY_ORACLE_DIR, else the
system temporary directory), named after a hash of its source, with the flags of oracle/Makefile and -frounding-math.
kernel_unproven runs the grow-side kernel itself through tests/certify_kernel_harness.cu, compiled the same way with
the library's nvcc flags (it needs a GPU to run).
"""
from __future__ import annotations

import ctypes as C
import hashlib
import math
import os
import subprocess
import tempfile
from fractions import Fraction
from math import isqrt

import numpy as np

import tree_shapes as ts

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "certify_oracle.cpp")
_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-frounding-math", "-pthread", "-shared"]
_lib = None
_harness = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    with open(_SRC, "rb") as f:
        digest = hashlib.sha256(f.read() + " ".join(_FLAGS).encode()).hexdigest()[:16]
    out_dir = os.environ.get("AZB_CERTIFY_ORACLE_DIR") or tempfile.gettempdir()
    path = os.path.join(out_dir, f"libazb_certify_oracle_{digest}.so")
    if not os.path.exists(path):
        os.makedirs(out_dir, exist_ok=True)
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CXX", "g++"), *_FLAGS, "-o", tmp, _SRC])
        os.replace(tmp, path)
    L = C.CDLL(path)
    u8p, u32p, f64p = C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_double)
    L.orc_cert_jt.restype = C.c_int
    L.orc_cert_jt.argtypes = [u8p, C.c_uint32, C.c_double]
    L.orc_cert_mu.restype = C.c_uint32
    L.orc_cert_mu.argtypes = [u8p, C.c_uint32]
    L.orc_cert_points.argtypes = [C.c_uint32, C.c_uint32, C.c_double, f64p, f64p]
    L.orc_cert_unproven.restype = C.c_int
    L.orc_cert_unproven.argtypes = [u8p, C.c_uint32, C.c_uint32, C.c_double, C.c_uint32, C.c_double, C.c_double]
    L.orc_certify.argtypes = [u8p, C.c_uint32, C.c_uint32, f64p, C.c_double, f64p, f64p, u32p, C.POINTER(C.c_int8)]
    _lib = L
    return L


def _u8(parents):
    a = np.ascontiguousarray(parents, dtype=np.uint8)
    return a, a.ctypes.data_as(C.POINTER(C.c_uint8))


def jt(parents, x) -> int:
    """The interval inertia count at x: the number of eigenvalues above x, or -1 when undecided."""
    a, p = _u8(parents)
    return int(lib().orc_cert_jt(p, a.shape[-1], float(x)))


def greedy_mu(parents) -> int:
    a, p = _u8(parents)
    return int(lib().orc_cert_mu(p, a.shape[-1]))


def points(n, mu, bound):
    """(t_lo, t_hi) around bound - mu; bound < 0 is sqrt(n - 1) + 1."""
    lo, hi = C.c_double(), C.c_double()
    lib().orc_cert_points(n, mu, float(bound), C.byref(lo), C.byref(hi))
    return lo.value, hi.value


def unproven(parents, lambda1, mu_cost, thr, bound, N) -> bool:
    """azb_certify_pruned_kernel's decision: the keep test at thr drops the class and key > bound is not proven."""
    a, p = _u8(parents)
    return bool(lib().orc_cert_unproven(p, a.shape[-1], N, float(lambda1), int(mu_cost), float(thr), float(bound)))


def kernel_unproven(parents, lambda1, mu_cost, thr, bound, N):
    """azb_certify_pruned_kernel's decision for each class u8[m, n] (one launch per class), as bool[m]."""
    global _harness
    if _harness is None:
        import importlib

        build = importlib.import_module("azdopt_b200.build")  # the module; the package exports its build() under that name

        here = os.path.dirname(_SRC)
        src = os.path.join(here, "certify_kernel_harness.cu")
        deps = [src] + [os.path.join(here, "..", "azdopt_b200", "csrc", f) for f in ("azb_certify.cuh", "azb_common.cuh")]
        h = hashlib.sha256(" ".join(build.NVCC_FLAGS).encode())
        for d in deps:
            with open(d, "rb") as f:
                h.update(f.read())
        out_dir = os.environ.get("AZB_CERTIFY_ORACLE_DIR") or tempfile.gettempdir()
        path = os.path.join(out_dir, f"libazb_certify_harness_{h.hexdigest()[:16]}.so")
        if not os.path.exists(path):
            os.makedirs(out_dir, exist_ok=True)
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.check_call([build._nvcc(), *build.NVCC_FLAGS, "-o", tmp, src])
            os.replace(tmp, path)
        _harness = C.CDLL(path)
        _harness.harness_unproven.restype = C.c_int
        _harness.harness_unproven.argtypes = [C.POINTER(C.c_uint8), C.c_uint32, C.c_uint32, C.POINTER(C.c_double),
                                              C.POINTER(C.c_uint32), C.POINTER(C.c_double), C.c_double, C.c_uint32,
                                              C.POINTER(C.c_uint8)]
    a, p = _u8(parents)
    m, n = a.shape
    l1 = np.ascontiguousarray(lambda1, dtype=np.float64)
    mu = np.ascontiguousarray(mu_cost, dtype=np.uint32)
    th = np.ascontiguousarray(thr, dtype=np.float64)
    out = np.zeros(m, dtype=np.uint8)
    rc = _harness.harness_unproven(p, m, n, l1.ctypes.data_as(C.POINTER(C.c_double)), mu.ctypes.data_as(C.POINTER(C.c_uint32)),
                                   th.ctypes.data_as(C.POINTER(C.c_double)), float(bound), N,
                                   out.ctypes.data_as(C.POINTER(C.c_uint8)))
    assert rc == 0, f"CUDA error {rc}"
    return out.astype(bool)


def grow_with_proof(n, bound, cost):
    """trees_within_ref.trees_within(n, bound) with azb_trees_within_proof's grow side restated: (classes, unproven,
    dropped), unproven = proof[4] when every level is one chunk (each distinct child is costed once), dropped = [(parents,
    lambda1, mu, is_unproven)] for every class the keep test dropped.  bound < 0: the star's computed key filters,
    sqrt(n - 1) + 1 is what is proven against.  cost(parents) -> (lambda1, mu) as for trees_within_ref."""
    import trees_within_ref as W

    fbound = W.star_key(cost, n) if bound < 0 else bound
    seen = []

    def recording(parents):
        lam, mu = cost(parents)
        seen.append((np.array(parents, dtype=np.uint8), lam, mu))
        return lam, mu

    classes, _, _ = W.trees_within(n, fbound, recording)
    dropped, count = [], 0
    for p, lam, mu in seen:
        thr = fbound if len(p) == n else fbound + W.EPS
        if not float(mu) + float(lam) <= thr:
            u = unproven(p, lam, mu, thr, bound, n)
            dropped.append((p, lam, mu, u))
            count += u
    return classes, count, dropped


SHIFTS = (0, 1, 3, 64, 1 << 20, -1, -3, -64, -(1 << 20))


def pruned_cases(cost, ns=(10, 14, 24, 33, 64)):
    """Inputs for the grow-side decision, including ones the cost kernel never gives: every family of
    tree_shapes.shape_batch(n) in its canonical labelling, its lambda_1 moved by SHIFTS ulps, a threshold one double below
    the key so the keep test drops it, and as bound that threshold or sqrt(n - 1) + 1: [(parents, c, mu, thr, bound, n)]."""
    import trees_within_ref as W
    from azdopt_b200 import observe

    cases = []
    for n in ns:
        for _, p in ts.shape_batch(n, relabellings=0):
            q = W.decode(observe.tree_code(p), n)
            lam, mu = cost(q)
            for k in SHIFTS:
                c = float(lam) + k * math.ulp(lam)
                thr = math.nextafter(float(mu) + c, -math.inf)
                for bound in (thr, -1.0):
                    cases.append((q, c, int(mu), thr, bound, n))
    return cases


def certify(parents, lambda1, bound=-1.0):
    """dict lambda1_lo, lambda1_hi (f64), mu (u32), verdict (i8) for trees u8[m, n] with the cost kernel's lambda1."""
    a, p = _u8(np.atleast_2d(parents))
    m, n = a.shape
    c = np.ascontiguousarray(lambda1, dtype=np.float64)
    assert c.shape == (m,)
    out = dict(lambda1_lo=np.zeros(m), lambda1_hi=np.zeros(m), mu=np.zeros(m, dtype=np.uint32),
               verdict=np.zeros(m, dtype=np.int8))
    f64p = C.POINTER(C.c_double)
    lib().orc_certify(p, m, n, c.ctypes.data_as(f64p), float(bound), out["lambda1_lo"].ctypes.data_as(f64p),
                      out["lambda1_hi"].ctypes.data_as(f64p), out["mu"].ctypes.data_as(C.POINTER(C.c_uint32)),
                      out["verdict"].ctypes.data_as(C.POINTER(C.c_int8)))
    return out


# ---- the exact answer the certificates are checked against ----------------------------------------------------------
def _x(t):
    """t as the integer X of tree_shapes.eigen_count_above (t = X / 2^SCALE)."""
    q = Fraction(t) * 2 ** ts.SCALE
    assert q.denominator == 1, f"{t!r} is not a multiple of 2^-{ts.SCALE}"
    return int(q)


def above(parents, t) -> int:
    """The exact number of eigenvalues above the dyadic t."""
    return ts.eigen_count_above(parents, _x(t))


def char_poly_at(parents, t):
    """det(t I - A) exactly: for a tree it is the matching polynomial, sum_k (-1)^k m_k t^(n - 2k)."""
    ch = ts._children(parents)
    n = len(parents)
    a, b = [None] * n, [None] * n
    for v in range(n - 1, -1, -1):
        av, bv = [1], [1]
        for c in ch[v]:
            av, bv = ts._padd(ts._pmul(av, a[c]), [0] + ts._pmul(bv, b[c])), ts._pmul(bv, a[c])
        a[v], b[v] = av, bv
    t = Fraction(t)
    return sum((-1) ** k * m * t ** (n - 2 * k) for k, m in enumerate(a[0]))


def exact_sign(parents, bound):
    """The sign of key - bound, key = mu + lambda_1 as real numbers, bound < 0 meaning sqrt(n - 1) + 1: -1, 0 or +1,
    or None where 2^-100 cannot separate them (lambda_1 irrational and that close to an irrational bound)."""
    n = len(parents)
    mu = ts.exact_mu(parents)
    if bound < 0.0:
        s = isqrt(n - 1)
        if s * s != n - 1:
            if mu == 1:
                return 0  # the star: lambda_1 = sqrt(n - 1)
            q = isqrt((n - 1) << 200)
            t_lo, t_hi = Fraction(q, 1 << 100) + 1 - mu, Fraction(q + 1, 1 << 100) + 1 - mu
            if ts.eigen_count_above(parents, int(t_hi * 2 ** ts.SCALE)) >= 1:
                return 1
            if ts.eigen_count_above(parents, int(t_lo * 2 ** ts.SCALE)) == 0:
                return -1
            return None
        t = Fraction(s + 1 - mu)
    else:
        t = Fraction(bound) - mu
    if above(parents, t) >= 1:
        return 1
    return 0 if char_poly_at(parents, t) == 0 else -1  # lambda_1 <= t, and equal iff t is an eigenvalue
