"""ctypes binding of the B64 bitset-graph oracle (tests/graph64_oracle.cpp): ConnectedBitsetGraph<N, B64>'s cost and
action kinds, N <= 64.  TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a cache directory outside the source tree ($AZB_GRAPH64_ORACLE_DIR, else the
system temporary directory), named after a hash of its sources, with the flags of oracle/Makefile.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "graph64_oracle.cpp")
_DEPS = [_SRC] + [os.path.join(os.path.dirname(_HERE), "oracle", f) for f in ("azb_oracle.cpp", "azb_oracle.h")]
_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-shared",
          "-Wno-subobject-linkage"]
_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    h = hashlib.sha256()
    for p in _DEPS:
        with open(p, "rb") as f:
            h.update(f.read())
    out_dir = os.environ.get("AZB_GRAPH64_ORACLE_DIR") or tempfile.gettempdir()
    path = os.path.join(out_dir, f"libazb_graph64_oracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(path):
        os.makedirs(out_dir, exist_ok=True)
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CXX", "g++"), *_FLAGS, "-o", tmp, _SRC])
        os.replace(tmp, path)
    L = C.CDLL(path)
    u32p, u64p = C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)
    L.orc_graph64_is_cut_edge.restype = C.c_int
    L.orc_graph64_is_cut_edge.argtypes = [C.c_uint32, u64p, C.c_uint32, C.c_uint32]
    L.orc_graph64_action_kinds.argtypes = [C.c_uint32, u64p, u32p]
    L.orc_graph64_matching_number.restype = C.c_uint32
    L.orc_graph64_matching_number.argtypes = [C.c_uint32, u64p]
    L.orc_graph64_lambda1.restype = C.c_double
    L.orc_graph64_lambda1.argtypes = [C.c_uint32, u64p]
    L.orc_graph64_cost.restype = C.c_int
    L.orc_graph64_cost.argtypes = [C.c_uint32, u64p, C.POINTER(C.c_double), u32p]
    _lib = L
    return L


def _u64(nbr):
    a = np.ascontiguousarray(nbr, dtype=np.uint64)
    return a, a.ctypes.data_as(C.POINTER(C.c_uint64))


def graph64_from_edges(n, edges):
    """Neighbourhood masks u64[n] of an edge list."""
    nbr = np.zeros(n, dtype=np.uint64)
    for u, v in edges:
        nbr[u] |= np.uint64(1 << v)
        nbr[v] |= np.uint64(1 << u)
    return nbr


def graph64_is_cut_edge(nbr, v, u) -> bool:
    a, p = _u64(nbr)
    return bool(lib().orc_graph64_is_cut_edge(a.shape[0], p, v, u))


def graph64_action_kinds(nbr):
    """Bit colex(e): Add(e) available; bit C(n,2)+colex(e): Delete(e) available, in ceil(n(n-1)/32) u32 words."""
    a, p = _u64(nbr)
    n = a.shape[0]
    out = np.zeros((n * (n - 1) + 31) // 32, dtype=np.uint32)
    lib().orc_graph64_action_kinds(n, p, out.ctypes.data_as(C.POINTER(C.c_uint32)))
    return out


def graph64_matching_number(nbr) -> int:
    a, p = _u64(nbr)
    return int(lib().orc_graph64_matching_number(a.shape[0], p))


def graph64_lambda1(nbr) -> float:
    """lambda_1 of A + 1e-4 I without the matching number (whose branch and bound is slow on sparse large graphs)."""
    a, p = _u64(nbr)
    return float(lib().orc_graph64_lambda1(a.shape[0], p))


def graph64_cost(nbr):
    """(lambda_1 of A + 1e-4 I, mu, rc) for one connected graph; rc = 1 where the reference asserts lambda_1 > 1.4."""
    a, p = _u64(nbr)
    lam, mu = C.c_double(), C.c_uint32()
    rc = lib().orc_graph64_cost(a.shape[0], p, C.byref(lam), C.byref(mu))
    return lam.value, mu.value, rc
