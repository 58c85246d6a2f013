"""ctypes binding of the PUCT oracle (tests/puct_oracle.cpp): the CPU oracle with include/azb.h's AZB_SELECT_PUCT rule
in place of the reference's next_action.  TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a cache directory outside the source tree ($AZB_PUCT_ORACLE_DIR, else the
system temporary directory), named after a hash of its sources, with the flags of oracle/Makefile.  Its two entry
points work on a handle of oracle/libazb_oracle.so; everything else (roots, priors, dumps, counters) goes through
oracle.Optimizer unchanged.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "puct_oracle.cpp")
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
    out_dir = os.environ.get("AZB_PUCT_ORACLE_DIR") or tempfile.gettempdir()
    path = os.path.join(out_dir, f"libazb_puct_oracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(path):
        os.makedirs(out_dir, exist_ok=True)
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CXX", "g++"), *_FLAGS, "-o", tmp, _SRC])
        os.replace(tmp, path)
    L = C.CDLL(path)
    L.orc_puct_rollout.restype = C.c_int
    L.orc_puct_rollout.argtypes = [C.c_void_p, C.c_float, C.POINTER(C.c_float)]
    L.orc_puct_steps_hash.restype = C.c_int
    L.orc_puct_steps_hash.argtypes = [C.c_void_p, C.c_float, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32,
                                      C.POINTER(C.c_uint32), C.c_uint32, C.POINTER(C.c_uint32)]
    _lib = L
    return L


class PuctOptimizer(oracle.Optimizer):
    """oracle.Optimizer whose walks select with PUCT at constant c_puct (finite, > 0)."""

    def __init__(self, n, n_roots, c_puct=1.0, **kw):
        self._h = None
        if not (math.isfinite(c_puct) and c_puct > 0):
            raise ValueError(f"c_puct={c_puct}: must be finite and > 0")
        super().__init__(n, n_roots, **kw)
        self.c_puct = float(c_puct)
        lib()

    def rollout(self, state_vecs=None):
        ptr = state_vecs.ctypes.data_as(C.POINTER(C.c_float)) if state_vecs is not None else None
        rc = lib().orc_puct_rollout(self._h, self.c_puct, ptr)
        if rc:
            raise RuntimeError(f"orc_puct_rollout rc={rc}")

    def steps_hash(self, seed, first_root, step0, n_steps):
        imp = np.zeros(max(1, n_steps), dtype=np.uint32)
        n_imp = C.c_uint32()
        rc = lib().orc_puct_steps_hash(self._h, self.c_puct, seed, first_root, step0, n_steps,
                                       imp.ctypes.data_as(C.POINTER(C.c_uint32)), len(imp), C.byref(n_imp))
        if rc:
            raise RuntimeError(f"orc_puct_steps_hash rc={rc}")
        return imp[: n_imp.value].tolist()
