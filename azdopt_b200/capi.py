"""ctypes binding of the C ABI in include/azb.h (lib/libazb.so).

No fallback: if the library has not been built this module raises at import
of :func:`lib`.  Buffers are numpy arrays in host memory.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .build import lib_path

NONE = 0xFFFFFFFF
OK, ERR_INVALID, ERR_CUDA, ERR_CAPACITY, ERR_NAN, ERR_LAMBDA, ERR_UNREACHABLE, ERR_STATE = range(8)
PRIOR_MLP, PRIOR_HASH, PRIOR_INJECTED = 0, 1, 2
MLP_FP32, MLP_TC, MLP_TC3 = 0, 1, 2
MAX_TOL = 8
ASYNC_AUTO = 0xFFFFFFFF
ASYNC_SHARED = 0xFFFFFFFE  # every SM walks trees and serves the model with its last warpgroup (include/azb.h)
SELECT_REFERENCE, SELECT_PUCT = 0, 1  # azb_config.selection: next_action, or PUCT (rule in include/azb.h; no reference)

COUNTER_FIELDS = [
    "n_sel", "d_sel", "n_cur", "n_cand", "n_probe", "n_ins", "n_term", "n_hit", "n_arc", "n_pred",
    "n_cn", "d_cn", "n_reset", "n_live", "n_noop", "n_visit",
]


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("n_vertices", C.c_uint32), ("n_roots", C.c_uint32), ("device", C.c_int32),
        ("first_root", C.c_uint64), ("c_lower", C.c_float), ("c_upper", C.c_float),
        ("n_as_tol", C.c_uint32 * MAX_TOL), ("n_as_tol_len", C.c_uint32), ("n_as_tol_default", C.c_uint32),
        ("mlp_hidden", C.c_uint32 * 3), ("mlp_mode", C.c_uint32), ("prior_mode", C.c_uint32),
        ("prior_seed", C.c_uint64), ("max_steps", C.c_uint32), ("cap_nodes", C.c_uint32), ("cap_preds", C.c_uint32),
        ("cap_parents", C.c_uint32), ("max_episodes", C.c_uint32), ("n_groups", C.c_uint32), ("async_workers", C.c_uint32),
        ("selection", C.c_uint32), ("puct_c", C.c_float), ("reserved", C.c_uint32 * 3),
    ]


class Counters(C.Structure):
    _fields_ = [(f, C.c_uint64) for f in COUNTER_FIELDS]

    def as_dict(self):
        return {f: int(getattr(self, f)) for f in COUNTER_FIELDS}


class Improvement(C.Structure):
    _fields_ = [("step", C.c_uint32), ("tree", C.c_uint32), ("node", C.c_uint32), ("eval", C.c_float)]


class AzbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"azb error {code} ({msg})")
        self.code = code


_lib = None
u8p, u32p, f32p, f64p = (C.POINTER(t) for t in (C.c_uint8, C.c_uint32, C.c_float, C.c_double))

# name -> (restype, argtypes); every symbol include/azb.h declares
SIGNATURES = {
    "azb_version": (C.c_int, []),
    "azb_strerror": (C.c_char_p, [C.c_int]),
    "azb_last_error": (C.c_char_p, [C.c_void_p]),
    "azb_config_default": (C.c_int, [C.POINTER(Config), C.c_uint32, C.c_uint32]),
    "azb_create": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "azb_destroy": (C.c_int, [C.c_void_p]),
    "azb_get_config": (C.c_int, [C.c_void_p, C.POINTER(Config)]),
    "azb_generate_roots": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, u8p, u32p]),
    "azb_set_roots": (C.c_int, [C.c_void_p, u8p, u32p]),
    "azb_get_roots": (C.c_int, [C.c_void_p, u8p, u32p]),
    "azb_mlp_num_params": (C.c_size_t, [C.c_void_p]),
    "azb_mlp_init": (C.c_int, [C.c_void_p, C.c_uint64]),
    "azb_mlp_set_params": (C.c_int, [C.c_void_p, f32p]),
    "azb_mlp_get_params": (C.c_int, [C.c_void_p, f32p]),
    "azb_model_write_predictions": (C.c_int, [C.c_void_p, f32p, f32p, C.c_uint32]),
    "azb_set_priors": (C.c_int, [C.c_void_p, f32p]),
    "azb_init_trees": (C.c_int, [C.c_void_p]),
    "azb_step": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(Improvement), C.c_uint32, u32p]),
    "azb_step_enqueue": (C.c_int, [C.c_void_p, C.c_uint32]),
    "azb_step_poll": (C.c_int, [C.c_void_p, C.POINTER(Improvement), C.POINTER(C.c_int)]),
    "azb_step_timed": (C.c_int, [C.c_void_p, C.c_uint32, f32p, u32p]),
    "azb_step_profile": (C.c_int, [C.c_void_p, C.c_uint32, f32p, f32p]),
    "azb_rollout_host": (C.c_int, [C.c_void_p, f32p]),
    "azb_add_actions_host": (C.c_int, [C.c_void_p, f32p, C.POINTER(C.c_int)]),
    "azb_get_argmin": (C.c_int, [C.c_void_p, u8p, u32p, f64p, u32p, f32p]),
    "azb_get_node_state": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, u8p, u32p]),
    "azb_tree_codes": (C.c_int, [C.c_void_p, u8p, C.c_uint32, C.POINTER(C.c_uint64), f32p]),
    "azb_best_trees": (C.c_int, [C.c_void_p, C.c_uint32, u32p, f32p, C.POINTER(C.c_uint64), u32p, u32p, u8p, u32p, f64p, u32p]),
    "azb_free_tree_count": (C.c_int, [C.c_uint32, C.POINTER(C.c_uint64)]),
    "azb_free_trees": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, u8p]),
    "azb_exhaustive_best": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_double, u32p, C.POINTER(C.c_uint64),
                                      C.POINTER(C.c_uint64), u8p, f64p, u32p, f32p, f32p]),
    "azb_trees_within": (C.c_int, [C.c_void_p, C.c_double, C.c_uint32, C.c_uint64, u32p, C.POINTER(C.c_uint64),
                                   C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), u8p, f64p, u32p, f32p, f32p]),
    "azb_trees_within_proof": (C.c_int, [C.c_void_p, C.c_double, C.c_uint32, C.c_uint64, u32p, C.POINTER(C.c_uint64),
                                         C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), u8p, f64p, u32p, f32p,
                                         C.POINTER(C.c_uint64), f32p]),
    "azb_certify_keys": (C.c_int, [C.c_void_p, u8p, C.c_uint32, C.c_double, f64p, f64p, u32p, C.POINTER(C.c_int8), f32p]),
    "azb_comm_trees_within": (C.c_int, [C.c_void_p, C.c_double, C.c_uint32, C.c_uint64, u32p, C.POINTER(C.c_uint64),
                                        C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), u8p, f64p, u32p, f32p, f32p]),
    "azb_checkpoint_size": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "azb_checkpoint_save": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "azb_checkpoint_load": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.c_uint32]),
    "azb_get_walkers": (C.c_int, [C.c_void_p, u8p, u32p, u32p, u32p, u32p]),
    "azb_tree_sizes": (C.c_int, [C.c_void_p, C.c_uint32, u32p, u32p, u32p]),
    "azb_dump_tree": (C.c_int, [C.c_void_p, C.c_uint32, u32p, u32p, u32p, u32p]),
    "azb_get_counters": (C.c_int, [C.c_void_p, C.POINTER(Counters)]),
    "azb_reset_counters": (C.c_int, [C.c_void_p]),
    "azb_set_counter_mode": (C.c_int, [C.c_void_p, C.c_int]),
    "azb_get_state_vecs": (C.c_int, [C.c_void_p, f32p]),
    "azb_get_priors": (C.c_int, [C.c_void_p, f32p]),
    "azb_eval_costs": (C.c_int, [C.c_void_p, u8p, C.c_uint32, f64p, u32p, f32p, f32p]),
    "azb_eval_graph_costs": (C.c_int, [C.c_void_p, u32p, C.c_uint32, C.c_uint32, f64p, u32p, u32p, f32p]),
    "azb_eval_graph_costs64": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.c_uint32, f64p, u32p, u32p, f32p]),
    "azb_write_observations": (C.c_int, [C.c_void_p, C.c_uint32, f32p, f32p, f32p]),
    "azb_adam_config": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float]),
    "azb_model_update": (C.c_int, [C.c_void_p, f32p, f32p, f32p, C.c_uint32, f32p]),
    "azb_model_gradients": (C.c_int, [C.c_void_p, f32p, f32p, f32p, C.c_uint32, f32p, f32p]),
    "azb_update_model": (C.c_int, [C.c_void_p, C.c_uint32, f32p]),
    "azb_reset_trees": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32]),
    "azb_comm_unique_id": (C.c_int, [u8p]),
    "azb_comm_init": (C.c_int, [C.c_void_p, u8p, C.c_int, C.c_int]),
    "azb_comm_destroy": (C.c_int, [C.c_void_p]),
    "azb_comm_allreduce_bench": (C.c_int, [C.c_void_p, C.c_uint32, f32p]),
    "azb_comm_argmin": (C.c_int, [C.c_void_p, u8p, u32p, f64p, u32p, f32p, C.POINTER(C.c_int)]),
    "azb_kernel_launches": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "azb_device_bytes": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "azb_flush_l2": (C.c_int, [C.c_void_p]),
    "azb_debug_cascade_spills": (C.c_int, [C.c_void_p, u32p]),
}


def lib():
    """The loaded library; raises if it has not been built (there is no CPU fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(azdopt_b200 has no CPU fallback)")
    L = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def action_dim(n: int) -> int:
    return (n - 1) * (n - 2) // 2 - 1


def mask_words(n: int) -> int:
    return (action_dim(n) + 31) // 32


def default_config(n_vertices: int, n_roots: int, **kw) -> Config:
    cfg = Config()
    rc = lib().azb_config_default(C.byref(cfg), n_vertices, n_roots)
    if rc:
        raise AzbError(rc, lib().azb_strerror(rc).decode())
    for k, v in kw.items():
        if k == "n_as_tol":
            v = list(v)
            if len(v) > MAX_TOL:
                raise ValueError("n_as_tol table too long")
            for i in range(MAX_TOL):
                cfg.n_as_tol[i] = v[i] if i < len(v) else 0
            cfg.n_as_tol_len = len(v)
        elif k == "mlp_hidden":
            for i in range(3):
                cfg.mlp_hidden[i] = v[i]
        else:
            if not hasattr(cfg, k):
                raise TypeError(f"unknown config field {k}")
            setattr(cfg, k, v)
    return cfg


def comm_unique_id() -> bytes:
    buf = (C.c_uint8 * 128)()
    rc = lib().azb_comm_unique_id(buf)
    if rc:
        raise AzbError(rc, "azb_comm_unique_id (is libnccl.so.2 loadable?)")
    return bytes(buf)


def generate_roots(seed, first_root, count, n, k_min=5, k_max=0):
    """Synthetic roots with the example's distribution (04-c21-tree.rs:85,108-112). Host-only."""
    parents = np.zeros((count, n), dtype=np.uint8)
    masks = np.zeros((count, mask_words(n)), dtype=np.uint32)
    rc = lib().azb_generate_roots(seed, first_root, count, n, k_min, k_max, _p(parents, C.c_uint8), _p(masks, C.c_uint32))
    if rc:
        raise AzbError(rc, lib().azb_strerror(rc).decode())
    return parents, masks


def free_tree_count(n: int) -> int:
    """A000055(n): the number of free trees on n vertices, 5 <= n <= 32 (host only)."""
    out = C.c_uint64()
    rc = lib().azb_free_tree_count(n, C.byref(out))
    if rc:
        raise AzbError(rc, f"{lib().azb_strerror(rc).decode()}: n must be in 5..32, got {n}")
    return int(out.value)


class Handle:
    """One azb_handle: the device-resident state of a NablaOptimizer shard."""

    def __init__(self, cfg: Config):
        self._h = C.c_void_p()
        self._L = lib()
        rc = self._L.azb_create(C.byref(cfg), C.byref(self._h))
        if rc:
            msg = self._L.azb_last_error(self._h).decode() if self._h else ""
            if self._h:
                self._L.azb_destroy(self._h)
                self._h = C.c_void_p()
            raise AzbError(rc, f"{self._L.azb_strerror(rc).decode()}: {msg}")
        out = Config()
        self._L.azb_get_config(self._h, C.byref(out))
        self.cfg = out
        self.n = int(out.n_vertices)
        self.b = int(out.n_roots)
        self.a = action_dim(self.n)
        self.w = mask_words(self.n)
        self.s = 2 * self.a

    def close(self):
        if getattr(self, "_h", None):
            self._L.azb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _ck(self, rc):
        if rc:
            raise AzbError(rc, f"{self._L.azb_strerror(rc).decode()}: {self._L.azb_last_error(self._h).decode()}")

    # ---- roots / model ----
    def set_roots(self, parents, permitted):
        p = np.ascontiguousarray(parents, dtype=np.uint8)
        m = np.ascontiguousarray(permitted, dtype=np.uint32)
        if p.shape != (self.b, self.n) or m.shape != (self.b, self.w):
            raise ValueError("root array shapes")
        self._ck(self._L.azb_set_roots(self._h, _p(p, C.c_uint8), _p(m, C.c_uint32)))

    def get_roots(self):
        p = np.zeros((self.b, self.n), dtype=np.uint8)
        m = np.zeros((self.b, self.w), dtype=np.uint32)
        self._ck(self._L.azb_get_roots(self._h, _p(p, C.c_uint8), _p(m, C.c_uint32)))
        return p, m

    def mlp_num_params(self) -> int:
        return int(self._L.azb_mlp_num_params(self._h))

    def mlp_init(self, seed: int):
        self._ck(self._L.azb_mlp_init(self._h, seed))

    def mlp_set_params(self, params):
        p = np.ascontiguousarray(params, dtype=np.float32)
        if p.size != self.mlp_num_params():
            raise ValueError("parameter count")
        self._ck(self._L.azb_mlp_set_params(self._h, _p(p, C.c_float)))

    def mlp_get_params(self):
        p = np.zeros(self.mlp_num_params(), dtype=np.float32)
        self._ck(self._L.azb_mlp_get_params(self._h, _p(p, C.c_float)))
        return p

    def model_write_predictions(self, states, out=None):
        x = np.ascontiguousarray(states, dtype=np.float32)
        rows = x.shape[0]
        if x.shape != (rows, self.s):
            raise ValueError("state rows")
        y = out if out is not None else np.empty((rows, self.a), dtype=np.float32)
        self._ck(self._L.azb_model_write_predictions(self._h, _p(x, C.c_float), _p(y, C.c_float), rows))
        return y

    # ---- search ----
    def set_priors(self, priors):
        pr = np.ascontiguousarray(priors, dtype=np.float32)
        if pr.shape != (self.b, self.a):
            raise ValueError("prior rows")
        self._ck(self._L.azb_set_priors(self._h, _p(pr, C.c_float)))

    def init_trees(self):
        self._ck(self._L.azb_init_trees(self._h))

    def step(self, n_steps=1, cap=64):
        imp = (Improvement * max(cap, 1))()
        n = C.c_uint32()
        self._ck(self._L.azb_step(self._h, n_steps, imp, cap, C.byref(n)))
        k = min(int(n.value), cap)
        return int(n.value), [(imp[i].step, imp[i].tree, imp[i].node, np.float32(imp[i].eval)) for i in range(k)]

    def step_enqueue(self, n_steps):
        self._ck(self._L.azb_step_enqueue(self._h, n_steps))

    def step_poll(self):
        """Result of the next enqueued step (azb_step_poll): (improved, (step, tree, node, eval))."""
        imp = Improvement()
        flag = C.c_int()
        self._ck(self._L.azb_step_poll(self._h, C.byref(imp), C.byref(flag)))
        return bool(flag.value), (imp.step, imp.tree, imp.node, np.float32(imp.eval))

    def step_timed(self, n_steps):
        ms = C.c_float()
        n = C.c_uint32()
        self._ck(self._L.azb_step_timed(self._h, n_steps, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def step_profile(self, n_steps):
        a, b = C.c_float(), C.c_float()
        self._ck(self._L.azb_step_profile(self._h, n_steps, C.byref(a), C.byref(b)))
        return float(a.value), float(b.value)

    def rollout_host(self, state_vecs):
        if state_vecs.dtype != np.float32 or state_vecs.shape != (self.b, self.s) or not state_vecs.flags.c_contiguous:
            raise ValueError("state_vecs buffer")
        self._ck(self._L.azb_rollout_host(self._h, _p(state_vecs, C.c_float)))

    def add_actions_host(self, h_theta) -> bool:
        pr = np.ascontiguousarray(h_theta, dtype=np.float32)
        if pr.shape != (self.b, self.a):
            raise ValueError("h_theta rows")
        imp = C.c_int()
        self._ck(self._L.azb_add_actions_host(self._h, _p(pr, C.c_float), C.byref(imp)))
        return bool(imp.value)

    # ---- results ----
    def argmin(self):
        p = np.zeros(self.n, dtype=np.uint8)
        m = np.zeros(self.w, dtype=np.uint32)
        lam, mu, ev = C.c_double(), C.c_uint32(), C.c_float()
        self._ck(self._L.azb_get_argmin(self._h, _p(p, C.c_uint8), _p(m, C.c_uint32), C.byref(lam), C.byref(mu), C.byref(ev)))
        return dict(parents=p, permitted=m, lambda1=lam.value, mu=mu.value, eval=np.float32(ev.value))

    # ---- checkpoints (format in include/azb.h; azdopt_b200/checkpoint.py reads it) ----
    def checkpoint_size(self) -> int:
        n = C.c_uint64()
        self._ck(self._L.azb_checkpoint_size(self._h, C.byref(n)))
        return int(n.value)

    def checkpoint_save(self, out=None) -> np.ndarray:
        """The handle's search and training state as a uint8 array (written into ``out`` when given: a writable
        uint8 array or np.memmap of at least checkpoint_size() bytes; the returned array is its used prefix)."""
        size = self.checkpoint_size()
        buf = np.empty(size, dtype=np.uint8) if out is None else out
        if buf.dtype != np.uint8 or buf.ndim != 1 or not buf.flags.c_contiguous or not buf.flags.writeable:
            raise ValueError("out must be a writable contiguous uint8 array")
        written = C.c_uint64()
        self._ck(self._L.azb_checkpoint_save(self._h, buf.ctypes.data_as(C.c_void_p), buf.size, C.byref(written)))
        return buf[:written.value]

    def checkpoint_load(self, blobs):
        """Rebuild the state from one blob or a list of blobs (bytes, uint8 numpy arrays or np.memmap) whose root
        ranges cover this handle's exactly once."""
        if isinstance(blobs, (bytes, bytearray, memoryview, np.ndarray)):
            blobs = [blobs]
        arrs = [np.frombuffer(b, dtype=np.uint8) if not isinstance(b, np.ndarray) else np.ascontiguousarray(b).view(np.uint8).reshape(-1)
                for b in blobs]
        ptrs = (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
        sizes = (C.c_uint64 * len(arrs))(*[a.size for a in arrs])
        self._ck(self._L.azb_checkpoint_load(self._h, ptrs, sizes, len(arrs)))

    def walkers(self):
        p = np.zeros((self.b, self.n), dtype=np.uint8)
        m = np.zeros((self.b, self.w), dtype=np.uint32)
        k = np.zeros((self.b, self.w), dtype=np.uint32)
        pos = np.zeros(self.b, dtype=np.uint32)
        ln = np.zeros(self.b, dtype=np.uint32)
        self._ck(self._L.azb_get_walkers(self._h, _p(p, C.c_uint8), _p(m, C.c_uint32), _p(k, C.c_uint32),
                                         _p(pos, C.c_uint32), _p(ln, C.c_uint32)))
        return dict(parents=p, permitted=m, path=k, pos=pos, path_len=ln)

    def tree_sizes(self, tree):
        a, b, c = C.c_uint32(), C.c_uint32(), C.c_uint32()
        self._ck(self._L.azb_tree_sizes(self._h, tree, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def dump_tree(self, tree):
        nn, na, npred = self.tree_sizes(tree)
        nodes = np.zeros((nn, 6), dtype=np.uint32)
        keys = np.zeros((nn, self.w), dtype=np.uint32)
        preds = np.zeros((max(npred, 1), 3), dtype=np.uint32)
        arcs = np.zeros((max(na, 1), 3), dtype=np.uint32)
        self._ck(self._L.azb_dump_tree(self._h, tree, _p(nodes, C.c_uint32), _p(keys, C.c_uint32), _p(preds, C.c_uint32),
                                       _p(arcs, C.c_uint32)))
        return dict(nodes=nodes, keys=keys, preds=preds[:npred], arcs=arcs[:na])

    def counters(self):
        c = Counters()
        self._ck(self._L.azb_get_counters(self._h, C.byref(c)))
        return c.as_dict()

    def set_counter_mode(self, full: bool):
        self._ck(self._L.azb_set_counter_mode(self._h, 1 if full else 0))

    def reset_counters(self):
        self._ck(self._L.azb_reset_counters(self._h))

    def state_vecs(self):
        v = np.zeros((self.b, self.s), dtype=np.float32)
        self._ck(self._L.azb_get_state_vecs(self._h, _p(v, C.c_float)))
        return v

    def priors(self):
        v = np.zeros((self.b, self.a), dtype=np.float32)
        self._ck(self._L.azb_get_priors(self._h, _p(v, C.c_float)))
        return v

    def eval_costs(self, parents):
        p = np.ascontiguousarray(parents, dtype=np.uint8)
        m = p.shape[0]
        lam = np.zeros(m, dtype=np.float64)
        mu = np.zeros(m, dtype=np.uint32)
        c = np.zeros(m, dtype=np.float32)
        ms = C.c_float()
        self._ck(self._L.azb_eval_costs(self._h, _p(p, C.c_uint8), m, _p(lam, C.c_double), _p(mu, C.c_uint32),
                                        _p(c, C.c_float), C.byref(ms)))
        return lam, mu, c, float(ms.value)

    def eval_graph_costs(self, nbr):
        """(lambda_1 f64[M], mu u32[M], kinds u32[M, ceil(n(n-1)/32)], kernel ms) for M connected graphs given as
        neighbourhood masks u32[M, n] (ConnectedBitsetGraph<N, B32>::conjecture_2_1_cost / action_kinds)."""
        g = np.ascontiguousarray(nbr, dtype=np.uint32)
        m, n = g.shape
        lam = np.zeros(m, dtype=np.float64)
        mu = np.zeros(m, dtype=np.uint32)
        kinds = np.zeros((m, (n * (n - 1) + 31) // 32), dtype=np.uint32)
        ms = C.c_float()
        self._ck(self._L.azb_eval_graph_costs(self._h, _p(g, C.c_uint32), m, n, _p(lam, C.c_double), _p(mu, C.c_uint32),
                                              _p(kinds, C.c_uint32), C.byref(ms)))
        return lam, mu, kinds, float(ms.value)

    def eval_graph_costs64(self, nbr):
        """eval_graph_costs for neighbourhood masks u64[M, n], 2 <= n <= 64 (ConnectedBitsetGraph<N, B64>)."""
        g = np.ascontiguousarray(nbr, dtype=np.uint64)
        m, n = g.shape
        lam = np.zeros(m, dtype=np.float64)
        mu = np.zeros(m, dtype=np.uint32)
        kinds = np.zeros((m, (n * (n - 1) + 31) // 32), dtype=np.uint32)
        ms = C.c_float()
        self._ck(self._L.azb_eval_graph_costs64(self._h, _p(g, C.c_uint64), m, n, _p(lam, C.c_double), _p(mu, C.c_uint32),
                                                _p(kinds, C.c_uint32), C.byref(ms)))
        return lam, mu, kinds, float(ms.value)

    def write_observations(self, n_obs_tol):
        v = np.zeros((self.b, self.s), dtype=np.float32)
        obs = np.zeros((self.b, self.a), dtype=np.float32)
        w = np.zeros((self.b, self.a), dtype=np.float32)
        self._ck(self._L.azb_write_observations(self._h, n_obs_tol, _p(v, C.c_float), _p(obs, C.c_float), _p(w, C.c_float)))
        return v, obs, w

    # ---- epoch boundary: training step and communicator ----
    def adam_config(self, lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, l2=1e-6):
        self._ck(self._L.azb_adam_config(self._h, lr, beta1, beta2, eps, l2))

    def _train_args(self, states, observations, weights):
        x = np.ascontiguousarray(states, dtype=np.float32).reshape(-1, self.s)
        o = np.ascontiguousarray(observations, dtype=np.float32).reshape(-1, self.a)
        w = np.ascontiguousarray(weights, dtype=np.float32).reshape(-1, self.a)
        assert x.shape[0] == o.shape[0] == w.shape[0]
        return x, o, w

    def model_update(self, states, observations, weights) -> float:
        x, o, w = self._train_args(states, observations, weights)
        loss = C.c_float()
        self._ck(self._L.azb_model_update(self._h, _p(x, C.c_float), _p(o, C.c_float), _p(w, C.c_float), x.shape[0],
                                          C.byref(loss)))
        return float(loss.value)

    def model_gradients(self, states, observations, weights):
        x, o, w = self._train_args(states, observations, weights)
        loss = C.c_float()
        g = np.zeros(self.mlp_num_params(), dtype=np.float32)
        self._ck(self._L.azb_model_gradients(self._h, _p(x, C.c_float), _p(o, C.c_float), _p(w, C.c_float), x.shape[0],
                                             C.byref(loss), _p(g, C.c_float)))
        return float(loss.value), g

    def update_model(self, n_obs_tol: int) -> float:
        loss = C.c_float()
        self._ck(self._L.azb_update_model(self._h, n_obs_tol, C.byref(loss)))
        return float(loss.value)

    def reset_trees(self, seed: int, k_min: int = 0, k_max: int = 0):
        self._ck(self._L.azb_reset_trees(self._h, seed, k_min, k_max))

    def comm_init(self, unique_id: bytes, rank: int, world: int):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        self._ck(self._L.azb_comm_init(self._h, buf, rank, world))

    def comm_argmin(self):
        p = np.zeros(self.n, dtype=np.uint8)
        m = np.zeros(self.w, dtype=np.uint32)
        lam, mu, ev, owner = C.c_double(), C.c_uint32(), C.c_float(), C.c_int()
        self._ck(self._L.azb_comm_argmin(self._h, _p(p, C.c_uint8), _p(m, C.c_uint32), C.byref(lam), C.byref(mu),
                                         C.byref(ev), C.byref(owner)))
        return p, m, float(lam.value), int(mu.value), float(ev.value), int(owner.value)

    def kernel_launches(self) -> int:
        n = C.c_uint64()
        self._ck(self._L.azb_kernel_launches(self._h, C.byref(n)))
        return int(n.value)

    def node_state(self, tree: int, node: int):
        """(parents, permitted mask) of a node: the root with the node's action set replayed; does not wait for steps"""
        parents = np.zeros(self.n, dtype=np.uint8)
        permitted = np.zeros(self.w, dtype=np.uint32)
        self._ck(self._L.azb_get_node_state(self._h, tree, node, _p(parents, C.c_uint8), _p(permitted, C.c_uint32)))
        return parents, permitted

    def tree_codes(self, parents):
        """Canonical codes u64[M, 2] of M trees given as parent arrays u8[M, N] (include/azb.h): equal rows <=> isomorphic."""
        p = np.ascontiguousarray(parents, dtype=np.uint8)
        m = p.shape[0]
        if p.shape != (m, self.n):
            raise ValueError("parent rows")
        codes = np.zeros((m, 2), dtype=np.uint64)
        self._ck(self._L.azb_tree_codes(self._h, _p(p, C.c_uint8), m, _p(codes, C.c_uint64), None))
        return codes

    def best_trees(self, k: int):
        """The k best isomorphism classes among all nodes of all trees (azb_best_trees), ascending by (eval, code):
        dict of arrays eval f32, code u64[., 2], tree, node, parents u8[., N], permitted u32[., W], lambda1 f64, mu."""
        kk = max(int(k), 1)
        out = dict(eval=np.zeros(kk, dtype=np.float32), code=np.zeros((kk, 2), dtype=np.uint64),
                   tree=np.zeros(kk, dtype=np.uint32), node=np.zeros(kk, dtype=np.uint32),
                   parents=np.zeros((kk, self.n), dtype=np.uint8), permitted=np.zeros((kk, self.w), dtype=np.uint32),
                   lambda1=np.zeros(kk, dtype=np.float64), mu=np.zeros(kk, dtype=np.uint32))
        n = C.c_uint32()
        self._ck(self._L.azb_best_trees(self._h, k, C.byref(n), _p(out["eval"], C.c_float), _p(out["code"], C.c_uint64),
                                        _p(out["tree"], C.c_uint32), _p(out["node"], C.c_uint32),
                                        _p(out["parents"], C.c_uint8), _p(out["permitted"], C.c_uint32),
                                        _p(out["lambda1"], C.c_double), _p(out["mu"], C.c_uint32)))
        return {name: a[:n.value] for name, a in out.items()}

    def free_trees(self, start: int, m: int):
        """Parent arrays u8[m, N] of the free trees with indices [start, start + m) of the enumeration in include/azb.h."""
        out = np.zeros((max(int(m), 1), self.n), dtype=np.uint8)
        self._ck(self._L.azb_free_trees(self._h, start, m, _p(out, C.c_uint8)))
        return out[:m]

    def exhaustive_best(self, start: int = 0, count=None, k: int = 100, bound=None):
        """The exact k best free trees of indices [start, start + count) (default: to the end) by key = mu + lambda1, ties
        by index (azb_exhaustive_best): dict of arrays index u64, parents u8[., N], lambda1 f64, mu u32, eval f32, plus
        n_below (trees with key < bound; default sqrt(N - 1) + 1, the star's key) and ms (device time)."""
        if count is None:
            count = free_tree_count(self.n) - start if self.n <= 32 else 1  # N > 32: the library refuses the handle
        if bound is None:
            bound = float(np.sqrt(self.n - 1)) + 1.0
        kk = max(min(int(k), int(count)), 1)
        out = dict(index=np.zeros(kk, dtype=np.uint64), parents=np.zeros((kk, self.n), dtype=np.uint8),
                   lambda1=np.zeros(kk, dtype=np.float64), mu=np.zeros(kk, dtype=np.uint32), eval=np.zeros(kk, dtype=np.float32))
        n, below, ms = C.c_uint32(), C.c_uint64(), C.c_float()
        self._ck(self._L.azb_exhaustive_best(self._h, start, count, k, bound, C.byref(n), C.byref(below),
                                             _p(out["index"], C.c_uint64), _p(out["parents"], C.c_uint8),
                                             _p(out["lambda1"], C.c_double), _p(out["mu"], C.c_uint32),
                                             _p(out["eval"], C.c_float), C.byref(ms)))
        res = {name: a[:n.value] for name, a in out.items()}
        res.update(n_below=int(below.value), ms=float(ms.value))
        return res

    def trees_within(self, bound=None, k: int = 100, max_level: int = 0, prove: bool = False):
        """Every isomorphism class on N vertices with key = mu + lambda1 <= bound (azb_trees_within; default: the star's
        key), the first k ascending by (key, code): dict of arrays code u64[., 2], parents u8[., N] (canonical labelling),
        lambda1 f64, mu u32, eval f32, plus n_within, n_below (key < bound) and ms (device time).  max_level caps the
        classes of any level (0: what fits in device memory); beyond it AzbError with ERR_CAPACITY.  prove=True runs
        azb_trees_within_proof (default bound: sqrt(N - 1) + 1 exactly) and adds proof = dict(below, equal, above, open,
        unproven_pruned) (include/azb.h)."""
        if prove:
            return self._trees_within(self._L.azb_trees_within_proof, bound, k, max_level, prove=True)
        return self._trees_within(self._L.azb_trees_within, bound, k, max_level)

    def comm_trees_within(self, bound=None, k: int = 100, max_level: int = 0):
        """trees_within split over the ranks of the attached communicator (azb_comm_trees_within): collective, every rank
        calls it with the same arguments and gets the same dict, bit for bit what trees_within gives on one handle."""
        return self._trees_within(self._L.azb_comm_trees_within, bound, k, max_level)

    def _trees_within(self, fn, bound, k, max_level, prove=False):
        kk = max(int(k), 1)
        out = dict(code=np.zeros((kk, 2), dtype=np.uint64), parents=np.zeros((kk, self.n), dtype=np.uint8),
                   lambda1=np.zeros(kk, dtype=np.float64), mu=np.zeros(kk, dtype=np.uint32), eval=np.zeros(kk, dtype=np.float32))
        n, within, below, ms = C.c_uint32(), C.c_uint64(), C.c_uint64(), C.c_float()
        proof = np.zeros(5, dtype=np.uint64)
        self._ck(fn(self._h, -1.0 if bound is None else float(bound), k, max_level, C.byref(n), C.byref(within), C.byref(below),
                    _p(out["code"], C.c_uint64), _p(out["parents"], C.c_uint8), _p(out["lambda1"], C.c_double),
                    _p(out["mu"], C.c_uint32), _p(out["eval"], C.c_float), *([_p(proof, C.c_uint64)] if prove else []),
                    C.byref(ms)))
        res = {name: a[:n.value] for name, a in out.items()}
        res.update(n_within=int(within.value), n_below=int(below.value), ms=float(ms.value))
        if prove:
            res["proof"] = dict(zip(("below", "equal", "above", "open", "unproven_pruned"), (int(x) for x in proof)))
        return res

    def certify_keys(self, parents, bound=None):
        """Certificates of the keys mu + lambda1 of trees u8[M, N] against bound (azb_certify_keys; default: sqrt(N - 1) + 1
        exactly): dict lambda1_lo, lambda1_hi (f64, lambda1_lo < lambda1 < lambda1_hi, NaN where not enclosed), mu (u32,
        greedy matching), verdict (i8: -1 key < bound, 0 key == bound, +1 key > bound, all proven; 2 open), ms."""
        p = np.ascontiguousarray(parents, dtype=np.uint8)
        m = p.shape[0]
        if p.shape != (m, self.n):
            raise ValueError("parent rows")
        out = dict(lambda1_lo=np.zeros(m, dtype=np.float64), lambda1_hi=np.zeros(m, dtype=np.float64),
                   mu=np.zeros(m, dtype=np.uint32), verdict=np.zeros(m, dtype=np.int8))
        ms = C.c_float()
        self._ck(self._L.azb_certify_keys(self._h, _p(p, C.c_uint8), m, -1.0 if bound is None else float(bound),
                                          _p(out["lambda1_lo"], C.c_double), _p(out["lambda1_hi"], C.c_double),
                                          _p(out["mu"], C.c_uint32), _p(out["verdict"], C.c_int8), C.byref(ms)))
        out["ms"] = float(ms.value)
        return out

    def comm_allreduce_bench(self, reps: int = 20) -> float:
        ms = C.c_float()
        self._ck(self._L.azb_comm_allreduce_bench(self._h, reps, C.byref(ms)))
        return float(ms.value)

    def cascade_spills(self) -> int:
        n = C.c_uint32()
        self._ck(self._L.azb_debug_cascade_spills(self._h, C.byref(n)))
        return int(n.value)

    def device_bytes(self) -> int:
        n = C.c_uint64()
        self._ck(self._L.azb_device_bytes(self._h, C.byref(n)))
        return int(n.value)

    def flush_l2(self):
        self._ck(self._L.azb_flush_l2(self._h))
