"""Host-side mirror of the reference's optimizer surface for the c21 path, on top of the C ABI.

Names follow az-discrete-opt: ``NablaOptimizer`` (nabla/optimizer/mod.rs:7-22) with ``par_new``,
``par_roll_out_episodes``, ``argmin_data``, ``par_update_model`` (observation pass) and ``par_reset_trees``;
``NablaStateActionSpace`` is represented by :class:`ROTModifyParentsOnce` (graph-state/src/rooted_tree/space.rs:37-125)
whose four closures travel as data; ``NablaModel`` (nabla/model/mod.rs:4-8) by :class:`ActionModel` (the built-in
device MLP), :class:`TrivialModel`, or any object with ``write_predictions(states, predictions)`` on host arrays.
"""
from __future__ import annotations

import dataclasses
import os
from typing import Callable, Optional, Sequence

import numpy as np

from . import capi


@dataclasses.dataclass
class ROTModifyParentsOnce:
    """The c21 space: rooted ordered trees on ``n`` vertices, each child re-parented at most once.
    cost = lambda_1 + matching number, evaluate = squish (examples/04-c21-tree.rs:58-105)."""

    n: int = 19
    c_lower: float = 2.0
    c_upper: float = 0.0  # 0 = ceil(sqrt(n-1)) + (n+1)//2, the example's C_UPPER_BOUND

    @property
    def ACTION_DIM(self) -> int:  # rooted_tree/space.rs:48
        return capi.action_dim(self.n)

    @property
    def STATE_DIM(self) -> int:  # rooted_tree/space.rs:46
        return 2 * capi.action_dim(self.n)

    @staticmethod
    def g_theta_star_sa(c_s, h_theta_sa):  # 04-c21-tree.rs:103 (hard-wired in the kernels)
        return np.float32(c_s) - np.float32(h_theta_sa)

    @staticmethod
    def h_sa(c_s, c_as_star):  # 04-c21-tree.rs:104
        return np.float32(c_as_star)


@dataclasses.dataclass
class ActionModel:
    """The example's MLP (04-c21-tree.rs:42-52) evaluated on the device inside the fused step."""

    seed: int = 0
    hidden: Sequence[int] = (512, 1024, 512)
    arithmetic: str = "fp32"  # "fp32" (what cuBLAS sgemm gives the reference) or "tc" (tcgen05 tensor cores)
    params: Optional[np.ndarray] = None  # dfdx order: weight[out][in], bias[out] per layer


class TrivialModel:
    """nabla/model/mod.rs:10-23: leaves the prediction buffer untouched (zeros after the optimizer's fill)."""

    def write_predictions(self, states: np.ndarray, predictions: np.ndarray) -> None:
        return None

    def update_model(self, states: np.ndarray, observations: np.ndarray, action_weights: np.ndarray) -> float:
        return 0.0


@dataclasses.dataclass
class ArgminData:  # log.rs:1-11
    parents: np.ndarray
    permitted: np.ndarray
    lambda_1: float
    mu: int
    eval: np.float32


@dataclasses.dataclass
class BestTree:
    """One isomorphism class of azb_best_trees: its value, its representative node's state and cost, the canonical
    code (two 64-bit words, include/azb.h) and where the representative lives (global root index, node)."""
    eval: np.float32
    lambda_1: float
    mu: int
    parents: np.ndarray
    permitted: np.ndarray
    code: tuple
    root: int
    node: int


class BestTrees:
    """The k best isomorphism classes over many best_trees lists (epochs, shards), ascending by (eval, code).  A class
    seen again keeps its existing entry unless the new one has a lower eval, so lists added in epoch or rank order keep
    the earliest representative.  Trimming to k after every merge is exact: a class in the top k of the union is in the
    top k of the list that holds its minimum, because every class ahead of it there is ahead of it in the union."""

    def __init__(self, k: int):
        if k < 1:
            raise ValueError("k >= 1")
        self.k = k
        self._by_code = {}

    def add(self, trees) -> "BestTrees":
        for t in trees:
            cur = self._by_code.get(t.code)
            if cur is None or np.float32(t.eval) < np.float32(cur.eval):
                self._by_code[t.code] = t
        keep = self.result()
        self._by_code = {t.code: t for t in keep}
        return self

    def result(self) -> list:
        return sorted(self._by_code.values(), key=lambda t: (np.float32(t.eval), t.code))[:self.k]

    def state(self) -> dict:
        """The accumulator as a dict of numpy arrays (np.savez can store it beside a checkpoint blob)."""
        r = self.result()
        n = r[0].parents.size if r else 0
        w = r[0].permitted.size if r else 0
        return dict(k=np.int64(self.k), eval=np.array([t.eval for t in r], dtype=np.float32),
                    lambda_1=np.array([t.lambda_1 for t in r], dtype=np.float64), mu=np.array([t.mu for t in r], dtype=np.uint32),
                    parents=np.array([t.parents for t in r], dtype=np.uint8).reshape(len(r), n),
                    permitted=np.array([t.permitted for t in r], dtype=np.uint32).reshape(len(r), w),
                    code=np.array([t.code for t in r], dtype=np.uint64).reshape(len(r), 2),
                    root=np.array([t.root for t in r], dtype=np.uint64), node=np.array([t.node for t in r], dtype=np.uint32))

    @classmethod
    def from_state(cls, st) -> "BestTrees":
        """The accumulator state() described (a dict or an np.load result)."""
        acc = cls(int(st["k"]))
        acc.add(BestTree(np.float32(st["eval"][i]), float(st["lambda_1"][i]), int(st["mu"][i]), np.array(st["parents"][i]),
                         np.array(st["permitted"][i]), (int(st["code"][i][0]), int(st["code"][i][1])), int(st["root"][i]),
                         int(st["node"][i])) for i in range(len(st["eval"])))
        return acc


class NablaOptimizer:
    def __init__(self):
        raise TypeError("use NablaOptimizer.par_new")

    @classmethod
    def par_new(cls, space: ROTModifyParentsOnce, init_states, model, batch: int, *, n_as_tol=(200, 50, 50),
                n_as_tol_default=25, device: int = 0, first_root: int = 0, max_steps: int = 800,
                async_workers: Optional[int] = None, selection: int = capi.SELECT_REFERENCE,
                puct_c: float = 1.0) -> "NablaOptimizer":
        """optimizer/mod.rs:39-118.  ``init_states`` is either ``(parents[B,N] u8, permitted[B,W] u32)`` or a callable
        ``i -> (parents[N], iterable of permitted action ids)`` (the reference's closure draws from thread_rng).
        ``selection=capi.SELECT_PUCT`` replaces the reference's next_action with PUCT at constant ``puct_c``
        (include/azb.h; a rule of this library with no reference to check it against)."""
        self = object.__new__(cls)
        self.space, self.model, self.batch = space, model, batch
        self._tol = (tuple(n_as_tol), n_as_tol_default)
        if isinstance(model, ActionModel):
            prior, mlp = capi.PRIOR_MLP, (capi.MLP_TC if model.arithmetic == "tc" else capi.MLP_FP32)
            hidden = tuple(model.hidden)
        else:
            prior, mlp, hidden = capi.PRIOR_INJECTED, capi.MLP_FP32, (512, 1024, 512)
        if async_workers is None:
            # the asynchronous search kernel (same results) wherever it applies; the library picks the model SMs
            async_workers = capi.ASYNC_AUTO
        cfg = capi.default_config(space.n, batch, device=device, first_root=first_root, c_lower=space.c_lower,
                                  c_upper=space.c_upper, n_as_tol=n_as_tol, n_as_tol_default=n_as_tol_default,
                                  prior_mode=prior, mlp_mode=mlp, mlp_hidden=hidden, max_steps=max_steps,
                                  async_workers=async_workers, selection=selection, puct_c=puct_c)
        self.h = capi.Handle(cfg)
        if isinstance(model, ActionModel):
            if model.params is not None:
                self.h.mlp_set_params(model.params)
            else:
                self.h.mlp_init(model.seed)
        self._host_vecs = np.zeros((batch, space.STATE_DIM), dtype=np.float32)
        self._host_h = np.zeros((batch, space.ACTION_DIM), dtype=np.float32)
        self._seed_roots(init_states)
        return self

    def _seed_roots(self, init_states):
        n, w = self.space.n, capi.mask_words(self.space.n)
        if callable(init_states):
            parents = np.zeros((self.batch, n), dtype=np.uint8)
            masks = np.zeros((self.batch, w), dtype=np.uint32)
            for i in range(self.batch):
                p, acts = init_states(i)
                parents[i] = p
                for a in acts:
                    masks[i, a >> 5] |= np.uint32(1 << (a & 31))
        else:
            parents, masks = init_states
        self.h.set_roots(parents, masks)
        if not isinstance(self.model, ActionModel):
            # one model call on the root vectors (optimizer/mod.rs:65-72)
            from . import spacefn

            for i in range(self.batch):
                self._host_vecs[i] = spacefn.write_vec(n, parents[i], masks[i])
            self._host_h.fill(0.0)
            self.model.write_predictions(self._host_vecs, self._host_h)
            self.h.set_priors(self._host_h)
        self.h.init_trees()

    def _check_tol(self, n_as_tol: Optional[Callable[[int], int]]):
        if n_as_tol is None:
            return
        table, default = self._tol
        for d in range(self.space.n):
            want = table[d] if d < len(table) else default
            if int(n_as_tol(d)) != want:
                raise ValueError("n_as_tol differs from the table this optimizer was built with (closures cannot cross "
                                 "the C ABI; pass n_as_tol= to par_new)")

    # optimizer/mod.rs:121-191
    def par_roll_out_episodes(self, n_as_tol: Optional[Callable[[int], int]] = None) -> Optional[ArgminData]:
        """One batched step.  Returns the new ArgminData if the argmin improved (ArgminImprovement::Improved)."""
        self._check_tol(n_as_tol)
        if isinstance(self.model, ActionModel):
            n_imp, _ = self.h.step(1)
            improved = n_imp > 0
        else:
            self.h.rollout_host(self._host_vecs)
            self.model.write_predictions(self._host_vecs, self._host_h)
            improved = self.h.add_actions_host(self._host_h)
        return self.argmin_data() if improved else None

    def roll_out(self, n_steps: int):
        """n_steps fused on the device (ActionModel only): list of (step, tree, node, eval) improvements."""
        if not isinstance(self.model, ActionModel):
            raise TypeError("the fused loop needs the device model")
        return self.h.step(n_steps, cap=max(64, n_steps))[1]

    def roll_out_ahead(self, n_steps: int):
        """The per-step loop of the example (04-c21-tree.rs:140-150: one par_roll_out_episodes per step, log when it
        improved) with the trees running ahead of the caller: yields (step, improved, (step, tree, node, eval)) for each
        of the n_steps as soon as every tree has finished that step (azb_step_enqueue + azb_step_poll), then completes
        the batch, so argmin_data() afterwards is what n_steps calls of par_roll_out_episodes would have left."""
        if not isinstance(self.model, ActionModel):
            raise TypeError("the fused loop needs the device model")
        self.h.step_enqueue(n_steps)
        for _ in range(n_steps):
            improved, rec = self.h.step_poll()
            yield rec[0], improved, rec
        self.h.step(0)

    # ---- checkpoints (azb_checkpoint_save / _load; format in include/azb.h)
    def save(self, path: str) -> int:
        """Write the search and training state to ``path`` (through a temporary file and os.replace, so the file is
        either the old or the new checkpoint); returns its size.  ActionModel only: a host model keeps its own state."""
        if not isinstance(self.model, ActionModel):
            raise TypeError("checkpoints hold the device model's state; a host model saves its own")
        blob = self.h.checkpoint_save()
        tmp = f"{path}.tmp{os.getpid()}"
        with open(tmp, "wb") as f:
            f.write(memoryview(blob))
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)
        return int(blob.size)

    @classmethod
    def resume(cls, paths, space: ROTModifyParentsOnce, model: ActionModel, batch: int, *, first_root: int = 0,
               device: int = 0, max_steps: int = 800, async_workers: Optional[int] = None) -> "NablaOptimizer":
        """A new optimizer over the global roots [first_root, first_root + batch) continuing from checkpoint files
        (one path or several, e.g. every rank's file of a run with another number of shards): exactly where the saved
        run stopped.  The search settings (n_as_tol, selection, model widths) come from the checkpoint; a different
        space or model arithmetic is refused by the load."""
        from . import checkpoint

        paths = [paths] if isinstance(paths, (str, os.PathLike)) else list(paths)
        blobs = [np.memmap(p, dtype=np.uint8, mode="r") for p in paths]
        hdr = checkpoint.read_header(blobs[0])
        self = object.__new__(cls)
        self.space, self.model, self.batch = space, model, batch
        self._tol = (tuple(hdr.n_as_tol), hdr.n_as_tol_default)
        mlp = capi.MLP_TC if model.arithmetic == "tc" else capi.MLP_FP32
        cfg = capi.default_config(space.n, batch, device=device, first_root=first_root, c_lower=space.c_lower,
                                  c_upper=space.c_upper, n_as_tol=hdr.n_as_tol, n_as_tol_default=hdr.n_as_tol_default,
                                  prior_mode=capi.PRIOR_MLP, mlp_mode=mlp, mlp_hidden=hdr.mlp_hidden, max_steps=max_steps,
                                  async_workers=capi.ASYNC_AUTO if async_workers is None else async_workers,
                                  selection=hdr.selection, puct_c=hdr.puct_c)
        self.h = capi.Handle(cfg)
        self._host_vecs = self._host_h = None
        self.h.checkpoint_load(blobs)
        return self

    def argmin_data(self) -> ArgminData:  # optimizer/mod.rs:361-363
        a = self.h.argmin()
        return ArgminData(a["parents"], a["permitted"], a["lambda1"], a["mu"], a["eval"])

    def best_trees(self, k: int) -> list:
        """The k best isomorphism classes among every node the search has evaluated since the last reset
        (azb_best_trees), as BestTree records ascending by (eval, code).  Call it before par_reset_trees, which
        discards the trees; a BestTrees accumulator merges the lists of several epochs."""
        r = self.h.best_trees(k)
        first = int(self.h.cfg.first_root)
        return [BestTree(r["eval"][i], float(r["lambda1"][i]), int(r["mu"][i]), r["parents"][i].copy(),
                         r["permitted"][i].copy(), (int(r["code"][i, 0]), int(r["code"][i, 1])), first + int(r["tree"][i]),
                         int(r["node"][i])) for i in range(len(r["eval"]))]

    def par_update_model_observations(self, n_obs_tol: int):
        """The data par_update_model hands to NablaModel::update_model (optimizer/mod.rs:253-280):
        (root state vectors, observations, action weights)."""
        return self.h.write_observations(n_obs_tol)

    def par_update_model(self, n_obs_tol: int) -> float:
        """optimizer/mod.rs:249-281: root vectors + observations + NablaModel::update_model; returns the loss.
        ActionModel: fused on the device (f32 forward/backward + Adam, NCCL all-reduce if a communicator is
        attached).  Any other model: its own ``update_model(states, observations, action_weights)`` on host arrays."""
        if isinstance(self.model, ActionModel):
            return self.h.update_model(n_obs_tol)
        sv, obs, w = self.h.write_observations(n_obs_tol)
        return float(self.model.update_model(sv, obs, w))

    def par_reset_trees(self, new_roots=None, *, seed: int = 0, num_permitted_actions_range=None):
        """optimizer/mod.rs:284-360.  ``new_roots=None``: the example's modify_root policy (04-c21-tree.rs:172-206)
        on the device, draws keyed by (seed, reset count, global root index).  Otherwise the caller re-selected the
        roots itself: ``new_roots`` as in par_new."""
        if new_roots is not None:
            self._seed_roots(new_roots)
            return
        lo, hi = num_permitted_actions_range or (0, 0)
        if not isinstance(self.model, ActionModel):
            raise TypeError("device-side root re-selection needs the device model (priors of the new roots)")
        self.h.reset_trees(seed, lo, hi)

    # ---- the example's on-disk outputs (04-c21-tree.rs:118-123,153-157; azdopt_b200/observe.py)
    def argmin_graph6(self) -> bytes:
        """graph6 of the best tree found so far (connected_bitset_graph/graph6.rs:11-39)."""
        from . import observe

        return observe.graph6_of_state(self.argmin_data().parents)

    def tree_dot(self, i: int) -> str:
        """Graphviz DOT of search DAG `i` with the reference's labels (nabla/tree/graphviz.rs:9-51)."""
        from . import observe

        return observe.search_tree_dot(self.h.dump_tree(i))

    def get_trees(self):  # optimizer/mod.rs:34-36, as canonical dumps
        return [self.h.dump_tree(i) for i in range(self.batch)]

    def close(self):
        self.h.close()
