"""PUCT selection (include/azb.h, AZB_SELECT_PUCT) in the CPU oracle (tests/puct_oracle.cpp): against the independent
restatement tests/pyref_puct.py, against scores worked out here from the rule, and against the reference mode.  CPU
only."""
import numpy as np
import pytest

import pyref_puct
from puct_oracle import PuctOptimizer
from test_oracle_tree import _same, digest

F = np.float32


def _run_both(orc, n, parents, masks, steps, prior_fn, c_puct):
    b = len(parents)
    o = PuctOptimizer(n, b, c_puct=c_puct, lambda_method=orc.LAMBDA_DENSE)
    o.set_roots(parents, masks)
    py = pyref_puct.Optimizer(n, parents, [orc.actions_from_mask(m) for m in masks], c_puct=c_puct)
    pri = prior_fn(0)
    o.init_trees(pri)
    py.init_trees(pri)
    for s in range(steps):
        pri = prior_fn(s + 1)
        o.rollout()
        assert o.add_actions(pri) == (py.step(pri) is not None), f"step {s}"
    w = o.walkers()
    for i in range(b):
        d_o, d_p = o.dump_tree(i), py.dump(i, orc.mask_words(n))
        bad = _same(d_o, d_p)
        assert bad is None, f"tree {i}: {bad} differ"
        assert digest(d_o) == digest(d_p)
        assert int(w["pos"][i]) == py.pos[i] and int(w["path_len"][i]) == len(py.paths[i])
        assert list(w["parents"][i]) == py.states[i].parents
        assert orc.actions_from_mask(w["permitted"][i]) == sorted(py.states[i].permitted)
    assert o.argmin()["eval"] == py.best
    k = o.counters()
    assert {key: k[key] for key in py.counters()} == py.counters()
    assert k["n_cur"] == k["n_sel"]
    return o


@pytest.mark.parametrize("n,seed", [(6, 0), (7, 1), (8, 2), (9, 3), (10, 4), (11, 5), (12, 6)])
def test_puct_tie_stress_oracle_matches_python_restatement(orc, n, seed):
    """Priors quantised to three values: equal scores (first maximum wins) at most selections."""
    b, steps = 5, 60
    a_dim = orc.action_dim(n)
    rng = np.random.default_rng(200 + seed)
    parents, masks = orc.generate_roots(seed, 0, b, n, k_min=min(5, a_dim // 2), k_max=a_dim // 2)
    vals = np.array([0.25, 0.5, 0.75], dtype=np.float32)
    _run_both(orc, n, parents, masks, steps, lambda s: rng.choice(vals, size=(b, a_dim)), 1.0)


@pytest.mark.parametrize("c_puct", [0.25, 1.0, 4.0])
def test_puct_hash_priors_oracle_matches_python_restatement(orc, c_puct):
    n, b = 19, 3
    a_dim = orc.action_dim(n)
    parents, masks = orc.generate_roots(11, 0, b, n)
    _run_both(orc, n, parents, masks, 40, lambda s: orc.hash_priors(11, 0, b, a_dim, s), c_puct)


def test_puct_wide_root_oracle_matches_python_restatement(orc):
    """Every action of children 36, 37 and 38 permitted at N = 40: > 100 predictions at the root (four butterfly
    chunks) and, as episodes end within three levels, > 32 kids there (kid slots beyond the first chunk)."""
    n, b = 40, 2
    a_dim = orc.action_dim(n)
    parents, _ = orc.generate_roots(5, 0, b, n)
    acts = [x for v in (36, 37, 38) for x in range(v * (v - 1) // 2 - 1, v * (v - 1) // 2 - 1 + v)]
    masks = np.stack([orc.mask_from_actions(n, acts) for _ in range(b)])
    o = _run_both(orc, n, parents, masks, 120, lambda s: orc.hash_priors(5, 0, b, a_dim, s), 4.0)
    for i in range(b):
        d = o.dump_tree(i)
        assert d["nodes"][0, 5] - d["nodes"][0, 4] > 96
        assert int((d["arcs"][:, 0] == 0).sum()) > 32


def test_puct_hand_built_node(orc):
    """The first two selections at a root worked out from the rule: with no kid N_s = 1 and the highest
    g_j + c_puct * p_j wins; then the root's one kid competes with q = c_s - c*_k, n = n_k + 1."""
    n, c_puct = 9, F(2.0)
    a_dim = orc.action_dim(n)
    parents = np.zeros((1, n), dtype=np.uint8)
    for v in range(2, n - 1):
        parents[0, v] = v - 1  # a path
    legal_all = orc.action_data(parents[0], orc.mask_from_actions(n, range(a_dim)))
    acts = legal_all[:6]
    masks = orc.mask_from_actions(n, acts)[None, :]
    h = np.full((1, a_dim), 0.9, dtype=np.float32)
    h[0, acts] = np.array([0.7, 0.2, 0.5, 0.2, 0.95, 0.6], dtype=np.float32)
    o = PuctOptimizer(n, 1, c_puct=float(c_puct), lambda_method=orc.LAMBDA_DENSE)
    o.set_roots(parents, masks)
    o.init_trees(h)
    d = o.dump_tree(0)
    c_s = d["nodes"][0, :1].view(np.float32)[0]
    legal = [int(a) for a in d["preds"][:, 0]]
    g = d["preds"][:, 1].view(np.float32)
    assert legal == acts and np.array_equal(g, (c_s - h[0, acts]).astype(np.float32))
    # selection 1: N_s = 1, sq = 1, n = 0, q = g_j
    w = [max(F(0), F(F(F(1) - c_s) + gj)) for gj in g]
    z = pyref_puct.prior_sum(w)
    scores = [F(gj + F(F(F(c_puct * F(wj / z)) * F(1)) / F(1))) for gj, wj in zip(g, w)]
    j1 = int(np.argmax(scores))  # the lowest index among equal maxima
    assert j1 == 1  # h = 0.2 twice (j = 1, 3): equal scores, the first one wins
    o.rollout()
    o.add_actions(h)
    d = o.dump_tree(0)
    assert d["arcs"].shape[0] == 1 and int(d["arcs"][0, 0]) == 0 and int(d["arcs"][0, 2]) == j1
    # selection 2 is at the kid, where the walker waits: its own c_s and predictions, no kid of its own
    kid = int(d["arcs"][0, 1])
    lo, hi = int(d["nodes"][kid, 4]), int(d["nodes"][kid, 5])
    c_k = d["nodes"][kid, :1].view(np.float32)[0]
    g2 = d["preds"][lo:hi, 1].view(np.float32)
    w2 = [max(F(0), F(F(F(1) - c_k) + gj)) for gj in g2]
    z2 = pyref_puct.prior_sum(w2)
    scores2 = [F(gj + F(F(c_puct * F(wj / z2)) * F(1))) for gj, wj in zip(g2, w2)]
    j2 = int(np.argmax(scores2))
    o.rollout()
    d2 = o.dump_tree(0)
    assert int(d2["arcs"][1, 0]) == kid and int(d2["arcs"][1, 2]) == lo + j2
    k = o.counters()
    assert k["n_sel"] == k["n_cur"] == 2 and k["n_cand"] == len(acts) + (hi - lo) and k["n_visit"] == 0


def test_puct_hand_built_node_with_kids():
    """A node built by hand with an active kid, an inactive kid and two open predictions; the scores are worked out
    here from the rule in float64 far from any tie and float32 agrees on the winner."""
    t = pyref_puct.PuctTree()
    t.c_puct = F(1.5)
    c_s = F(0.5)
    t.add_node((), c_s)
    t.preds = [[3, F(0.1), None], [5, F(0.4), None], [8, F(0.3), None], [9, F(-0.2), None]]
    t.nodes[0].lo, t.nodes[0].hi = 0, 4
    k1 = t.add_node((5,), F(0.45))
    t.add_arc(0, k1, 1)
    t.nodes[k1].lo, t.nodes[k1].hi, t.nodes[k1].nt, t.nodes[k1].cstar = 0, 2, 3, F(0.2)  # active, n_t = 3
    k2 = t.add_node((8,), F(0.1))
    t.add_arc(0, k2, 2)
    t.nodes[k2].lo, t.nodes[k2].hi, t.nodes[k2].ex = 0, 1, 1  # inactive: skipped
    w = [max(0.0, (1 - 0.5) + g) for g in (0.1, 0.4, 0.3, -0.2)]  # 0.6, 0.9, 0.8, 0.3
    p = [x / sum(w) for x in w]
    sq = np.sqrt(1 + (3 + 1) + (0 + 1))
    s0 = 0.1 + 1.5 * p[0] * sq / 1
    s1 = (0.5 - 0.2) + 1.5 * p[1] * sq / (1 + 4)
    s3 = -0.2 + 1.5 * p[3] * sq / 1
    assert s0 > s1 and s0 > s3
    assert t.next_action(0, 0) == ("U", 0)
    # a larger c* gap makes the kid win: q = 0.5 - (-1.0)
    t.nodes[k1].cstar = F(-1.0)
    assert 1.5 + 1.5 * p[1] * sq / 5 > s0
    assert t.next_action(0, 0) == ("V", 0)  # arc 0 leads to the active kid


def test_puct_changes_trees(orc):
    n, b, steps = 19, 4, 60
    a_dim = orc.action_dim(n)
    parents, masks = orc.generate_roots(2, 0, b, n)

    def run(o):
        o.set_roots(parents, masks)
        o.init_trees(orc.hash_priors(2, 0, b, a_dim, 0))
        imp = o.steps_hash(2, 0, 1, steps)
        return imp, [digest(o.dump_tree(i)) for i in range(b)], o.counters()

    ref = run(orc.Optimizer(n, b, lambda_method=orc.LAMBDA_DENSE))
    puct = run(PuctOptimizer(n, b, c_puct=1.0, lambda_method=orc.LAMBDA_DENSE))
    assert all(x != y for x, y in zip(puct[1], ref[1]))
    assert puct[2]["n_cur"] == puct[2]["n_sel"] and ref[2]["n_cur"] < ref[2]["n_sel"]
    assert puct[2]["n_live"] + puct[2]["n_noop"] == b * steps


@pytest.mark.parametrize("c_puct", [0.0, -1.0, float("inf"), float("nan")])
def test_puct_oracle_rejects_bad_c_puct(orc, c_puct):
    with pytest.raises(ValueError):
        PuctOptimizer(7, 1, c_puct=c_puct)


def test_butterfly_sum_is_the_xor_tree():
    """The chunk sum pairs lanes (i, i^16), then (i, i^8), ...: for these values a left fold rounds differently."""
    vals = [F(1.0)] + [F(2.0 ** -24)] * 31
    fold = F(0)
    for v in vals:
        fold = F(fold + v)
    assert fold == F(1.0)  # each tiny term is lost against 1
    assert pyref_puct.butterfly_sum(vals) > F(1.0)  # the tiny terms meet each other first
