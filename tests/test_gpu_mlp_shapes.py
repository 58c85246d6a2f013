"""The prior model and the training step against the float64 reference (tests/mlp_ref.py) at every tiling branch of the
tensor-core kernels, at non-default layer widths, inside the search, and block by block for the gradients.

The three forward modes and their bounds:
  * AZB_MLP_FP32 and AZB_MLP_TC3: 1e-5 relative to the float64 forward (the project's bound for f32 results);
  * AZB_MLP_TC (bf16 operands): 2e-3 absolute to the bf16 restatement ``forward_bf16``, 2e-2 absolute to the float64
    forward (the bf16 rounding of weights and activations itself).
Head widths by N (A = (N-1)(N-2)/2 - 1 outputs, 2A inputs): N = 5..23 give a single head tile whose width is npad, a
multiple of 16 (N = 5, 6, 10, 13, 23: npad % 32 == 16); N = 24 two 128-column tiles; N >= 25 64-column tiles over a
64-padded width.  Layer 0 runs 1 (N = 5) to 61 (N = 64) k-blocks of 64, 3x as many in TC3."""
import numpy as np
import pytest

import mlp_ref
from test_oracle_tree import digest

pytestmark = pytest.mark.gpu

B = 300  # rows: two full 128-row tiles and a ragged third
DEFAULT = (512, 1024, 512)


def _mode(capi, mode):
    return {"fp32": capi.MLP_FP32, "tc": capi.MLP_TC, "tc3": capi.MLP_TC3}[mode]


def _mk(capi, n, b, **kw):
    return capi.Handle(capi.default_config(n, b, **kw))


def _dims(capi, n, hidden):
    a = capi.action_dim(n)
    return [2 * a, *hidden, a]


def _assert_forward(y, params, dims, x, mode, what=""):
    """The mode's bound against the float64 reference (module docstring)."""
    y = y.astype(np.float64)
    p, _, _ = mlp_ref.forward(params, dims, x)
    if mode == "tc":
        q, _, _ = mlp_ref.forward_bf16(params, dims, x)
        err_bf16 = np.abs(y - q).max()
        assert err_bf16 <= 2e-3, (what, err_bf16)  # f32 accumulation order only: 2e-3 absolute
        err = np.abs(y - p).max()
        assert err <= 2e-2, (what, err)  # + bf16 weights and activations: 2e-2 absolute
    else:
        rel = (np.abs(y - p) / p).max()
        assert rel <= 1e-5, (what, rel)  # 1e-5 relative (sigmoid outputs are > 0)


def _dsigmoid(z):
    e = np.exp(-np.abs(z))  # sigma'(z) without the cancellation of p (1 - p) at saturated p
    return e / (1.0 + e) ** 2


# how far a mode may move the head's pre-activation, relative to its size |W3| |a3| + |b3|: FP32 and TC3 the 1e-5 of
# their stated bound; TC 2^-6 (a bf16 operand is off by up to 2^-8 of itself, weights and activations alike, and the
# activations carry the earlier layers' roundings)
Z_REL = {"fp32": 1e-5, "tc3": 1e-5, "tc": 2.0 ** -6}


def _stress_bound(params, dims, x, mode):
    """A bound on |p_device - p| derived from a bound on the head's pre-activation z: e_z = Z_REL (|W3| |a3| + |b3|),
    then |dp| <= max sigma'(z') over |z' - z| <= e_z, times e_z, plus 1e-5 p for the sigmoid's own evaluation
    (__expf / expf and one division) in f32.  A saturated output (sigma'(z) ~ 1e-40 at |z| = 90) is held to almost
    exactly 0 or 1; an output near 1/2 to e_z / 4."""
    p, zs, acts = mlp_ref.forward(params, dims, x)
    w3, b3 = mlp_ref.layers(params, dims)[3]
    ez = Z_REL[mode] * (np.abs(acts[3]) @ np.abs(w3).T + np.abs(b3))
    return _dsigmoid(np.maximum(np.abs(zs[3]) - ez, 0.0)) * ez + 1e-5 * p, p


def _stress_params(params, dims):
    """Every parameter times 3 and the head's weights another 10 times (|z| up to ~100: saturated sigmoids), and every
    5th unit of each hidden layer with all-zero incoming weights and bias (its ReLU input is exactly 0)."""
    p = np.asarray(params, dtype=np.float64) * 3.0
    lay = mlp_ref.layers(p, dims)  # views into p
    for l in range(3):
        lay[l][0][::5, :] = 0.0
        lay[l][1][::5] = 0.0
    lay[3][0][:] *= 10.0
    return p.astype(np.float32)


def _forward_case(capi, n, mode, hidden, stress):
    dims = _dims(capi, n, hidden)
    rng = np.random.default_rng(1000 * n + sum(hidden) + len(mode))
    with _mk(capi, n, B, mlp_mode=_mode(capi, mode), mlp_hidden=hidden, max_steps=4) as h:
        h.mlp_init(n)
        params = h.mlp_get_params()
        xs = [(rng.random((B, dims[0])) < 0.3).astype(np.float32)]
        if mode != "tc":  # NablaModel::write_predictions takes any f32 rows; TC is for the 0/1 state vectors
            xs.append((rng.standard_normal((B, dims[0])) * 0.7).astype(np.float32))
        for i, x in enumerate(xs):
            y = h.model_write_predictions(x)
            _assert_forward(y, params, dims, x, mode, f"inputs {i}")
            for k in (1, 127, 128, 129):  # a row's result does not depend on the rows around it
                assert np.array_equal(h.model_write_predictions(x[:k]), y[:k]), (i, k)
        if stress:
            ps = _stress_params(params, dims)
            h.mlp_set_params(ps)
            x = xs[0]
            y = h.model_write_predictions(x).astype(np.float64)
            bound, p = _stress_bound(ps, dims, x, mode)
            assert (np.minimum(p, 1 - p) < 1e-6).mean() > 0.05  # the stress set does saturate
            excess = (np.abs(y - p) - bound).max()
            assert excess <= 0.0, excess
            assert np.all(np.isfinite(y)) and y.min() >= 0.0 and y.max() <= 1.0


@pytest.mark.parametrize("mode", ["fp32", "tc", "tc3"])
@pytest.mark.parametrize("n", [5, 6, 10, 13, 17, 19, 23, 24, 25, 33, 47, 64])
def test_forward_matches_float64_reference_at_every_tiling(capi, n, mode):
    _forward_case(capi, n, mode, DEFAULT, stress=True)


@pytest.mark.parametrize("mode", ["fp32", "tc", "tc3"])
@pytest.mark.parametrize("n,hidden", [(8, (64, 128, 64)), (8, (36, 300, 150)), (8, DEFAULT), (33, (64, 128, 64)),
                                      (33, (36, 300, 150))])
def test_forward_with_non_default_layer_widths(capi, n, hidden, mode):
    """36 pads inside a k-block (to 64), 300 gives npad 320 in 64-column tiles, 150 gives one 192-column tile."""
    _forward_case(capi, n, mode, hidden, stress=False)


WIDE = (36, 300, 150)


@pytest.mark.parametrize("n,mode,hidden,workers", [
    *[(n, m, DEFAULT, 0) for n in (5, 12, 33, 64) for m in ("fp32", "tc", "tc3")],
    *[(n, m, DEFAULT, 4) for n in (12, 33, 64) for m in ("tc", "tc3")],
    (33, "tc", DEFAULT, "shared"),
    (33, "fp32", WIDE, 0), (33, "tc", WIDE, 0), (33, "tc3", WIDE, 0), (33, "tc", WIDE, 4), (33, "tc3", WIDE, 4),
])
def test_search_priors_match_float64_forward_of_the_state_vectors(capi, n, mode, hidden, workers):
    """The priors the search computed for itself — lock step, asynchronous kernel, shared-SM form — equal the float64
    forward of the walkers' state vectors within the mode's bound.  Unlike lock step == async, this fails when both
    forms share a wrong forward."""
    b, steps = 150, 6
    dims = _dims(capi, n, hidden)
    a = dims[4]
    parents, masks = capi.generate_roots(n, 0, b, n, k_min=min(5, a // 2), k_max=a // 2)
    aw = capi.ASYNC_SHARED if workers == "shared" else workers
    with _mk(capi, n, b, mlp_mode=_mode(capi, mode), mlp_hidden=hidden, max_steps=2 * steps + 2, async_workers=aw) as h:
        h.mlp_init(n + 1)
        h.set_roots(parents, masks)
        h.init_trees()
        h.step(steps)
        sv, pr = h.state_vecs(), h.priors()
        assert np.all((sv == 0) | (sv == 1))
        if workers:
            # the asynchronous kernel answers a row when its tree asks: an exhausted root's prior row is an older one
            rows = h.walkers()["path_len"] > 0
            assert rows.sum() >= b // 4
        else:
            rows = np.ones(b, dtype=bool)  # the lock step's last forward covers every row
        params = h.mlp_get_params()
        _assert_forward(pr[rows], params, dims, sv[rows], mode)


# ---- training step ---------------------------------------------------------------------------------------------------
def _grid_params(dims, seed):
    """Weights and biases in {-1, 0, 1} / 32, every 7th hidden unit with zero incoming weights and bias.

    On 0/1 inputs every hidden pre-activation is then a multiple of 2^-5, 2^-10, 2^-15 whose partial sums fit f32's 24
    bits (checked below): the device computes them exactly, in any order, so the ReLU derivative — 0 or 1, with
    ReLU'(0) = 0 — is the same as the reference's for every unit and row.  With random f32 parameters a pre-activation
    within rounding of 0 flips it once in ~10^6 units and moves a whole gradient row, and no elementwise comparison at
    small row counts could be stable."""
    rng = np.random.default_rng(seed)
    p = rng.integers(-1, 2, mlp_ref.num_params(dims)).astype(np.float64) / 32.0
    lay = mlp_ref.layers(p, dims)
    for l in range(3):
        lay[l][0][3::7, :] = 0.0
        lay[l][1][3::7] = 0.0
    return p.astype(np.float32)


def _assert_exact_hidden_layers(params, dims, x):
    a = np.asarray(x, dtype=np.float64)
    for l, (w, b) in enumerate(mlp_ref.layers(params, dims)[:3]):
        grid = 2.0 ** (-5 * (l + 1))
        assert (np.abs(a) @ np.abs(w).T + np.abs(b)).max() < 2.0 ** 24 * grid  # every partial sum is an f32 number
        a = np.maximum(a @ w.T + b, 0.0)


def _weights(rng, kind, rows, a):
    if kind == "random":
        w = (rng.random((rows, a)) < 0.2).astype(np.float32)
        w[0, rng.integers(a)] = 1.0
    elif kind == "single":
        w = np.zeros((rows, a), dtype=np.float32)
        w[rng.integers(rows), rng.integers(a)] = 1.0
    else:  # whole rows of zeros (every row but the first of each pair)
        w = (rng.random((rows, a)) < 0.3).astype(np.float32)
        w[1::2] = 0.0
        w[0, 0] = 1.0
    return w


TRAIN_CASES = [(5, DEFAULT), (12, DEFAULT), (33, DEFAULT), (64, DEFAULT), (8, (64, 128, 64)), (8, WIDE),
               (33, (64, 128, 64)), (33, WIDE)]


@pytest.mark.parametrize("n,hidden", TRAIN_CASES)
def test_gradients_match_float64_block_by_block(capi, n, hidden):
    dims = _dims(capi, n, hidden)
    a = dims[4]
    rng = np.random.default_rng(n + sum(hidden))
    params = _grid_params(dims, n)
    zero_units = [np.arange(3, dims[l + 1], 7) for l in range(3)]
    with _mk(capi, n, B, prior_mode=capi.PRIOR_HASH, mlp_hidden=hidden, max_steps=4) as h:
        h.mlp_set_params(params)
        for rows in (1, 7, 63, 64, 65, B):  # < 8 row groups of the bias sums; around the 64-row GEMM tile; B
            for kind in ("random", "single", "zero_rows"):
                x = (rng.random((rows, dims[0])) < 0.3).astype(np.float32)
                o = rng.random((rows, a)).astype(np.float32)
                w = _weights(rng, kind, rows, a)
                _assert_exact_hidden_layers(params, dims, x)
                loss, g = h.model_gradients(x, o, w)
                want_loss, want = mlp_ref.loss_and_gradients(params, dims, x, o, w)
                what = (rows, kind)
                assert abs(loss - want_loss) <= 1e-5 * want_loss, what  # 1e-5 relative
                for name, s in mlp_ref.blocks(dims):
                    gd, gr = g[s].astype(np.float64), want[s]
                    # per block, so that a small block (a bias) is not hidden under the largest weight block:
                    # 1e-5 relative norm-wise, and elementwise rtol 1e-3 with atol 1e-6 of the block's largest entry
                    assert np.linalg.norm(gd - gr) <= 1e-5 * np.linalg.norm(gr), (what, name)
                    assert np.allclose(gd, gr, rtol=1e-3, atol=1e-6 * np.abs(gr).max()), (what, name)
                gl = mlp_ref.layers(g, dims)
                for l in range(3):  # zero incoming weights and bias: z = 0, ReLU'(0) = 0, gradient exactly 0
                    assert np.all(gl[l][0][zero_units[l]] == 0.0) and np.all(gl[l][1][zero_units[l]] == 0.0), (what, l)


@pytest.mark.parametrize("n,hidden", [(12, DEFAULT), (33, WIDE), (64, DEFAULT)])
def test_adam_steps_match_float64_adam_on_the_device_gradients(capi, n, hidden):
    """model_update against the float64 Adam fed the device's own gradients (model_gradients on the same inputs and
    parameters), so that the Adam kernel is compared alone: agreement to 1e-6 absolute, 1 % of one step's lr."""
    dims = _dims(capi, n, hidden)
    a, rows = dims[4], 65
    rng = np.random.default_rng(n)
    with _mk(capi, n, B, prior_mode=capi.PRIOR_HASH, mlp_hidden=hidden, max_steps=4) as h:
        h.mlp_init(n)
        p0 = h.mlp_get_params()
        cur = p0.astype(np.float64)
        st = mlp_ref.adam_state(cur.size)
        for it in range(3):
            x = (rng.random((rows, dims[0])) < 0.3).astype(np.float32)
            o = rng.random((rows, a)).astype(np.float32)
            w = (rng.random((rows, a)) < 0.2).astype(np.float32)
            _, g = h.model_gradients(x, o, w)
            h.model_update(x, o, w)
            cur = mlp_ref.adam(cur, g, st, lr=1e-4, b1=0.9, b2=0.999, eps=1e-8, l2=1e-6)  # the handle's defaults
            err = np.abs(h.mlp_get_params() - cur).max()
            assert err <= 1e-6, (it, err)
        assert np.abs(h.mlp_get_params() - p0).max() > 1e-4  # it did train


def test_training_rejects_zero_rows_and_more_rows_than_roots(capi):
    n, b = 12, 64
    with _mk(capi, n, b, prior_mode=capi.PRIOR_HASH) as h:
        h.mlp_init(1)
        params = h.mlp_get_params()
        for rows in (0, b + 1):
            x = np.ones((rows, h.s), dtype=np.float32)
            o = np.zeros((rows, h.a), dtype=np.float32)
            w = np.ones((rows, h.a), dtype=np.float32)
            for call in (h.model_gradients, h.model_update):
                with pytest.raises(capi.AzbError) as e:
                    call(x, o, w)
                assert e.value.code == capi.ERR_INVALID, (rows, call.__name__)
        assert np.array_equal(h.mlp_get_params(), params)
        x = np.ones((b, h.s), dtype=np.float32)
        h.model_update(x, np.zeros((b, h.a), dtype=np.float32), np.ones((b, h.a), dtype=np.float32))  # b rows are fine


# ---- the host-facing model call and the walkers' state vectors ------------------------------------------------------
@pytest.mark.parametrize("mode", ["tc", "tc3"])
@pytest.mark.parametrize("n", [19, 64])
def test_host_model_call_leaves_the_search_state_alone(capi, n, mode):
    """With AZB_PRIOR_MLP on the tensor cores the walkers' state vectors are the first layer's input rows.  A host call
    of the model between steps must not change them, nor anything the search does next: same trees, priors and
    improvement log as a twin handle that never made the call."""
    b, steps = 200, 6
    parents, masks = capi.generate_roots(3, 0, b, n)
    kw = dict(mlp_mode=_mode(capi, mode), max_steps=3 * steps + 2)
    rng = np.random.default_rng(n)
    with _mk(capi, n, b, **kw) as h, _mk(capi, n, b, **kw) as twin:
        for t in (h, twin):
            t.mlp_init(4)
            t.set_roots(parents, masks)
            t.init_trees()
            t.step(steps)
        sv = h.state_vecs()
        assert np.array_equal(sv, twin.state_vecs())
        for rows in (b // 2 + 1, b):
            if mode == "tc":
                x = (rng.random((rows, h.s)) < 0.5).astype(np.float32)
            else:  # general rows fill the lo half of the bf16x3 input too
                x = (rng.standard_normal((rows, h.s)) * 0.7).astype(np.float32)
            h.model_write_predictions(x)
            assert np.array_equal(h.state_vecs(), sv), rows
        for k in (1, steps):  # the single-step graph, then a multi-step launch
            assert h.step(k, cap=256) == twin.step(k, cap=256), k
        assert [digest(h.dump_tree(i)) for i in range(b)] == [digest(twin.dump_tree(i)) for i in range(b)]
        assert np.array_equal(h.priors(), twin.priors())
        assert np.array_equal(h.state_vecs(), twin.state_vecs())
