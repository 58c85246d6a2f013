"""The float64 model reference (tests/mlp_ref.py) pinned against torch float64 autograd and torch.optim.Adam, against the
oracle's f32 forward and gradients, and on hand-made bf16 rounding cases.  CPU only."""
import numpy as np
import pytest

import mlp_ref

torch = pytest.importorskip("torch")

# small widths that are not multiples of 16, and one that is
DIMS = [[28, 13, 37, 21, 14], [18, 5, 9, 3, 9], [70, 48, 64, 48, 35]]


def _problem(dims, rows, seed):
    rng = np.random.default_rng(seed)
    params = rng.standard_normal(mlp_ref.num_params(dims)) * 0.4
    x = (rng.random((rows, dims[0])) < 0.3).astype(np.float64)
    o = rng.random((rows, dims[4]))
    w = (rng.random((rows, dims[4])) < 0.3).astype(np.float64)
    w[0, 0] = 1.0
    return params, x, o, w


def _torch_model(params, dims):
    mods = []
    for l, (wt, b) in enumerate(mlp_ref.layers(params, dims)):
        lin = torch.nn.Linear(dims[l], dims[l + 1]).double()
        with torch.no_grad():
            lin.weight.copy_(torch.from_numpy(wt.copy()))
            lin.bias.copy_(torch.from_numpy(b.copy()))
        mods += [lin, torch.nn.ReLU() if l < 3 else torch.nn.Sigmoid()]
    return torch.nn.Sequential(*mods)


def _flat(model, grads=False):
    out = []
    for m in model:
        if isinstance(m, torch.nn.Linear):
            out += [(m.weight.grad if grads else m.weight).detach().reshape(-1), (m.bias.grad if grads else m.bias).detach()]
    return torch.cat(out).numpy()


def _torch_loss(model, x, o, w):
    wt = torch.from_numpy(w)
    return (((model(torch.from_numpy(x)) - torch.from_numpy(o)) ** 2) * (wt / wt.sum())).sum()


def test_blocks_cover_the_parameter_vector_in_dfdx_order():
    dims = DIMS[0]
    bl = mlp_ref.blocks(dims)
    assert [name for name, _ in bl] == ["w0", "b0", "w1", "b1", "w2", "b2", "w3", "b3"]
    assert bl[0][1].start == 0 and all(bl[i][1].stop == bl[i + 1][1].start for i in range(7))
    assert mlp_ref.num_params(dims) == sum(dims[l] * dims[l + 1] + dims[l + 1] for l in range(4))
    assert [s.stop - s.start for _, s in bl] == [28 * 13, 13, 13 * 37, 37, 37 * 21, 21, 21 * 14, 14]


@pytest.mark.parametrize("dims", DIMS)
def test_forward_and_gradients_match_torch_float64(dims):
    params, x, o, w = _problem(dims, 23, 1)
    model = _torch_model(params, dims)
    p, zs, acts = mlp_ref.forward(params, dims, x)
    tp = model(torch.from_numpy(x)).detach().numpy()
    assert np.abs(p - tp).max() <= 1e-12 * np.abs(tp).max()  # float64 against float64: 1e-12 relative
    assert len(zs) == 4 and len(acts) == 5 and acts[0] is not None and np.array_equal(acts[4], p)
    assert all(np.array_equal(acts[l + 1], np.maximum(zs[l], 0)) for l in range(3))
    loss, g = mlp_ref.loss_and_gradients(params, dims, x, o, w)
    tl = _torch_loss(model, x, o, w)
    tl.backward()
    tg = _flat(model, grads=True)
    assert abs(loss - tl.item()) <= 1e-12 * abs(tl.item())
    for name, s in mlp_ref.blocks(dims):
        assert np.abs(g[s] - tg[s]).max() <= 1e-12 * max(np.abs(tg[s]).max(), 1e-300), name


def test_relu_derivative_at_zero_is_zero():
    """A hidden unit with zero incoming weights and bias has z = 0 exactly: its weights get gradient exactly 0."""
    dims = DIMS[0]
    params, x, o, w = _problem(dims, 9, 2)
    lay = mlp_ref.layers(params, dims)  # views into params
    lay[1][0][5, :] = 0.0
    lay[1][1][5] = 0.0
    _, g = mlp_ref.loss_and_gradients(params, dims, x, o, w)
    gl = mlp_ref.layers(g, dims)
    assert np.all(gl[1][0][5, :] == 0.0) and gl[1][1][5] == 0.0
    assert np.any(gl[1][0] != 0.0)


def test_adam_matches_torch_adam_float64():
    dims = DIMS[0]
    params, x, o, w = _problem(dims, 17, 3)
    model = _torch_model(params, dims)
    hp = dict(lr=3e-3, b1=0.8, b2=0.95, eps=1e-7, l2=1e-2)  # away from the defaults so a swapped argument shows
    opt = torch.optim.Adam(model.parameters(), lr=hp["lr"], betas=(hp["b1"], hp["b2"]), eps=hp["eps"], weight_decay=hp["l2"])
    st = mlp_ref.adam_state(params.size)
    cur = params.copy()
    for _ in range(4):
        _, g = mlp_ref.loss_and_gradients(cur, dims, x, o, w)
        cur = mlp_ref.adam(cur, g, st, **hp)
        opt.zero_grad()
        _torch_loss(model, x, o, w).backward()
        opt.step()
        want = _flat(model)
        assert np.abs(cur - want).max() <= 1e-12 * np.abs(want).max()  # 1e-12 relative
    assert st["t"] == 4 and np.abs(cur - params).max() > 1e-3


@pytest.mark.parametrize("dims", DIMS[:2])
def test_agrees_with_the_oracle_f32_model(orc, dims):
    """The float64 reference and the oracle's f32 restatement cannot drift apart: forward and gradients agree within
    f32 accuracy (1e-5 relative; the gradients block by block, norm-wise)."""
    params, x, o, w = _problem(dims, 31, 4)
    p32 = params.astype(np.float32)
    p64 = p32.astype(np.float64)
    y = orc.mlp_forward(p32, dims, x.astype(np.float32))
    p, _, _ = mlp_ref.forward(p64, dims, x)
    assert np.abs(y - p).max() <= 1e-5 * np.abs(p).max()
    loss32, g32 = orc.model_gradients(p32, dims, x.astype(np.float32), o.astype(np.float32), w.astype(np.float32))
    loss, g = mlp_ref.loss_and_gradients(p64, dims, x, o.astype(np.float32), w)
    assert abs(loss32 - loss) <= 1e-5 * loss
    for name, s in mlp_ref.blocks(dims):
        assert np.linalg.norm(g32[s] - g[s]) <= 1e-5 * np.linalg.norm(g[s]), name


def test_bf16_rounding_by_hand():
    u = 2.0 ** -8  # half a bf16 ulp at 1.0
    cases = [
        (1.0, 1.0),
        (1.0 + u, 1.0),                          # halfway, even neighbour is 1.0
        (1.0 + 3 * u, 1.0 + 4 * u),              # halfway, even neighbour is 1 + 2^-6
        (1.0 + u + 2.0 ** -20, 1.0 + 2 * u),     # just above halfway: up
        (-(1.0 + u), -1.0),                      # negative halfway: to even, magnitude down
        (-(1.0 + 3 * u), -(1.0 + 4 * u)),        # negative halfway: to even, magnitude up
        (-(1.0 + u + 2.0 ** -20), -(1.0 + 2 * u)),
        (0.0, 0.0),
        (255.5, 256.0),                          # 255.5 is halfway between 255 and 256 (8 bits): to even 256
        (2.0 ** -130, 2.0 ** -130),              # kept as is (no flushing below bf16's normal range)
    ]
    got = mlp_ref.bf16_round(np.array([c for c, _ in cases]))
    assert got.tolist() == [w for _, w in cases]


def test_bf16_rounding_matches_torch_on_float32_values():
    rng = np.random.default_rng(5)
    v = np.concatenate([rng.standard_normal(20000), rng.standard_normal(2000) * 1e4]).astype(np.float32)
    # exact halfway cases (low 16 bits = 0x8000) with odd and even bf16 neighbours, both signs
    hi = rng.integers(0x3000, 0x5000, 4096, dtype=np.uint32)
    bits = (hi << np.uint32(16)) | np.uint32(0x8000)
    v = np.concatenate([v, bits.view(np.float32), -bits.view(np.float32)])
    want = torch.from_numpy(v).to(torch.bfloat16).to(torch.float64).numpy()
    assert np.array_equal(mlp_ref.bf16_round(v), want)


def test_forward_bf16_rounds_operands_and_hidden_activations():
    dims = DIMS[0]
    params, x, _, _ = _problem(dims, 11, 6)
    x = x * 1.1  # not bf16-exact inputs
    p, zs, acts = mlp_ref.forward_bf16(params, dims, x)
    assert np.array_equal(acts[0], mlp_ref.bf16_round(x))
    for l in range(3):
        assert np.array_equal(acts[l + 1], mlp_ref.bf16_round(np.maximum(zs[l], 0)))
    assert np.array_equal(p, mlp_ref.sigmoid(zs[3]))
