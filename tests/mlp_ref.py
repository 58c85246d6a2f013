"""A plain float64 restatement of the prior model and its training step (test infrastructure, CPU only).

Independent of oracle/oracle.py: the parameter vector is in dfdx order — per layer weight[out][in], then bias[out] —
for three ReLU layers and a Sigmoid head.  ``forward_bf16`` restates what AZB_MLP_TC computes (bf16 operands, full
precision bias and accumulation), with the rounding done on float64 bit patterns.
"""
from __future__ import annotations

import numpy as np


def blocks(dims):
    """[(name, slice)] of every weight and bias block in parameter order: w0, b0, w1, b1, w2, b2, w3, b3."""
    out, off = [], 0
    for l in range(4):
        k, n = int(dims[l]), int(dims[l + 1])
        out.append((f"w{l}", slice(off, off + k * n)))
        out.append((f"b{l}", slice(off + k * n, off + k * n + n)))
        off += k * n + n
    return out


def num_params(dims):
    return blocks(dims)[-1][1].stop


def layers(params, dims):
    """[(weight [out][in], bias [out])] as float64 views of the flat parameter vector."""
    p = np.asarray(params, dtype=np.float64)
    bl = blocks(dims)
    return [(p[bl[2 * l][1]].reshape(int(dims[l + 1]), int(dims[l])), p[bl[2 * l + 1][1]]) for l in range(4)]


def sigmoid(z):
    # the two branches keep exp's argument <= 0: no overflow for large |z|
    e = np.exp(-np.abs(z))
    return np.where(z >= 0, 1.0 / (1.0 + e), e / (1.0 + e))


def forward(params, dims, x):
    """(p, zs, acts): the head's output, the four pre-activations and the activations acts[0] = x .. acts[4] = p."""
    acts = [np.asarray(x, dtype=np.float64)]
    zs = []
    for l, (w, b) in enumerate(layers(params, dims)):
        z = acts[-1] @ w.T + b
        zs.append(z)
        acts.append(np.maximum(z, 0.0) if l < 3 else sigmoid(z))
    return acts[-1], zs, acts


def bf16_round(a):
    """Round to the nearest bfloat16 (8 significant bits), ties to even, on float64 bit patterns; returned as float64.

    For float32 inputs this is exactly the float32 -> bf16 conversion.  Values below bf16's normal range are not
    flushed (the model never produces them at a size that matters)."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    u = a.view(np.uint64)
    drop = np.uint64(45)  # 52 stored bits of float64 - 7 stored bits of bf16
    lsb = (u >> drop) & np.uint64(1)
    r = (u + (np.uint64(1) << (drop - np.uint64(1))) - np.uint64(1) + lsb) & ~((np.uint64(1) << drop) - np.uint64(1))
    r = np.where(np.isfinite(a), r, u)
    return r.view(np.float64)


def forward_bf16(params, dims, x):
    """(p, zs, acts) of AZB_MLP_TC: inputs, weights and every hidden activation (after the ReLU) rounded to bf16;
    bias added in full precision, accumulation in float64."""
    acts = [bf16_round(x)]
    zs = []
    for l, (w, b) in enumerate(layers(params, dims)):
        z = acts[-1] @ bf16_round(w).T + b
        zs.append(z)
        acts.append(bf16_round(np.maximum(z, 0.0)) if l < 3 else sigmoid(z))
    return acts[-1], zs, acts


def loss_and_gradients(params, dims, x, o, w):
    """ActionModel::update_model's objective: w_n = w / sum(w), loss = sum (p - o)^2 w_n, and d loss / d params flat
    in parameter order.  ReLU'(0) = 0."""
    p, zs, acts = forward(params, dims, x)
    o = np.asarray(o, dtype=np.float64)
    w = np.asarray(w, dtype=np.float64)
    wn = w / w.sum()
    d = p - o
    loss = float((d * d * wn).sum())
    dz = 2.0 * d * wn * p * (1.0 - p)
    grads = np.zeros(num_params(dims), dtype=np.float64)
    bl = blocks(dims)
    lay = layers(params, dims)
    for l in range(3, -1, -1):
        grads[bl[2 * l][1]] = (dz.T @ acts[l]).reshape(-1)
        grads[bl[2 * l + 1][1]] = dz.sum(axis=0)
        if l > 0:
            dz = (dz @ lay[l][0]) * (zs[l - 1] > 0)
    return loss, grads


def adam(params, grads, state, lr=1e-4, b1=0.9, b2=0.999, eps=1e-8, l2=1e-6):
    """One dfdx 0.13 Adam step with WeightDecay::L2 (l2 * p added to the gradient before the moments), float64.
    ``state`` is a dict with "m", "v" (arrays) and "t" (steps taken), updated in place; returns the new parameters."""
    p = np.asarray(params, dtype=np.float64)
    g = np.asarray(grads, dtype=np.float64) + l2 * p
    state["t"] += 1
    t = state["t"]
    state["m"] = b1 * state["m"] + (1.0 - b1) * g
    state["v"] = b2 * state["v"] + (1.0 - b2) * g * g
    mh = state["m"] / (1.0 - b1 ** t)
    vh = state["v"] / (1.0 - b2 ** t)
    return p - lr * mh / (np.sqrt(vh) + eps)


def adam_state(n):
    return {"m": np.zeros(n), "v": np.zeros(n), "t": 0}
