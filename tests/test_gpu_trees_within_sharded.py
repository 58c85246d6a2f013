"""azb_comm_trees_within (include/azb.h) on the GPU: the growth of azb_trees_within split over the ranks of a
communicator must return, on every rank, bit for bit what azb_trees_within returns on one handle.  One GPU: a
communicator of one rank, the state refusal, the read-only property, and three ranks that share the GPU.  Two or more
GPUs: up to 4 ranks, one GPU each.  The ranks run with different chunk sizes and are checked against the one-handle
result computed in rank 0's process, together with refusals every rank must agree on."""
import multiprocessing
import os
import re
import sys
import time

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("code", "parents", "lambda1", "mu", "eval")
TIMEOUT_S = 900


def _star_key(h):
    lam, mu, _, _ = h.eval_costs(np.zeros((1, h.n), dtype=np.uint8))
    return float(mu[0]) + float(lam[0])


def _same(a, b):
    """Every output equal bit for bit (arrays compared as raw bytes)."""
    assert (a["n_within"], a["n_below"]) == (b["n_within"], b["n_below"])
    for f in FIELDS:
        x, y = np.asarray(a[f]), np.asarray(b[f])
        assert x.shape == y.shape and x.tobytes() == y.tobytes(), f


def _solo_comm(capi, h):
    h.comm_init(capi.comm_unique_id(), 0, 1)


@pytest.mark.parametrize("n,offset,chunk", [(26, 0.5, None), (26, 0.5, "97"), (33, 0.0, None), (48, 0.0, None)])
def test_one_rank_equals_the_local_call(capi, monkeypatch, n, offset, chunk):
    if chunk:
        monkeypatch.setenv("AZB_TEST_GROW_CHUNK", chunk)
    with capi.Handle(capi.default_config(n, 1)) as h:
        bound = None if offset == 0.0 else _star_key(h) + offset
        local = h.trees_within(bound, k=65536)
        _solo_comm(capi, h)
        sharded = h.comm_trees_within(bound, k=65536)
        _same(sharded, local)
        assert local["n_within"] >= 1
        _same(h.trees_within(bound, k=65536), local)  # with a communicator attached the local call stays local


def test_without_a_communicator_the_call_is_refused(capi):
    with capi.Handle(capi.default_config(20, 1)) as h:
        with pytest.raises(capi.AzbError) as e:
            h.comm_trees_within(k=10)
        assert e.value.code == capi.ERR_STATE
        assert h.trees_within(k=10)["n_within"] >= 1


def test_a_call_on_a_handle_with_trees_changes_nothing(capi):
    n, b = 30, 64
    cfg = capi.default_config(n, b, prior_mode=capi.PRIOR_HASH, prior_seed=3, max_steps=200)
    with capi.Handle(cfg) as h:
        p, m = capi.generate_roots(3, 0, b, n)
        h.set_roots(p, m)
        h.init_trees()
        h.step(40)
        _solo_comm(capi, h)
        before = h.checkpoint_save().copy()
        got = h.comm_trees_within(k=500)
        assert got["n_within"] >= 1
        assert np.array_equal(h.checkpoint_save(), before)


# ---- several ranks ----------------------------------------------------------------------------------------------------
CASES = [(26, 0.0), (26, 0.5), (40, 0.0), (64, 0.0)]  # (N, offset from the star's key), one GPU per rank
SHARED_CASES = [(26, 0.0), (26, 0.5), (40, 0.0)]      # ranks sharing one GPU exchange through host sockets: smaller
KS = (3, 65536)


def _chunk(n, rank):
    # different on every rank, so the ranks' round counts differ and some take part with empty chunks; small chunks
    # (many rounds) where the levels are small, larger ones as they grow
    return str(97 + 50 * rank) if n < 40 else str(4001 + 500 * rank) if n < 64 else str((1 << 20) + 50007 * rank)


def _uid(capi, rank, path):
    if rank == 0:
        with open(path + ".tmp", "wb") as f:
            f.write(capi.comm_unique_id())
        os.replace(path + ".tmp", path)
    deadline = time.monotonic() + 300
    while not os.path.exists(path):
        if time.monotonic() > deadline:
            raise TimeoutError(path)
        time.sleep(0.05)
    return open(path, "rb").read()


def _save(out, key, r):
    for f in FIELDS:
        out[f"{key}/{f}"] = np.asarray(r[f])
    out[f"{key}/counts"] = np.array([r["n_within"], r["n_below"]], dtype=np.uint64)


def _refusal(capi, out, key, call):
    try:
        call()
        out[key] = np.array([-1])
        out[key + "/msg"] = np.array("")
    except capi.AzbError as e:
        out[key] = np.array([e.code])
        out[key + "/msg"] = np.array(str(e))


def _worker(rank, world, tmp, cases, shared):
    sys.path.insert(0, ROOT)
    if shared:
        # NCCL refuses two ranks of one communicator on one GPU of one host; a host id of its own per rank makes them
        # peers on different hosts, which exchange through sockets (here over the loopback interface)
        os.environ.update(NCCL_HOSTID=f"azb-rank-{rank}", NCCL_SOCKET_IFNAME="lo", NCCL_IB_DISABLE="1")
    from azdopt_b200 import capi

    os.environ.pop("AZB_TEST_GROW_CHUNK", None)
    out = {}
    if rank == 0:  # the one-handle results, in rank 0's process
        for n, off in cases:
            with capi.Handle(capi.default_config(n, 1)) as h:
                bound = None if off == 0.0 else _star_key(h) + off
                for k in KS:
                    _save(out, f"ref/{n}/{off}/{k}", h.trees_within(bound, k=k))
                if n == 26:
                    _refusal(capi, out, "ref/cap", lambda: h.trees_within(k=10, max_level=4))
    for n in sorted({n for n, _ in cases}):
        os.environ["AZB_TEST_GROW_CHUNK"] = _chunk(n, rank)
        with capi.Handle(capi.default_config(n, 1, device=0 if shared else rank)) as h:
            h.comm_init(_uid(capi, rank, os.path.join(tmp, f"id{n}")), rank, world)
            star = _star_key(h)
            for nn, off in cases:
                if nn == n:
                    for k in KS:
                        _save(out, f"got/{n}/{off}/{k}", h.comm_trees_within(None if off == 0.0 else star + off, k=k))
            if n == 26:
                _save(out, "got/none", h.comm_trees_within(1.0, k=10))  # below every key
                refusals = [("k0", lambda: h.comm_trees_within(k=0 if rank == 1 else 10)),
                            ("bounds", lambda: h.comm_trees_within(star + 0.5 + 0.01 * rank, k=10)),
                            ("cap", lambda: h.comm_trees_within(k=10, max_level=4))]
                for name, call in refusals:
                    _refusal(capi, out, f"got/{name}", call)
                    _save(out, f"got/after_{name}", h.comm_trees_within(star + 0.5, k=3))  # the communicator still works
    np.savez(os.path.join(tmp, f"r{rank}.npz"), **out)


def _spawn(world, tmp, cases, shared):
    """The ranks as processes; ones still running after TIMEOUT_S are terminated and reaped, and the test fails."""
    ctx = multiprocessing.get_context("spawn")
    procs = [ctx.Process(target=_worker, args=(r, world, str(tmp), cases, shared)) for r in range(world)]
    for p in procs:
        p.start()
    deadline = time.monotonic() + TIMEOUT_S
    for p in procs:
        p.join(max(0.0, deadline - time.monotonic()))
    hung = [r for r, p in enumerate(procs) if p.is_alive()]
    for p in procs:
        if p.is_alive():
            p.terminate()
            p.join(10)
        if p.is_alive():
            p.kill()
            p.join()
    assert not hung, f"ranks {hung} still running after {TIMEOUT_S} s"
    assert [p.exitcode for p in procs] == [0] * world


def _get(d, key):
    return dict(n_within=int(d[f"{key}/counts"][0]), n_below=int(d[f"{key}/counts"][1]),
                **{f: d[f"{key}/{f}"] for f in FIELDS})


def _level(msg):
    m = re.search(r"level (\d+) \(trees on", msg)
    assert m, msg
    return int(m.group(1))


def _check(capi, tmp, world, cases, shared):
    _spawn(world, tmp, cases, shared)
    r = [dict(np.load(tmp / f"r{k}.npz")) for k in range(world)]
    ref = r[0]
    for n, off in cases:
        for k in KS:
            want = _get(ref, f"ref/{n}/{off}/{k}")
            for rank in range(world):
                _same(_get(r[rank], f"got/{n}/{off}/{k}"), want)
    after = _get(ref, "ref/26/0.5/3")
    assert int(ref["ref/cap"][0]) == capi.ERR_CAPACITY
    cap_level = _level(str(ref["ref/cap/msg"]))
    for rank in range(world):
        d = r[rank]
        none = _get(d, "got/none")
        assert none["n_within"] == 0 and len(none["code"]) == 0
        assert int(d["got/k0"][0]) == capi.ERR_INVALID and "rank 1" in str(d["got/k0/msg"])
        assert int(d["got/bounds"][0]) == capi.ERR_INVALID and "bound" in str(d["got/bounds/msg"])
        assert int(d["got/cap"][0]) == capi.ERR_CAPACITY and _level(str(d["got/cap/msg"])) == cap_level
        for name in ("k0", "bounds", "cap"):
            _same(_get(d, f"got/after_{name}"), after)
    return ref


def test_ranks_equal_one_handle(capi, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ref = _check(capi, tmp_path, min(torch.cuda.device_count(), 4), CASES, shared=False)
    star64 = _get(ref, "ref/64/0.0/65536")
    assert (star64["n_within"], star64["n_below"]) == (27618, 27617)


def test_ranks_sharing_one_gpu_equal_one_handle(capi, tmp_path):
    """Three ranks on GPU 0: the routing by owner, the rounds with empty chunks and the agreed refusals on any machine."""
    _check(capi, tmp_path, 3, SHARED_CASES, shared=True)
