"""azb_checkpoint_size / _save / _load (include/azb.h) on the GPU: a run saved anywhere between calls and loaded into a
fresh handle continues bit for bit like an uninterrupted twin fed the same calls — trees (azb_dump_tree), walkers,
improvement records, argmin, parameters and loss, the roots of later resets, and counters (saved + continued =
uninterrupted) — across execution forms, layouts, resharding, capacities and staging chunks; every malformed blob is
refused before the handle changes."""
import os
import sys

import numpy as np
import pytest
import torch

from azdopt_b200 import checkpoint

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 3


def _handle(capi, n, b, *, first=0, mlp=False, **kw):
    if mlp:
        kw.setdefault("mlp_mode", capi.MLP_TC)
    else:
        kw.setdefault("prior_mode", capi.PRIOR_HASH)
        kw.setdefault("prior_seed", 7)
    return capi.Handle(capi.default_config(n, b, first_root=first, **kw))


def _start(capi, h, seed=3):
    if h.cfg.prior_mode == capi.PRIOR_MLP:
        h.mlp_init(5)
    h.set_roots(*capi.generate_roots(seed, int(h.cfg.first_root), h.b, h.n))
    h.init_trees()
    return h


def _run(h, ops):
    """Feed `ops` to a handle; the log holds every result the calls return."""
    log = []
    for op in ops:
        if op[0] == "step":
            log.append(h.step(op[1], cap=4096))
        elif op[0] == "update":
            log.append(("loss", h.update_model(TOL), h.mlp_get_params()))
        elif op[0] == "reset":
            h.reset_trees(op[1])
            log.append(("roots",) + h.get_roots())
    return log


def _same_log(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        if x[0] == "loss":
            assert x[1] == y[1] and np.array_equal(x[2], y[2])
        elif x[0] == "roots":
            assert np.array_equal(x[1], y[1]) and np.array_equal(x[2], y[2])
        else:
            assert x == y


def _snap(h, trees=None):
    trees = range(h.b) if trees is None else trees
    return dict(trees=[h.dump_tree(i) for i in trees], walkers=h.walkers(), argmin=h.argmin())


def _same_trees(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        for k in x:
            assert np.array_equal(x[k], y[k]), k


def _same_snap(a, b):
    _same_trees(a["trees"], b["trees"])
    for k in a["walkers"]:
        assert np.array_equal(a["walkers"][k], b["walkers"][k]), k
    for k in ("parents", "permitted"):
        assert np.array_equal(a["argmin"][k], b["argmin"][k])
    assert a["argmin"]["eval"] == b["argmin"]["eval"] and a["argmin"]["mu"] == b["argmin"]["mu"]


def _add(c1, c2):
    return {k: c1[k] + c2[k] for k in c1}


def _resume_check(capi, make_saver, make_loader, before, after):
    """Saver runs `before`, saves and is destroyed; a fresh handle from make_loader() loads and runs `after`; the twin
    (make_saver()) runs both.  Returns the blob."""
    twin = _start(capi, make_saver())
    with _start(capi, make_saver()) as h:
        _run(h, before)
        blob = h.checkpoint_save()
        assert blob.size == h.checkpoint_size()
        saved_ct = h.counters()
    checkpoint.verify(blob)
    with make_loader() as r:
        r.checkpoint_load(blob)
        log_r = _run(r, after)
        log_t = _run(twin, before)
        log_t = _run(twin, after)
        _same_log(log_r, log_t)
        _same_snap(_snap(r), _snap(twin))
        assert _add(saved_ct, r.counters()) == twin.counters()
    twin.close()
    return blob


def test_mid_epoch_default_path(capi):
    mk = lambda: _handle(capi, 19, 512, mlp=True, async_workers=capi.ASYNC_AUTO)
    _resume_check(capi, mk, mk, [("step", 800), ("update",), ("reset", 11), ("step", 300)],
                  [("step", 500), ("update",), ("reset", 11), ("step", 200)])


@pytest.mark.parametrize("save_kw,load_kw", [
    (dict(async_workers=0xFFFFFFFF), dict(async_workers=0)),
    (dict(async_workers=0, n_groups=2), dict(async_workers=0xFFFFFFFF)),
    (dict(async_workers=0xFFFFFFFF), dict(async_workers=0, max_episodes=2)),
])
def test_across_execution_forms(capi, save_kw, load_kw):
    _resume_check(capi, lambda: _handle(capi, 19, 1024, mlp=True, **save_kw), lambda: _handle(capi, 19, 1024, mlp=True, **load_kw),
                  [("step", 120)], [("step", 80), ("update",), ("reset", 2), ("step", 30)])


@pytest.mark.parametrize("n,kw", [(19, {}), (19, dict(selection=1, puct_c=1.5)), (33, {}), (64, {})])
def test_layouts(capi, n, kw):
    mk = lambda: _handle(capi, n, 256, max_steps=200, **kw)
    _resume_check(capi, mk, mk, [("step", 90), ("reset", 4), ("step", 40)], [("step", 60), ("reset", 4), ("step", 7)])


def _record_bound(n):
    a = (n - 1) * (n - 2) // 2 - 1
    w = (a + 31) // 32
    ws = 80 + 2 * ((n + 3) // 4) + 3 * w
    return 4 * (ws + 16 + w + 2 * (3 * a + 2) + 1) + 8


@pytest.mark.parametrize("when", ["init", "reset"])
def test_epoch_boundary_blobs_are_small(capi, when):
    mk = lambda: _handle(capi, 19, 512, mlp=True)
    before = [] if when == "init" else [("step", 100), ("update",), ("reset", 5)]
    blob = _resume_check(capi, mk, mk, before, [("step", 50)])
    h = checkpoint.verify(blob)
    t = checkpoint.tree_offsets(blob, h)
    for i in range(h.n_roots):
        nn, _, intop, _ = checkpoint.record_sizes(checkpoint.tree_record(blob, i, h), 19)
        assert nn == 1 and intop == 0
    assert int(t[-1]) <= 512 * _record_bound(19)
    assert blob.size == checkpoint.HEADER_BYTES + h.model[1] + 8 * 513 + int(t[-1])
    assert blob.size < checkpoint.HEADER_BYTES + h.model[1] + 512 * 3000


def test_resharding_on_one_gpu(capi):
    ops1, ops2 = [("step", 70), ("reset", 9), ("step", 30)], [("step", 40), ("reset", 9), ("step", 20)]
    blobs = []
    for lo in (0, 256):
        with _start(capi, _handle(capi, 19, 256, first=lo)) as h:
            _run(h, ops1)
            blobs.append(h.checkpoint_save())
    with _start(capi, _handle(capi, 19, 512)) as one:
        one_log = _run(one, ops1 + ops2)
        ref = _snap(one)
        am = one.argmin()
    for parts in (1, 4):
        b = 512 // parts
        trees, best = [], []
        for k in range(parts):
            with _handle(capi, 19, b, first=k * b) as h:
                h.checkpoint_load(blobs[::-1])  # order does not matter
                log = _run(h, ops2)
                for j in (1, 2):  # the roots the reset drew
                    assert np.array_equal(log[1][j], one_log[4][j][k * b:(k + 1) * b])
                trees += [h.dump_tree(i) for i in range(b)]
                a = h.argmin()
                best.append((a["eval"], k, a["parents"], a["permitted"]))
        _same_trees(trees, ref["trees"])
        ev, _, p, m = min(best, key=lambda x: (x[0], x[1]))
        assert ev == am["eval"] and np.array_equal(p, am["parents"]) and np.array_equal(m, am["permitted"])


def test_capacities(capi):
    mk = lambda: _handle(capi, 19, 256, max_steps=200)
    _resume_check(capi, mk, lambda: _handle(capi, 19, 256, max_steps=500, cap_nodes=900), [("step", 150)], [("step", 50), ("reset", 1), ("step", 150)])
    with _start(capi, mk()) as h:
        h.step(150)
        blob = h.checkpoint_save()
    with _handle(capi, 19, 256, max_steps=100) as r:
        with pytest.raises(capi.AzbError) as e:
            r.checkpoint_load(blob)
        assert e.value.code == capi.ERR_CAPACITY
    with _handle(capi, 19, 256, max_steps=200, cap_nodes=60) as r:
        with pytest.raises(capi.AzbError) as e:
            r.checkpoint_load(blob)
        hd = checkpoint.read_header(blob)
        first = min(i for i in range(256) if checkpoint.record_sizes(checkpoint.tree_record(blob, i, hd), 19)[0] > 60)
        assert e.value.code == capi.ERR_CAPACITY and f"global root {first} " in str(e.value)


def _reheader(blob, word, value):
    b = blob.copy()
    w = b[:checkpoint.HEADER_BYTES].view("<u8")
    w[word] = value
    w[95] = checkpoint.digest(b[:checkpoint.HEADER_BYTES - 8])
    return b


def test_rejections_leave_the_handle_unchanged(capi):
    mk = lambda **kw: _handle(capi, 19, 256, max_steps=200, **kw)
    with _start(capi, mk()) as src:
        src.step(60)
        blob = src.checkpoint_save()
    with _start(capi, _handle(capi, 19, 128, max_steps=200, first=128)) as other:
        other.step(60)
        half = other.checkpoint_save()
    with _start(capi, _handle(capi, 19, 128, max_steps=200)) as other:
        other.step(65)
        q0 = other.checkpoint_save()
    twin, h = _start(capi, mk()), _start(capi, mk())
    twin.step(33)
    h.step(33)
    bad = {
        "c_lower": [(mk(c_lower=2.5), blob)], "c_upper": [(mk(c_upper=9.0), blob)],
        "n_as_tol": [(mk(n_as_tol=(200, 50, 51)), blob)], "mlp_hidden": [(mk(mlp_hidden=(512, 1024, 256)), blob)],
        "mlp_mode": [(mk(mlp_mode=capi.MLP_TC), blob)], "prior_mode": [(mk(prior_mode=capi.PRIOR_INJECTED), blob)],
        "prior_seed": [(mk(prior_seed=8), blob)], "selection": [(mk(selection=1), blob)], "puct_c": [(mk(puct_c=2.0), blob)],
    }
    for field, cases in bad.items():
        for r, b in cases:
            with r:
                with pytest.raises(capi.AzbError) as e:
                    r.checkpoint_load(b)
                assert e.value.code == capi.ERR_INVALID and field in str(e.value), field
    with _handle(capi, 20, 256, max_steps=200) as r:
        with pytest.raises(capi.AzbError) as e:
            r.checkpoint_load(blob)
        assert e.value.code == capi.ERR_INVALID and "n_vertices" in str(e.value)
    cases = [
        [_reheader(blob, 0, 1)], [_reheader(blob, 1, 2)], [_reheader(blob, 2, 99)], [blob[:-8]], [blob[:100]],
        [blob, half],                 # overlapping ranges
        [half],                       # roots 0..127 missing
        [q0, half],                   # different steps
        [_reheader(blob, 25, 256), half],  # roots 0..127 missing, different steps
    ]
    x = blob.copy()
    x[checkpoint.HEADER_BYTES + 5] ^= 1  # the model section
    cases.append([x])
    for bl in cases:
        with pytest.raises(capi.AzbError) as e:
            h.checkpoint_load(bl)
        assert e.value.code == capi.ERR_INVALID
    _same_log(_run(h, [("step", 20)]), _run(twin, [("step", 20)]))
    _same_snap(_snap(h), _snap(twin))
    # one flipped byte inside the record of global root 77
    hd = checkpoint.read_header(blob)
    t = checkpoint.tree_offsets(blob, hd)
    y = blob.copy()
    y[hd.trees[0] + int(t[77]) + 4 * 100 + 2] ^= 0x10
    with pytest.raises(capi.AzbError) as e:
        h.checkpoint_load(y)
    assert e.value.code == capi.ERR_INVALID and "global root 77 " in str(e.value)
    with pytest.raises(capi.AzbError) as e:
        h.step(1)
    assert e.value.code == capi.ERR_STATE
    with pytest.raises(capi.AzbError) as e:
        h.checkpoint_save()
    assert e.value.code == capi.ERR_STATE
    h.checkpoint_load(blob)
    twin.checkpoint_load(blob)
    _same_log(_run(h, [("step", 25)]), _run(twin, [("step", 25)]))
    _same_snap(_snap(h), _snap(twin))
    h.close()
    twin.close()


def test_save_state_errors(capi):
    with _handle(capi, 19, 256, max_steps=200) as h:
        with pytest.raises(capi.AzbError) as e:
            h.checkpoint_save()
        assert e.value.code == capi.ERR_STATE
        _start(capi, h)
        h.step_enqueue(10)
        for fn in (h.checkpoint_save, h.checkpoint_size):
            with pytest.raises(capi.AzbError) as e:
                fn()
            assert e.value.code == capi.ERR_STATE
        h.step(0)
        h.checkpoint_save()
    with _handle(capi, 19, 128, prior_mode=capi.PRIOR_INJECTED) as h:
        h.set_priors(np.full((128, h.a), 0.5, np.float32))
        _start(capi, h)
        sv = np.zeros((128, h.s), np.float32)
        h.rollout_host(sv)
        with pytest.raises(capi.AzbError) as e:
            h.checkpoint_save()
        assert e.value.code == capi.ERR_STATE
        h.add_actions_host(np.full((128, h.a), 0.25, np.float32))
        assert checkpoint.verify(h.checkpoint_save()).steps_done == 1


def test_save_is_read_only(capi):
    mk = lambda: _handle(capi, 19, 512, mlp=True)
    with _start(capi, mk()) as a, _start(capi, mk()) as b:
        la, lb = [], []
        for k in range(4):
            la += _run(a, [("step", 100)])
            s1, s2 = a.checkpoint_save(), a.checkpoint_save()
            assert np.array_equal(s1, s2)
            lb += _run(b, [("step", 100)])
        la += _run(a, [("update",), ("reset", 3), ("step", 10)])
        lb += _run(b, [("update",), ("reset", 3), ("step", 10)])
        _same_log(la, lb)
        _same_snap(_snap(a), _snap(b))
        assert a.counters() == b.counters()


def test_many_staging_chunks(capi, monkeypatch):
    mk = lambda: _handle(capi, 33, 300, max_steps=200)
    with _start(capi, mk()) as h:
        h.step(80)
        one = h.checkpoint_save()
    monkeypatch.setenv("AZB_TEST_CKPT_CHUNK", "4096")
    with _start(capi, mk()) as h:
        h.step(80)
        many = h.checkpoint_save()
    assert np.array_equal(one, many)
    _resume_check(capi, mk, mk, [("step", 80)], [("step", 60), ("reset", 2), ("step", 10)])


def test_reader_restates_every_digest(capi):
    with _start(capi, _handle(capi, 64, 128, mlp=True, max_steps=100)) as h:
        h.step(40)
        blob = h.checkpoint_save()
        a = h.argmin()
    hd = checkpoint.verify(blob)
    assert (hd.n_vertices, hd.n_roots, hd.first_root, hd.steps_done, hd.resets) == (64, 128, 0, 40, 0)
    assert hd.params_set and hd.adam_t == 0
    p, m = hd.best_state
    assert hd.best_eval == a["eval"] and np.array_equal(p, a["parents"]) and np.array_equal(m, a["permitted"])
    params = np.frombuffer(blob[hd.model[0]:hd.model[0] + 4 * hd.n_params].tobytes(), np.float32)
    with _start(capi, _handle(capi, 64, 128, mlp=True, max_steps=100)) as h2:
        assert np.array_equal(params, h2.mlp_get_params())


# ---- 2 GPUs: NCCL training, saved and resumed at world 2 and at world 1
N2, TOTAL2, STEPS2 = 19, 256, 60


def _rank(rank, world, id_path, out_dir, ckpt_dir, phase):
    sys.path.insert(0, ROOT)
    import time

    from azdopt_b200 import capi, shard

    lo, hi = shard.shard_range(TOTAL2, rank, world)
    cfg = capi.default_config(N2, hi - lo, mlp_mode=capi.MLP_TC, max_steps=2 * STEPS2, device=rank, first_root=lo)
    with capi.Handle(cfg) as h:
        if phase == "save":
            _start(capi, h)
            h.step(STEPS2)
        else:
            blobs = [np.memmap(p, dtype=np.uint8, mode="r") for p in shard.checkpoint_paths(ckpt_dir)]
            h.checkpoint_load(blobs)
        uid_file = f"{id_path}.{phase}"
        if rank == 0:
            with open(uid_file + ".tmp", "wb") as f:
                f.write(capi.comm_unique_id())
            os.replace(uid_file + ".tmp", uid_file)
        else:
            for _ in range(600):
                if os.path.exists(uid_file):
                    break
                time.sleep(0.05)
        h.comm_init(open(uid_file, "rb").read(), rank, world)
        if phase == "save":
            loss = h.update_model(TOL)
            h.reset_trees(5)
            h.step(20)
            blob = h.checkpoint_save()
            with open(shard.checkpoint_path(ckpt_dir, rank), "wb") as f:
                f.write(blob.tobytes())
        h.step(STEPS2)
        loss = h.update_model(TOL)
        np.savez(os.path.join(out_dir, f"{phase}{rank}.npz"), loss=loss, params=h.mlp_get_params(),
                 trees=np.concatenate([np.concatenate([v.reshape(-1) for v in h.dump_tree(i).values()]) for i in range(hi - lo)]))


def test_two_gpu_resume(capi, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    ck = tmp_path / "ckpt"
    ck.mkdir()
    for phase in ("save", "load"):
        mp.spawn(_rank, args=(2, str(tmp_path / "id"), str(tmp_path), str(ck), phase), nprocs=2, join=True)
    for k in range(2):
        a, b = np.load(tmp_path / f"save{k}.npz"), np.load(tmp_path / f"load{k}.npz")
        assert a["loss"] == b["loss"] and np.array_equal(a["params"], b["params"]) and np.array_equal(a["trees"], b["trees"])
    # world 1: one handle over all roots from both files; training sums run in another order
    with capi.Handle(capi.default_config(N2, TOTAL2, mlp_mode=capi.MLP_TC, max_steps=2 * STEPS2)) as h:
        from azdopt_b200 import shard

        h.checkpoint_load([np.memmap(p, dtype=np.uint8, mode="r") for p in shard.checkpoint_paths(str(ck))])
        h.step(STEPS2)
        loss = h.update_model(TOL)
        a = np.load(tmp_path / "save0.npz")
        assert abs(float(a["loss"]) - loss) <= 1e-5 * abs(loss)
        assert np.abs(a["params"] - h.mlp_get_params()).max() <= 1e-6
