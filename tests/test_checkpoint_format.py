"""CPU checks of the checkpoint format (include/azb.h) as azdopt_b200/checkpoint.py reads it, on blobs built here by hand;
the BestTrees state round trip; the shard helper's choice of files."""
import os

import numpy as np
import pytest

from azdopt_b200 import checkpoint, shard
from azdopt_b200.nabla import BestTree, BestTrees

M64 = (1 << 64) - 1


def _mix(z):
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def _digest_loop(words):
    """The digest written as the header states it, one word at a time."""
    s = 0
    for i, w in enumerate(words):
        s = (s + _mix(int(w) ^ ((i * 0x9E3779B97F4A7C15) & M64))) & M64
    return _mix(s ^ len(words))


def _record(n, rng, nn, nblk, intop):
    a = (n - 1) * (n - 2) // 2 - 1
    w = (a + 31) // 32
    ws = 80 + 2 * ((n + 3) // 4) + 3 * w
    data = ws + nn * (16 + w) + 2 * (nblk - 64) + 2 * intop
    words = rng.integers(0, 1 << 32, size=(data + 1) & ~1, dtype=np.uint64).astype(np.uint32)
    words[2], words[3], words[5] = nn, nblk, intop
    if data & 1:
        words[-1] = 0
    d = _digest_loop(words.view("<u8"))
    return np.concatenate([words, np.array([d], dtype=np.uint64).view(np.uint32)])


def _blob(n=7, roots=3, first=10, n_params=5, seed=0):
    rng = np.random.default_rng(seed)
    recs = [_record(n, rng, nn=1 + r, nblk=64 + 3 * r, intop=r) for r in range(roots)]
    trees = np.concatenate(recs).view(np.uint8)
    off = np.cumsum([0] + [r.size * 4 for r in recs]).astype(np.uint64)
    model = np.zeros((12 * n_params + 7) & ~7, np.uint8)
    model[:12 * n_params] = rng.integers(0, 256, 12 * n_params)
    hw = np.zeros(96, np.uint64)
    hdr, mo = 768, 768
    to = mo + model.size
    tr = to + off.size * 8
    vals = {0: checkpoint.MAGIC, 1: 1, 2: 100, 3: tr + trees.size, 4: n, 15: 3, 16: 25, 25: first, 26: roots, 27: 42, 28: 2,
            29: 1, 35: 1, 36: 0xC0000000, 37: first + 1, 38: 4, 78: n_params, 79: mo, 80: model.size, 81: to, 82: off.size * 8,
            83: tr, 84: trees.size}
    for k, v in vals.items():
        hw[k] = v
    hw[85] = _digest_loop(model.view("<u8"))
    hw[86] = _digest_loop(off)
    hw[95] = _digest_loop(hw[:95])
    assert hdr == hw.nbytes
    return np.concatenate([hw.view(np.uint8), model, off.view(np.uint8), trees])


def test_digest_matches_the_stated_formula():
    rng = np.random.default_rng(1)
    for n in (0, 1, 2, 31, 257):
        w = rng.integers(0, 1 << 63, size=n, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
        assert checkpoint.digest(w.view(np.uint8)) == _digest_loop(w)
        assert checkpoint.digest(w.tobytes()) == _digest_loop(w)
    assert checkpoint.mix64(np.array([0, 5, M64], np.uint64)).tolist() == [_mix(0), _mix(5), _mix(M64)]


def test_order_independent():
    rng = np.random.default_rng(2)
    w = rng.integers(0, 1 << 62, size=100, dtype=np.uint64)
    terms = [_mix(int(x) ^ ((i * 0x9E3779B97F4A7C15) & M64)) for i, x in enumerate(w)]
    s1 = sum(terms) & M64
    s2 = sum(reversed(terms)) & M64
    assert s1 == s2 and _mix(s1 ^ 100) == checkpoint.digest(w.view(np.uint8))


def test_reader_parses_a_hand_built_blob():
    b = _blob()
    h = checkpoint.verify(b)
    assert (h.n_vertices, h.first_root, h.n_roots, h.steps_done, h.resets, h.adam_t, h.n_params) == (7, 10, 3, 42, 2, 1, 5)
    assert h.params_set and h.best_root == 11 and h.best_node == 4 and h.best_eval == np.float32(2.0)
    assert h.n_as_tol == [0, 0, 0] and h.n_as_tol_default == 25
    for i in range(3):
        nn, nblk, intop, _ = checkpoint.record_sizes(checkpoint.tree_record(b, i, h), 7)
        assert (nn, nblk, intop) == (1 + i, 64 + 3 * i, i)
    checkpoint.verify(b.tobytes())


@pytest.mark.parametrize("where,what", [(0, "magic"), (8 * 95 + 1, "header digest"), (768 + 3, "model"),
                                        (-9, "record digest"), (-1, "record digest")])
def test_reader_detects_corruption(where, what):
    b = _blob()
    b[where] ^= 0x20
    with pytest.raises(ValueError, match=what):
        checkpoint.verify(b)


def test_reader_detects_truncation():
    b = _blob()
    with pytest.raises(ValueError):
        checkpoint.verify(b[:-8])
    with pytest.raises(ValueError):
        checkpoint.verify(b[:700])


def _tree(ev, code, root, n=7):
    return BestTree(np.float32(ev), 3.5 + ev, 2, np.arange(n, dtype=np.uint8) // 2, np.array([root, 1], np.uint32), code, root, 9)


def test_best_trees_state_round_trip(tmp_path):
    acc = BestTrees(3).add([_tree(2.0, (5, 1), 4), _tree(1.5, (7, 0), 8), _tree(2.0, (1, 1), 2), _tree(3.0, (9, 9), 1)])
    np.savez(tmp_path / "best.npz", **acc.state())
    back = BestTrees.from_state(np.load(tmp_path / "best.npz"))
    assert back.k == 3
    a, b = acc.result(), back.result()
    assert [(t.eval, t.code, t.root, t.node, t.mu, t.lambda_1) for t in a] == [(t.eval, t.code, t.root, t.node, t.mu, t.lambda_1) for t in b]
    for x, y in zip(a, b):
        assert np.array_equal(x.parents, y.parents) and np.array_equal(x.permitted, y.permitted)
    # merging continues exactly as before the round trip
    more = [_tree(1.0, (9, 9), 0), _tree(2.0, (5, 1), 1)]
    assert [t.code for t in back.add(more).result()] == [t.code for t in acc.add(more).result()]
    empty = BestTrees.from_state(BestTrees(4).state())
    assert empty.k == 4 and empty.result() == []


def test_shard_helper_picks_every_rank_file(tmp_path):
    for r in (2, 0, 1):
        open(shard.checkpoint_path(str(tmp_path), r), "wb").write(b"x")
    open(os.path.join(tmp_path, "rank00003.azbckpt.tmp123"), "wb").write(b"x")
    open(os.path.join(tmp_path, "best.npz"), "wb").write(b"x")
    os.mkdir(os.path.join(tmp_path, "rank00009.azbckpt.d"))
    got = shard.checkpoint_paths(str(tmp_path))
    assert [os.path.basename(p) for p in got] == [f"rank{r:05d}.azbckpt" for r in range(3)]
    assert shard.shard_range(10, 1, 4) == (3, 6)
    with pytest.raises(FileNotFoundError):
        shard.resume_sharded(str(tmp_path / "none"), None, None, 10, 0, 1)
