"""Hidden layers handed over in tensor memory (azb_async.cuh, "Hidden layers in tensor memory").  A single model SM with
bf16 operands keeps every hidden layer of width <= 512 that follows a layer fed through shared memory in TMEM, as the
next layer's A operand; wider layers, worker groups (G > 1) and AZB_MLP_TC3 keep the hand-over through the L2 scratch.
Either way the asynchronous kernel must give exactly what the lock step gives: the same bf16 activations, accumulated
over K in the same order of 16-deep k-steps."""
import pytest

from test_gpu_async import _mk, _same

pytestmark = pytest.mark.gpu

DEFAULT = (512, 1024, 512)


@pytest.mark.parametrize("n,hidden,group,mlp", [
    # default widths: H1 and H3 in TMEM, H2 through L2; the head in one pass (N <= 23) or 128-column passes (N = 64)
    (5, DEFAULT, 1, "tc"), (19, DEFAULT, 1, "tc"), (23, DEFAULT, 1, "tc"), (64, DEFAULT, 1, "tc"),
    # H1 and H3 in TMEM, the 768-wide H2 through L2 inside the same tile
    (19, (256, 768, 384), 1, "tc"),
    # the 384-wide H2 through L2 all the same: its layer reads H1 from TMEM, whose columns it would overwrite
    (19, (256, 384, 512), 1, "tc"),
    # a 64-wide H1 (one 64-column block), 128-column passes over 320 columns with a 64-column last pass, a 192-wide H3
    (33, (36, 300, 150), 1, "tc"),
    # the L2 hand-over throughout
    (19, DEFAULT, 2, "tc"), (19, DEFAULT, 1, "tc3"),
])
def test_tmem_handover_equals_lock_step(capi, monkeypatch, n, hidden, group, mlp):
    steps, b = 20, 300
    monkeypatch.setenv("AZB_ASYNC_GROUP", str(group))
    a = capi.action_dim(n)
    parents, masks = capi.generate_roots(n, 0, b, n, k_min=min(5, a // 2), k_max=a // 2)
    kw = dict(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC3 if mlp == "tc3" else capi.MLP_TC, mlp_hidden=hidden,
              max_steps=2 * steps + 2)
    with _mk(capi, n, b, **kw) as lock, _mk(capi, n, b, async_workers=4, **kw) as asy:
        for h in (lock, asy):
            h.mlp_init(7)
            h.set_roots(parents, masks)
            h.init_trees()
        n1, log1 = lock.step(steps, cap=256)
        n2, log2 = asy.step(steps, cap=256)
        assert n1 == n2 and [tuple(x) for x in log1] == [tuple(x) for x in log2]
        _same(lock, asy, b)
        for h in (lock, asy):
            h.step(steps)
        _same(lock, asy, b)
