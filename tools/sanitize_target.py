"""Small workload for compute-sanitizer: every kernel of the library once or more (N=19 and N=33)."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from azdopt_b200 import capi

CASES = ((19, 24, 30, "tc"), (19, 9, 25, "hash"), (33, 6, 12, "fp32"), (19, 130, 6, "groups"), (19, 200, 10, "async"),
         (19, 300, 8, "steal"), (33, 96, 6, "steal"), (64, 40, 4, "steal"))
if len(sys.argv) > 1:  # e.g. `sanitize_target.py async`
    CASES = tuple(c for c in CASES if c[3] in sys.argv[1:])
for n, b, steps, mode in CASES:
    kw = dict(max_steps=steps + 4)
    if mode == "hash":
        kw.update(prior_mode=capi.PRIOR_HASH, max_episodes=2)
    elif mode in ("async", "steal"):
        kw.update(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, async_workers=2)
        os.environ["AZB_ASYNC_STEAL"] = "1" if mode == "steal" else "0"  # the table form / the register form of a tree CTA
    elif mode == "groups":
        kw.update(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC, n_groups=2)
    else:
        kw.update(prior_mode=capi.PRIOR_MLP, mlp_mode=capi.MLP_TC if mode == "tc" else capi.MLP_FP32)
    p, m = capi.generate_roots(1, 0, b, n)
    with capi.Handle(capi.default_config(n, b, **kw)) as h:
        if mode != "hash":
            h.mlp_init(3)
        h.set_roots(p, m)
        h.init_trees()
        h.step(steps)
        h.dump_tree(0)
        h.write_observations(2)
        h.argmin()
        h.eval_costs(p)
        h.init_trees()
        h.step(3)
        print(n, mode, "ok", h.counters()["n_live"])
