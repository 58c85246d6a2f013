"""Throughput of azb_eval_graph_costs64 (ConnectedBitsetGraph<N, B64>) at 33, 48 and 64 vertices.
usage: python tools/graph64_probe.py [m]      prints the card, then one JSON line per (n, density)
Each n runs as trees, with +6 % edges and with +50 % edges (a spanning tree plus G(n, p) edges, p = 0.06 * 2 / n or
0.5 * 2 / n of the n - 1 tree edges, i.e. 1.06 (n - 1) or 1.5 (n - 1) edges on average).  A sample of 64 graphs is
checked: kinds and lambda_1 against the oracle, mu against networkx (the oracle's branch and bound is too slow there)."""
import json
import os
import subprocess
import sys
import time

import networkx as nx
import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from azdopt_b200 import build, capi  # noqa: E402
import graph64_oracle as g64  # noqa: E402  (the checker only)
from graphs64_util import random_connected_graph64  # noqa: E402
from graphs_util import edges_of  # noqa: E402

build()
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
m = int(sys.argv[1]) if len(sys.argv) > 1 else 262144
h = capi.Handle(capi.default_config(6, 2, prior_mode=capi.PRIOR_HASH))
for n in (33, 48, 64):
    for extra in (0.0, 0.06, 0.5):
        p = extra * 2.0 / n
        rng = np.random.default_rng(n + int(100 * extra))
        base = np.stack([random_connected_graph64(rng, n, p) for _ in range(2048)])
        graphs = np.ascontiguousarray(np.tile(base, (m // 2048, 1)))
        h.eval_graph_costs64(graphs[:4096])
        best = min(h.eval_graph_costs64(graphs)[3] for _ in range(3))
        call_ms = 1e30
        for _ in range(3):  # the whole call through the C ABI with host buffers: H2D, kernel, D2H of all three outputs
            t0 = time.perf_counter()
            l1, mu, kinds, _ = h.eval_graph_costs64(graphs)
            call_ms = min(call_ms, (time.perf_counter() - t0) * 1e3)
        for i in range(64):
            assert mu[i] == len(nx.max_weight_matching(nx.Graph(edges_of(base[i])), maxcardinality=True))
            lo = g64.graph64_lambda1(base[i])
            assert abs(lo - l1[i]) <= 1e-12 * lo and np.array_equal(g64.graph64_action_kinds(base[i]), kinds[i])
        print(json.dumps({"n": n, "extra_edges": extra, "mean_edges": float(np.mean([len(edges_of(g)) for g in base[:256]])),
                          "graphs": len(graphs), "kernel_ms": best, "graphs_per_s": len(graphs) / best * 1e3,
                          "call_ms_host_buffers": call_ms, "graphs_per_s_through_the_call": len(graphs) / call_ms * 1e3,
                          "algorithmic_bytes_per_graph": 8 * n + 12 + 4 * ((n * (n - 1) + 31) // 32)}), flush=True)
