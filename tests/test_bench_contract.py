"""bench.py's host-side pieces that run without a GPU: the reference arm (the restated CPU path timed on the host
cores, the one leg of bench.py that may execute oracle/), the bounded cpu_baseline sample, and the algorithmic-byte
formula of SURVEY.md 8(d)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line(orc):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "12", "--warmup", "3",
                          "--roots", "48"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "mcts_simulations_per_sec" and d["unit"] == "simulations/s"
    assert d["higher_is_better"] is True and d["steps"] == 12 and d["warmup"] == 3 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["config"]["steps_run"] == 12


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                         text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_cpu_sample_is_bounded_in_time(orc):
    import bench

    val, dt, k = bench.cpu_reference_run(19, 64, 400, 2, 0, 2, budget_s=0.05)
    assert k["steps_run"] < 400 and k["steps_run"] % 50 == 0 and val > 0  # stopped after the chunk that crossed the budget
    val2, dt2, k2 = bench.cpu_reference_run(19, 64, 30, 2, 0, 2)
    assert k2["steps_run"] == 30 and k2["n_live"] > 0


def test_algorithmic_bytes_formula():
    import bench

    # SURVEY 8(d) at N = 19: NODE 32, EDGE 20, PRED 12, KEY 24, ST 40, VEC 1216, H 608
    zero = dict(n_sel=0, d_sel=0, n_cand=0, n_probe=0, n_ins=0, n_arc=0, n_pred=0, n_cn=0, d_cn=0, n_reset=0, n_live=0)
    assert bench.algorithmic_bytes(dict(zero, n_live=1), 19) == 2 * 40 + 1216 + 608
    assert bench.algorithmic_bytes(dict(zero, n_probe=1, n_ins=1), 19) == 24 + 32 + 24
    assert bench.algorithmic_bytes(dict(zero, n_sel=1, d_sel=3, n_cand=5), 19) == 32 + 3 * 52 + 5 * 12
    assert bench.algorithmic_bytes(dict(zero, n_cn=2, d_cn=1, n_arc=1, n_pred=7, n_reset=1), 19) == 128 + 20 + 24 + 84 + 40
    assert bench.algorithmic_bytes(dict(zero, n_live=1), 64) == 2 * 308 + 15616 + 7808


class _HostHandle:
    """The reads dump_outputs makes of a handle, answered from host arrays (no device)."""

    def __init__(self, n, b, nodes_per_tree):
        from azdopt_b200 import capi

        self.n, self.b, self.a, self.w, self.nn = n, b, capi.action_dim(n), capi.mask_words(n), nodes_per_tree
        self.rng = np.random.default_rng(0)

    def counters(self):
        from azdopt_b200 import capi

        return {f: i for i, f in enumerate(capi.COUNTER_FIELDS)}

    def argmin(self):
        return dict(parents=np.zeros(self.n, np.uint8), permitted=np.ones(self.w, np.uint32), lambda1=3.5, mu=4,
                    eval=np.float32(1.25))

    def priors(self):
        return self.rng.random((self.b, self.a), dtype=np.float32)

    def state_vecs(self):
        return np.ones((self.b, 2 * self.a), np.float32)

    def walkers(self):
        return dict(path_len=np.arange(self.b, dtype=np.uint32) % 3)

    def tree_sizes(self, i):
        return self.nn, self.nn - 1, 2 * self.nn

    def dump_tree(self, i):
        nodes = np.full((self.nn, 6), i, np.uint32)
        nodes[:, 0], nodes[:, 1] = np.float32(-0.25).view(np.uint32), np.float32(2.75).view(np.uint32)  # c, c* bits
        return dict(nodes=nodes)


def _dump_files(d):
    return {os.path.relpath(os.path.join(dp, f), d): os.path.join(dp, f) for dp, _, fs in os.walk(d) for f in fs}


@pytest.mark.parametrize("b,nodes,budgets", [(300, 50, {}), (3000, 400, dict(row_budget=1_000_000, budget=1_300_000))])
def test_dump_outputs_fit_the_byte_budget(tmp_path, b, nodes, budgets):
    import bench
    from azdopt_b200 import capi

    h = _HostHandle(19, b, nodes)
    bench.dump_outputs(str(tmp_path / "a"), h, capi, 7, 0, **budgets)
    files = _dump_files(tmp_path / "a")
    assert sum(os.path.getsize(f) for f in files.values()) <= budgets.get("budget", 64_000_000)
    got = {name[:-4]: np.load(f) for name, f in files.items()}
    assert all(x.dtype in (np.float32, np.float64) for x in got.values())
    k = len(got["walker_path_len"])
    assert got["priors"].shape == (k, h.a) and got["state_vecs"].shape == (k, 2 * h.a) and got["tree_sizes"].shape == (k, 3)
    assert (k == b) == (not budgets)  # every tree when they fit, else a sample
    dead = got["walker_path_len"] == 0
    assert dead.any() and not got["priors"][dead].any() and not got["state_vecs"][dead].any()
    assert got["state_vecs"][~dead].all() and got["n_improved"][0] == 7 and got["argmin_lambda1"][0] == 3.5
    tn = got["tree_nodes"]
    assert len(tn) and len(tn) % nodes == 0 and (len(tn) // nodes < 32) == bool(budgets)  # the budget stops the trees
    assert (tn[:, 1] == -0.25).all() and (tn[:, 2] == 2.75).all()  # c and c* as values, not bit patterns
    assert (tn[:, 3:] == tn[:, :1]).all()
    bench.dump_outputs(str(tmp_path / "b"), _HostHandle(19, b, nodes), capi, 7, 0, **budgets)  # the sample: seed alone
    assert np.array_equal(np.load(tmp_path / "b" / "tree_sizes.npy"), got["tree_sizes"])
    assert np.array_equal(np.load(tmp_path / "b" / "tree_nodes.npy"), tn)


def test_dump_outputs_of_all_ranks_fit_the_byte_budget(tmp_path):
    """bench.py's layout with 8 ranks: rank 0 in DIR, rank r in DIR/rank<r>; together within the 64 MB."""
    import bench
    from azdopt_b200 import capi

    world = 8
    for r in range(world):
        bench.dump_outputs(str(tmp_path if r == 0 else tmp_path / f"rank{r}"), _HostHandle(19, 4096, 3000), capi, 7, 0,
                           world=world)
    files = _dump_files(tmp_path)
    assert len(files) == 12 * world
    assert 60_000_000 < sum(os.path.getsize(f) for f in files.values()) <= 64_000_000


@pytest.mark.gpu
def test_dump_outputs_repeat_bit_for_bit(tmp_path):
    """Two runs with the same arguments compute the same outputs on the asynchronous kernel (the benchmark's default
    from 1024 roots); --steps sets the timed steps."""
    runs = []
    for d in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "24", "--warmup", "3", "--roots", "1024",
                              "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / d)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr
        line = json.loads(out.stdout)
        assert line["steps"] == 24 and line["config"]["search"].startswith("asynchronous")
        runs.append({f[:-4]: np.load(tmp_path / d / f) for f in os.listdir(tmp_path / d)})
    a, b = runs
    assert sorted(a) == sorted(b) and {"priors", "state_vecs", "counters", "argmin_eval", "tree_nodes"} <= set(a)
    for name in a:
        assert a[name].dtype in (np.float32, np.float64) and np.array_equal(a[name], b[name]), name
    assert a["priors"].shape == (1024, 152)
    live = a["walker_path_len"] > 0
    assert live.any() and ((a["priors"][live] > 0) & (a["priors"][live] < 1)).all()
    assert a["counters"][13] + a["counters"][14] == 1024 * 24  # n_live + n_noop: every root, every timed step
    assert (a["tree_nodes"][:, 1] >= a["tree_nodes"][:, 2]).all()  # c* <= c (decoded costs)
