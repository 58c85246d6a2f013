"""Checkpoint cost on the GPU: blob bytes, the pack and unpack kernel times (torch.profiler, CUDA activities) as GB/s
against a device-to-device copy measured in the same process, and the whole azb_checkpoint_save / _load calls into
pageable and pinned host memory, after an epoch of 800 steps with the tensor-core model.

    python tools/checkpoint_probe.py --out DIR      (writes DIR/checkpoint_probe.json)
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from azdopt_b200 import capi  # noqa: E402

CASES = [(19, 4096), (19, 65536), (64, 1024)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def copy_peak_gbs():
    """device-to-device copy of 2 GiB, best of 10: bytes read + written over time"""
    a = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    best = 1e9
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return 2 * a.numel() / (best * 1e-3) / 1e9


def kernel_ms(fn, names):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in names}
    for ev in prof.events():
        for k in names:
            if k in ev.name and ev.device_type.name == "CUDA":
                out[k] += ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3
    return out


def timed(fn, reps=3):
    best = 1e9
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t0)
    return best * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for checkpoint_probe.json")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    res = dict(gpu=gpu_info(), copy_peak_gbs=copy_peak_gbs(), cases=[])
    for n, b in CASES:
        cfg = capi.default_config(n, b, mlp_mode=capi.MLP_TC, async_workers=capi.ASYNC_AUTO)
        with capi.Handle(cfg) as h:
            h.mlp_init(1)
            h.set_roots(*capi.generate_roots(2, 0, b, n))
            h.init_trees()
            t0 = time.perf_counter()
            h.step(800)
            search_ms = (time.perf_counter() - t0) * 1e3
            size = h.checkpoint_size()
            pageable = np.empty(size, np.uint8)
            pinned = torch.empty(size, dtype=torch.uint8, pin_memory=True).numpy()
            h.checkpoint_save(pageable)  # warm-up: the staging slab
            save_pageable = timed(lambda: h.checkpoint_save(pageable))
            save_pinned = timed(lambda: h.checkpoint_save(pinned))
            assert np.array_equal(pageable, pinned)
            km_save = kernel_ms(lambda: h.checkpoint_save(pinned), ["azb_ckpt_pack_kernel", "azb_ckpt_size_kernel"])
            from azdopt_b200 import checkpoint

            hd = checkpoint.read_header(pinned)
            trees_bytes = hd.trees[1]
        with capi.Handle(cfg) as r:
            r.checkpoint_load(pageable)  # warm-up
            load_pageable = timed(lambda: r.checkpoint_load(pageable))
            load_pinned = timed(lambda: r.checkpoint_load(pinned))
            km_load = kernel_ms(lambda: r.checkpoint_load(pinned), ["azb_ckpt_unpack_kernel", "azb_ckpt_hash_kernel"])
            assert np.array_equal(r.checkpoint_save(), pinned)
        row = dict(n=n, roots=b, steps=800, search_ms_800=search_ms, blob_bytes=size, tree_bytes=trees_bytes, model_bytes=hd.model[1],
                   save_ms_pageable=save_pageable, save_ms_pinned=save_pinned, load_ms_pageable=load_pageable, load_ms_pinned=load_pinned,
                   pack_ms=km_save["azb_ckpt_pack_kernel"], size_ms=km_save["azb_ckpt_size_kernel"],
                   unpack_ms=km_load["azb_ckpt_unpack_kernel"], hash_ms=km_load["azb_ckpt_hash_kernel"])
        # pack and unpack read the records once and write them once
        row["pack_gbs"] = 2 * trees_bytes / (row["pack_ms"] * 1e-3) / 1e9 if row["pack_ms"] else None
        row["unpack_gbs"] = 2 * trees_bytes / (row["unpack_ms"] * 1e-3) / 1e9 if row["unpack_ms"] else None
        res["cases"].append(row)
        print(json.dumps(row), flush=True)
    with open(os.path.join(args.out, "checkpoint_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"], copy_peak_gbs=res["copy_peak_gbs"])))


if __name__ == "__main__":
    main()
