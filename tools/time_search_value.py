"""Timing of the game-value search (hironaka_b200.search_value).

    python tools/time_search_value.py [--reps 5] [--out results.json]

Workloads (reposition on, max_depth 8, node budget 2^14 per root, capacity 2^26 states, history 2^29 states):
16 384 roots of (5, 3) with entries in [0, 10] and 4 096 roots of (10, 3) in [0, 20], after the Newton filter.  Times
are CUDA events around whole calls (each call ends in a device synchronise), medians of the repeats; two calls must give
the same outputs.  "States created" are nodes - 1 per root.  A separate profiled call splits the GPU time between the
search's own kernels (hk_value_*) and hk_step, which makes the children.  The card's name and power limit are read in
the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import hironaka_b200 as hb  # noqa: E402
from hironaka_b200 import constants as C, ops  # noqa: E402

OPS = C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON


def timed(fn):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    out = fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end), out


def gpu_facts():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the measurement still stands; say what is missing
        q = f"nvidia-smi unavailable: {e}"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def run(name, B, N, d, max_value, reps, capacity, history, max_depth, max_nodes):
    g = torch.Generator(device="cuda").manual_seed(B + N)
    pts = torch.randint(0, max_value + 1, (B, N, d), generator=g, device="cuda", dtype=torch.int32)
    roots = hb.GameBatch(pts, semantics="jax", reposition=True, initial_filter=True).points
    ws = torch.empty(ops.search_value_workspace_bytes(B, N, d, capacity, history), dtype=torch.uint8, device="cuda")

    def call():
        return ops.search_value(roots, ops=OPS, max_depth=max_depth, max_nodes=max_nodes, capacity=capacity,
                                history=history, workspace=ws)
    a, b = call(), call()  # warm-up, and the repeatability of the two
    same = all(torch.equal(x, y) for x, y in zip(a, b))
    times = [timed(call)[0] for _ in range(reps)]
    value, best_mask, nodes, status = (x.cpu().numpy() for x in a)
    created = int(nodes.sum() - B)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    own_us = step_us = 0.0
    per_kernel = {}
    for ev in prof.key_averages():
        t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if "hk" not in ev.key:
            continue
        per_kernel[ev.key[:90]] = {"us": t, "launches": ev.count}
        if "hk_value" in ev.key:
            own_us += t
        else:
            step_us += t
    med = float(np.median(times))
    resolved = status == C.HK_SEARCH_RESOLVED
    return {
        "workload": name, "roots": B, "N": N, "d": d, "max_value": max_value, "max_depth": max_depth,
        "max_nodes": max_nodes, "capacity": capacity, "history": history, "repeatable": bool(same),
        "status_counts": np.bincount(status, minlength=6).tolist(),
        "value_counts_resolved": np.bincount(value[resolved], minlength=max_depth + 1).tolist(),
        "states_created": created, "ms": times, "ms_median": med, "states_per_s": created / (med * 1e-3),
        "profiled_kernel_us": {"hk_value_kernels": own_us, "hk_step_kernels": step_us,
                               "value_share": own_us / max(own_us + step_us, 1e-9), "per_kernel": per_kernel},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--capacity", type=int, default=1 << 26)
    ap.add_argument("--history", type=int, default=1 << 29)
    ap.add_argument("--max-depth", type=int, default=8)
    ap.add_argument("--max-nodes", type=int, default=1 << 14)
    ap.add_argument("--out", default=None, help="also write every result, repeats included, to this JSON file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "time_search_value.py measures on the GPU"
    res = {"gpu": gpu_facts(), "runs": []}
    t0 = time.time()
    for name, B, N, d, mv in [("16384 x (5,3) max 10", 16384, 5, 3, 10), ("4096 x (10,3) max 20", 4096, 10, 3, 20)]:
        r = run(name, B, N, d, mv, a.reps, a.capacity, a.history, a.max_depth, a.max_nodes)
        res["runs"].append(r)
        print(json.dumps({k: v for k, v in r.items() if k != "ms"}), flush=True)
    res["wall_s"] = time.time() - t0
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
