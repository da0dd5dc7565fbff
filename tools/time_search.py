"""Timing of the game-tree search (hironaka_b200.search_depth) against the same search written as a Python loop over
the existing ops (ops.host_policy, torch indexing, ops.step).

    python tools/time_search.py [--reps 5] [--out results.json]

Workloads (Zeillinger's host, reposition on, max_depth 64, the default node budget 2^16, capacity 2^24 states):
65 536 roots of (5, 3) with entries in [0, 10] and 16 384 roots of (10, 3) in [0, 20], after the Newton filter.  Both
searches must give the same depth, nodes and status.  Times are CUDA events around whole calls (each call ends in a
device synchronise), medians of repeats that alternate the two implementations.  "Nodes stepped" are the states the
search created (nodes - 1 per root).  A separate profiled call splits the GPU time of search_depth between the new
bookkeeping kernels (hk_search_*) and the existing kernels it launches (hk_host_policy and hk_step).  The card's name and
power limit are read in the same run.
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


def torch_search(roots, max_depth, max_nodes, capacity):
    """The same search as a Python loop: one host_policy and one step launch per level, the bookkeeping in torch."""
    B, N, d = roots.shape
    dev = roots.device
    bound = (1 << 30) // d
    depth = torch.zeros(B, dtype=torch.int32, device=dev)
    nodes = torch.ones(B, dtype=torch.int64, device=dev)
    status = torch.zeros(B, dtype=torch.int8, device=dev)
    front, froot = roots, torch.arange(B, device=dev)
    bitpos = torch.arange(d, device=dev)
    for level in range(max_depth + 1):
        live = front[:, :, 0] >= 0
        is_open = live.sum(1) > 1
        if level == max_depth:
            status[froot[is_open]] = C.HK_SEARCH_MAX_DEPTH
            break
        S = ops.host_policy(front, "zeillinger")
        bits = (S[:, None] >> bitpos) & 1
        c = torch.where(is_open, bits.sum(1), 0).to(torch.int64)
        big = is_open & ((front >= bound) & live[:, :, None]).any(2).any(1)
        ch = torch.zeros(B, dtype=torch.int64, device=dev).index_add_(0, froot, c)
        flagged = torch.zeros(B, dtype=torch.int64, device=dev).index_add_(0, froot, big.to(torch.int64)) > 0
        has = ch > 0
        status[has & flagged] = C.HK_SEARCH_INT32_BOUND
        over = has & ~flagged & (nodes + ch > max_nodes)
        status[over] = C.HK_SEARCH_MAX_NODES
        cand = has & ~flagged & ~over
        keep = cand & (torch.cumsum(torch.where(cand, ch, 0), 0) <= capacity)
        status[cand & ~keep] = C.HK_SEARCH_CAPACITY
        nodes += torch.where(keep, ch, 0)
        depth[keep] = level + 1
        parents = torch.nonzero(keep[froot] & (c > 0)).squeeze(1)
        if parents.numel() == 0:
            break
        cp = c[parents]
        idx = torch.repeat_interleave(parents, cp)
        start = torch.repeat_interleave(torch.cumsum(cp, 0) - cp, cp)
        rank = torch.arange(idx.numel(), device=dev) - start  # j: this child plays the j-th axis of the set
        cb = torch.cumsum(bits[idx], 1)
        axis = ((cb == (rank + 1)[:, None]) & (bits[idx] == 1)).to(torch.int32).argmax(1).to(torch.int32)
        front = front[idx].contiguous()
        ops.step(front, S[idx], axis, ops=OPS, flags=0, inplace=True)
        froot = froot[idx]
    return depth, nodes, status


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


def run(name, B, N, d, max_value, reps, capacity, max_depth=64, max_nodes=1 << 16):
    g = torch.Generator(device="cuda").manual_seed(B + N)
    pts = torch.randint(0, max_value + 1, (B, N, d), generator=g, device="cuda", dtype=torch.int32)
    roots = hb.GameBatch(pts, semantics="jax", reposition=True, initial_filter=True).points
    ws = torch.empty(ops.search_workspace_bytes(B, N, d, capacity), dtype=torch.uint8, device="cuda")

    def gpu():
        return ops.search_depth(roots, flags=C.HK_F_HOST_ZEILLINGER, ops=OPS, max_depth=max_depth, max_nodes=max_nodes,
                                capacity=capacity, workspace=ws)

    def loop():
        return torch_search(roots, max_depth, max_nodes, capacity)
    a, b = gpu(), loop()  # warm-up, and the parity of the two
    same = all(torch.equal(x, y) for x, y in zip(a, b))
    t_gpu, t_loop = [], []
    for _ in range(reps):  # alternated
        t_gpu.append(timed(gpu)[0])
        t_loop.append(timed(loop)[0])
    depth, nodes, status = (x.cpu().numpy() for x in a)
    levels = int(min(depth.max() + 1, max_depth + 1))
    stepped = int(nodes.sum() - B)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        gpu()
        torch.cuda.synchronize()
    new_us = old_us = 0.0
    per_kernel = {}
    for ev in prof.key_averages():
        t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if "hk" not in ev.key:
            continue
        per_kernel[ev.key[:90]] = {"us": t, "launches": ev.count}
        if "hk_search" in ev.key:
            new_us += t
        else:
            old_us += t
    mg, ml = float(np.median(t_gpu)), float(np.median(t_loop))
    return {
        "workload": name, "roots": B, "N": N, "d": d, "max_value": max_value, "max_depth": max_depth,
        "max_nodes": max_nodes, "capacity": capacity, "same_outputs": bool(same),
        "status_counts": np.bincount(status, minlength=5).tolist(), "depth_max": int(depth.max()),
        "depth_mean": float(depth.mean()), "nodes_mean": float(nodes.mean()), "nodes_stepped": stepped, "levels": levels,
        "search_ms": t_gpu, "loop_ms": t_loop, "search_ms_median": mg, "loop_ms_median": ml,
        "search_nodes_per_s": stepped / (mg * 1e-3), "loop_nodes_per_s": stepped / (ml * 1e-3),
        "search_ms_per_level": mg / levels, "loop_ms_per_level": ml / levels, "speedup": ml / mg,
        "profiled_kernel_us": {"hk_search_kernels": new_us, "existing_kernels": old_us,
                               "new_share": new_us / max(new_us + old_us, 1e-9), "per_kernel": per_kernel},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--capacity", type=int, default=1 << 24)
    ap.add_argument("--out", default=None, help="also write every result, repeats included, to this JSON file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "time_search.py measures on the GPU"
    res = {"gpu": gpu_facts(), "runs": []}
    t0 = time.time()
    for name, B, N, d, mv in [("65536 x (5,3) max 10", 65536, 5, 3, 10), ("16384 x (10,3) max 20", 16384, 10, 3, 20)]:
        r = run(name, B, N, d, mv, a.reps, a.capacity)
        res["runs"].append(r)
        print(json.dumps({k: v for k, v in r.items() if k not in ("search_ms", "loop_ms")}), flush=True)
    res["wall_s"] = time.time() - t0
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
