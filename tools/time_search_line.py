"""What the lines of play cost: search_depth against search_depth_line, and search_value against search_value_line.

    python tools/time_search_line.py [--reps 5] [--out results.json]

Workloads are those of tools/time_search.py (Zeillinger's host, reposition on, max_depth 64, node budget 2^16 per
root, capacity 2^24 states; 65 536 roots of (5, 3) in [0, 10] and 16 384 of (10, 3) in [0, 20]) and of
tools/time_search_value.py (reposition on, max_depth 8, node budget 2^14, capacity 2^26, history 2^29; 16 384 roots of
(5, 3) in [0, 10] and 4 096 of (10, 3) in [0, 20]), after the Newton filter.  The depth line gets a history of 2^28
states, more than these trees hold, so its shared outputs must equal search_depth's.  Each pair of calls runs in the
same process, alternated, with its workspaces allocated once; times are CUDA events around whole calls (each call ends
in a device synchronise), medians of the repeats.  The shared outputs of the two calls must be equal.  The card's name
and power limit are read in the same run.
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


def roots_of(B, N, d, max_value):
    g = torch.Generator(device="cuda").manual_seed(B + N)
    pts = torch.randint(0, max_value + 1, (B, N, d), generator=g, device="cuda", dtype=torch.int32)
    return hb.GameBatch(pts, semantics="jax", reposition=True, initial_filter=True).points


def compare(name, base, line, shared, reps, extra):
    a, b = base(), line()  # warm-up, and the equality of the shared outputs
    same = all(torch.equal(x, y) for x, y in zip(a, b[:shared]))
    t_base, t_line = [], []
    for _ in range(reps):  # alternated
        t_base.append(timed(base)[0])
        t_line.append(timed(line)[0])
    mb, ml = float(np.median(t_base)), float(np.median(t_line))
    status = b[shared - 1].cpu().numpy()
    length = b[0].cpu().numpy()
    return dict(extra, workload=name, same_outputs=bool(same), status_counts=np.bincount(status, minlength=6).tolist(),
                created=int(b[shared - 2].sum().item() - len(status)), line_len_max=int(length.max()),
                base_ms=t_base, line_ms=t_line, base_ms_median=mb, line_ms_median=ml, overhead=ml / mb - 1)


def run_depth(name, B, N, d, mv, reps, max_depth=64, max_nodes=1 << 16, capacity=1 << 24, history=1 << 28):
    roots = roots_of(B, N, d, mv)
    ws = torch.empty(ops.search_workspace_bytes(B, N, d, capacity), dtype=torch.uint8, device="cuda")
    wl = torch.empty(ops.search_depth_line_workspace_bytes(B, N, d, capacity, history), dtype=torch.uint8, device="cuda")
    args = dict(flags=C.HK_F_HOST_ZEILLINGER, ops=OPS, max_depth=max_depth, max_nodes=max_nodes, capacity=capacity)

    def base():
        return ops.search_depth(roots, workspace=ws, **args)

    def line():
        return ops.search_depth_line(roots, history=history, workspace=wl, **args)
    return compare(name, base, line, 3, reps, dict(search="depth", roots=B, N=N, d=d, max_value=mv, max_depth=max_depth,
                                                     max_nodes=max_nodes, capacity=capacity, history=history))


def run_value(name, B, N, d, mv, reps, max_depth=8, max_nodes=1 << 14, capacity=1 << 26, history=1 << 29):
    roots = roots_of(B, N, d, mv)
    ws = torch.empty(ops.search_value_workspace_bytes(B, N, d, capacity, history), dtype=torch.uint8, device="cuda")
    args = dict(ops=OPS, max_depth=max_depth, max_nodes=max_nodes, capacity=capacity, history=history, workspace=ws)

    def base():
        return ops.search_value(roots, **args)

    def line():
        return ops.search_value_line(roots, **args)
    return compare(name, base, line, 4, reps, dict(search="value", roots=B, N=N, d=d, max_value=mv, max_depth=max_depth,
                                                     max_nodes=max_nodes, capacity=capacity, history=history))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write every result, repeats included, to this JSON file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "time_search_line.py measures on the GPU"
    res = {"gpu": gpu_facts(), "runs": []}
    t0 = time.time()
    for fn, name, B, N, d, mv in [(run_depth, "65536 x (5,3) max 10", 65536, 5, 3, 10),
                                  (run_depth, "16384 x (10,3) max 20", 16384, 10, 3, 20),
                                  (run_value, "16384 x (5,3) max 10", 16384, 5, 3, 10),
                                  (run_value, "4096 x (10,3) max 20", 4096, 10, 3, 20)]:
        r = fn(name, B, N, d, mv, a.reps)
        res["runs"].append(r)
        print(json.dumps({k: v for k, v in r.items() if k not in ("base_ms", "line_ms")}), flush=True)
    res["wall_s"] = time.time() - t0
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
