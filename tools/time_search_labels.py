"""What the value labels cost: search_value against search_value_labels, with and without the state replay.

    python tools/time_search_labels.py [--reps 7] [--out results.json]

Workloads are those of tools/time_search_value.py (reposition on, max_depth 8, node budget 2^14, capacity 2^26,
history 2^29; 16 384 roots of (5, 3) in [0, 10] and 4 096 of (10, 3) in [0, 20]), after the Newton filter, with
max_labels 2^24, more labels than these searches find.  Three calls per workload run in the same process, alternated:
ops.search_value and ops.search_value_labels with their workspaces allocated once, and hironaka_b200.search_value_labels,
which adds the replay of the labels' rows (one ops.step per level) and takes its workspace from torch's caching
allocator.  Times are CUDA events around whole calls (each ends in a device synchronise), medians of the repeats.  The
shared outputs of the calls must be equal.  The run prints the label count, the histogram of label values and of
their levels, the labels under roots that did not resolve, and the card's name and power limit.
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


def run(name, B, N, d, mv, reps, max_depth=8, max_nodes=1 << 14, capacity=1 << 26, history=1 << 29,
        max_labels=1 << 24):
    roots = roots_of(B, N, d, mv)
    ws = torch.empty(ops.search_value_workspace_bytes(B, N, d, capacity, history), dtype=torch.uint8, device="cuda")
    wl = torch.empty(ops.search_value_labels_workspace_bytes(B, N, d, capacity, history), dtype=torch.uint8,
                     device="cuda")
    args = dict(max_depth=max_depth, max_nodes=max_nodes, capacity=capacity, history=history)

    def base():
        return ops.search_value(roots, ops=OPS, workspace=ws, **args)

    def labels():
        return ops.search_value_labels(roots, ops=OPS, max_labels=max_labels, workspace=wl, **args)

    def replay():
        return hb.search_value_labels(roots, max_labels=max_labels, **args)
    a, b, c = base(), labels(), replay()  # warm-up, and the equality of the shared outputs
    same = (all(torch.equal(x, y) for x, y in zip(a, b[:4])) and all(torch.equal(x, y) for x, y in zip(a, c[:4])) and
            b[4] == c.count and all(torch.equal(x, y) for x, y in zip(b[5:8], (c.root, c.level, c.label_value))))
    t = {"base": [], "labels": [], "replay": []}
    for _ in range(reps):  # alternated
        t["base"].append(timed(base)[0])
        t["labels"].append(timed(labels)[0])
        t["replay"].append(timed(replay)[0])
    med = {k: float(np.median(v)) for k, v in t.items()}
    status = a[3].cpu().numpy()
    lv, level, root = c.label_value.cpu().numpy(), c.level.cpu().numpy(), c.root.cpu().numpy()
    return dict(workload=name, roots=B, N=N, d=d, max_value=mv, max_depth=max_depth, max_nodes=max_nodes,
                capacity=capacity, history=history, max_labels=max_labels, same_outputs=bool(same),
                status_counts=np.bincount(status, minlength=6).tolist(),
                history_used=int(a[2].sum().item()), labels=int(c.count),
                label_values=np.bincount(lv).tolist(), label_levels=np.bincount(level).tolist(),
                labels_unresolved_roots=int((status[root] != C.HK_SEARCH_RESOLVED).sum()),
                base_ms_median=med["base"], labels_ms_median=med["labels"], replay_ms_median=med["replay"],
                overhead_labels=med["labels"] / med["base"] - 1, overhead_replay=med["replay"] / med["base"] - 1,
                ms=t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None, help="also write every result, repeats included, to this JSON file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "time_search_labels.py measures on the GPU"
    res = {"gpu": gpu_facts(), "runs": []}
    t0 = time.time()
    for name, B, N, d, mv in [("16384 x (5,3) max 10", 16384, 5, 3, 10), ("4096 x (10,3) max 20", 4096, 10, 3, 20)]:
        r = run(name, B, N, d, mv, a.reps)
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
