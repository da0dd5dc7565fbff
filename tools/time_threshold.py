"""Rollouts with a value threshold against the plain seeded rollout, on one GPU.

    python tools/time_threshold.py [--baseline LIB] [--reps R]

Workloads: C2 (1 Mi games of (20, 3)) and C5 (256 Ki games of (64, 5)), root states filtered as the bench does, one
20-step random-vs-random rollout of the JAX flavour, no per-step outputs.  Arms, alternated within every repeat, device
time from CUDA events around the arm alone (the state is restored outside the events; every state is larger than L2):
  (base) hk_rollout_seeded of LIB, a build of the parent commit (--baseline; skipped without it);
  (a)    hk_rollout_seeded of this build;
  (b)    hk_rollout_threshold, value_threshold 1e8 (the reference's default), no stop, over_step written;
  (c)    hk_rollout_threshold with a threshold low enough that games stop (30), over_step written.
Prints the GPU name and power limit, the median ms per rollout of each arm (min, max), the overhead of (b) and (c) over
(a), the share of games stopped in (c), and whether (base), (a) and (b) leave the same state.
"""
import argparse
import ctypes
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hironaka_b200 import constants as C  # noqa: E402
from hironaka_b200._lib import SIGNATURES, check, lib  # noqa: E402

T = 20
SEED = 12345
OPS = C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON
PLAYERS = C.HK_F_HOST_RANDOM | C.HK_F_AGENT_RANDOM
LOW = 30.0


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def load_baseline(path):
    L = ctypes.CDLL(os.path.abspath(path))
    res, args = SIGNATURES["hk_rollout_seeded"]
    L.hk_rollout_seeded.restype = res
    L.hk_rollout_seeded.argtypes = args
    return L


def workload(name, B, N, d, base, reps):
    L = lib()
    dev = torch.device("cuda")
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(3)
    root = torch.from_numpy(rng.integers(0, 20, size=(B, N, d), dtype=np.int32)).to(dev)
    check(L.hk_step(root.data_ptr(), root.data_ptr(), None, None, None, None, None, None, None, None, B, N, d,
                    C.HK_DTYPE_I32, C.HK_OP_NEWTON | C.HK_OP_REPOSITION, 0, -1.0, 1e8, st), "root filter")
    x = root.clone()
    over = torch.empty(B, dtype=torch.int32, device=dev)

    def seeded(lb):
        def arm():
            check(lb.hk_rollout_seeded(x.data_ptr(), x.data_ptr(), None, None, None, None, None, None, B, N, d, T,
                                       C.HK_DTYPE_I32, OPS, PLAYERS, -1.0, SEED, 0, st), "hk_rollout_seeded")
        return arm

    def threshold(thr, stop):
        def arm():
            check(L.hk_rollout_threshold(x.data_ptr(), x.data_ptr(), None, None, None, 0, None, None, None, None, None, None,
                                         B, N, d, T, C.HK_DTYPE_I32, OPS, PLAYERS, -1.0, SEED, 0, thr, stop,
                                         over.data_ptr(), st), "hk_rollout_threshold")
        return arm

    arms = {"a": seeded(L), "b": threshold(1e8, 0), "c": threshold(LOW, 1)}
    if base is not None:
        arms["base"] = seeded(base)
    order = list(arms)
    times = {k: [] for k in arms}
    finals = {}
    for rep in range(reps + 1):  # the first round warms every arm up and is not counted
        for k in (order if rep % 2 == 0 else order[::-1]):
            x.copy_(root)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            arms[k]()
            e1.record()
            torch.cuda.synchronize()
            if rep > 0:
                times[k].append(e0.elapsed_time(e1))
            else:
                finals[k] = x.clone()
                if k == "c":
                    stopped = float((over <= T).float().mean())
    print(f"{name}: {B} games of ({N}, {d}), {T} random-play steps (JAX flavour), {reps} alternated repeats")
    med = {k: float(np.median(v)) for k, v in times.items()}
    labels = {"base": "hk_rollout_seeded, parent build", "a": "hk_rollout_seeded", "b": "threshold 1e8, no stop",
              "c": f"threshold {LOW:g}, stop"}
    for k in order:
        extra = f"  {100 * (med[k] / med['a'] - 1):+.1f} % vs (a)" if k in ("b", "c", "base") else ""
        print(f"  ({k}) {labels[k]:34s} {med[k]:8.3f} ms  (min {min(times[k]):.3f}, max {max(times[k]):.3f}){extra}")
    print(f"  (c) stopped {100 * stopped:.1f} % of the games")
    same = [k for k in ("base", "b") if k in finals and torch.equal(finals[k], finals["a"])]
    print(f"  same final state as (a): {', '.join(same) if same else 'none'}")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline", default=None, help="libhironaka_b200.so built from the parent commit")
    ap.add_argument("--reps", type=int, default=15)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_threshold.py measures on a CUDA device; none is visible")
    print("GPU:", gpu_info())
    base = load_baseline(a.baseline) if a.baseline else None
    workload("C2", 1 << 20, 20, 3, base, a.reps)
    workload("C5", 1 << 18, 64, 5, base, a.reps)
