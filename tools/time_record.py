"""Recorded rollouts against the same data from the per-step entry points, on one GPU.

    python tools/time_record.py [reps]

Workloads: C2 (1 Mi games of (20, 3)) and C5 (256 Ki games of (64, 5)), root states filtered as the bench does, one
20-step random-vs-random rollout of the JAX flavour.  Three arms, alternated within every repeat, device time from CUDA
events around the arm alone (the state is restored outside the events; every state is larger than L2):
  (a) hk_rollout_seeded, no per-step outputs;
  (b) hk_rollout_record: obs_t (lex order, rescaled), the played host masks and axes, done_t and reward_t;
  (c) the same data from one launch per step: hk_random_actions, hk_features of the root, then one fused
      step + observation per step (hk_step_census_obs on the thread-per-game shapes, hk_step otherwise).
Prints the GPU name and power limit, the median ms per rollout of each arm, and obs bytes / time as a fraction of the
copy bandwidth bench.py reports against (measured_peak: MEASURED_PEAKS.json, or its stated fallback).
"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import measured_peak  # noqa: E402
from hironaka_b200 import constants as C  # noqa: E402
from hironaka_b200._lib import check, lib  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 7
T = 20
SEED = 12345
OPS = C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON
PLAYERS = C.HK_F_HOST_RANDOM | C.HK_F_AGENT_RANDOM
OBS = C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def workload(name, B, N, d):
    L = lib()
    dev = torch.device("cuda")
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(3)
    root = torch.from_numpy(rng.integers(0, 20, size=(B, N, d), dtype=np.int32)).to(dev)
    check(L.hk_step(root.data_ptr(), root.data_ptr(), None, None, None, None, None, None, None, None, B, N, d,
                    C.HK_DTYPE_I32, C.HK_OP_NEWTON | C.HK_OP_REPOSITION, 0, -1.0, 1e8, st), "root filter")
    x = root.clone()
    OW = N * d
    obs = torch.empty((T, B, OW), dtype=torch.float32, device=dev)
    hm = torch.empty((T, B), dtype=torch.int32, device=dev)
    axp = torch.empty((T, B), dtype=torch.int32, device=dev)
    done = torch.empty((T, B), dtype=torch.uint8, device=dev)
    reward = torch.empty((T, B), dtype=torch.float32, device=dev)
    census = torch.empty(L.hk_census_bytes(B, N, d), dtype=torch.uint8, device=dev)
    small = L.hk_kernel_class(N, d) == 1

    def arm_a():
        check(L.hk_rollout_seeded(x.data_ptr(), x.data_ptr(), None, None, None, None, None, None, B, N, d, T, C.HK_DTYPE_I32,
                                  OPS, PLAYERS, -1.0, SEED, 0, st), "hk_rollout_seeded")

    def arm_b():
        check(L.hk_rollout_record(x.data_ptr(), x.data_ptr(), None, None, obs.data_ptr(), 0, hm.data_ptr(), axp.data_ptr(),
                                  done.data_ptr(), reward.data_ptr(), None, None, B, N, d, T, C.HK_DTYPE_I32, OPS,
                                  PLAYERS | OBS, -1.0, SEED, 0, st), "hk_rollout_record")

    def arm_c():
        census.zero_()
        check(L.hk_random_actions(hm.data_ptr(), axp.data_ptr(), B, d, T, SEED, 0, st), "hk_random_actions")
        check(L.hk_features(x.data_ptr(), obs[0].data_ptr(), None, B, N, d, C.HK_DTYPE_I32, OBS, -1.0, st), "hk_features")
        for t in range(T):
            o = obs[t + 1].data_ptr() if t + 1 < T else None
            args = (hm[t].data_ptr(), axp[t].data_ptr(), done[t].data_ptr())
            if small:
                rc = L.hk_step_census_obs(x.data_ptr(), *args, None, reward[t].data_ptr(), None, o, None, census.data_ptr(),
                                          None, None, B, N, d, C.HK_DTYPE_I32, OPS, C.HK_F_ACT_DISCRETE | OBS, -1.0, 1e8, st)
            else:
                rc = L.hk_step(x.data_ptr(), x.data_ptr(), *args, reward[t].data_ptr(), None, o, None, None, B, N, d,
                               C.HK_DTYPE_I32, OPS, C.HK_F_ACT_DISCRETE | OBS, -1.0, 1e8, st)
            check(rc, "per-step arm")

    arms = {"a": arm_a, "b": arm_b, "c": arm_c}
    times = {k: [] for k in arms}
    for rep in range(REPS + 1):  # the first round warms every arm up and is not counted
        for k in (("a", "b", "c") if rep % 2 == 0 else ("c", "b", "a")):
            x.copy_(root)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            arms[k]()
            e1.record()
            torch.cuda.synchronize()
            if rep > 0:
                times[k].append(e0.elapsed_time(e1))
    peak, peak_src = measured_peak()
    obs_bytes = T * B * OW * 4
    print(f"{name}: {B} games of ({N}, {d}), {T} random-play steps (JAX flavour); obs {obs_bytes / 1e9:.2f} GB per rollout")
    for k, label in (("a", "hk_rollout_seeded, no outputs"), ("b", "hk_rollout_record"), ("c", "per-step launches")):
        ms = float(np.median(times[k]))
        frac = (obs_bytes / (ms * 1e-3)) / (peak * 1e9) if k != "a" else None
        print(f"  ({k}) {label:32s} {ms:8.3f} ms  (min {min(times[k]):.3f}, max {max(times[k]):.3f})" +
              (f"  obs {obs_bytes / (ms * 1e-3) / 1e12:.2f} TB/s = {frac:.2f} of {peak / 1e3:.2f} TB/s" if frac else ""))
    print(f"  copy bandwidth: {peak_src}")


if __name__ == "__main__":
    if not torch.cuda.is_available():
        sys.exit("time_record.py measures on a CUDA device; none is visible")
    print("GPU:", gpu_info())
    workload("C2", 1 << 20, 20, 3)
    workload("C5", 1 << 18, 64, 5)
