#!/usr/bin/env python
"""bench.py — game-steps/sec of the batched Hironaka env step on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this engine
    python bench.py ... --dump-outputs DIR                          # also write the last timed step's outputs
    python bench.py --impl reference [--gpus N] [--steps K] ...     # CPU arm: the unmodified reference (baseline/_ref)
    torchrun --nproc-per-node N ... bench.py --gpus N ...           # one rank per GPU

Workload (config.workload = "C2"): BASELINE.json configs[1] — dim=3, max_num_points=20
random-play rollout (SURVEY.md section 8d): root states randint[0,20) -> newton -> reposition,
then per step a uniform random host action id and a uniform random agent axis over ALL d axes
(invalid actions occur; JAX semantics apply them), step = shift -> reposition -> newton ->
done/reward.  All inputs are generated on the CPU from a seed and copied (never device RNG).
1 Mi games per GPU (weak scaling; the state, 252 MB, exceeds the 126 MB L2, so every step
streams from HBM).  A "step" is one game-step of all B slots = one launch of the in-place step with a
census (hk_step_census: games at rest are answered from their census byte, games in play are ordered by
live count); consecutive steps walk through independent 20-step rollouts, each on its own pre-generated
batch, so the live-point dynamics are those of real play and nothing but steps sits in the timed region.

One JSON line on stdout (rank 0).  See DESIGN.md section "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "game_steps_per_sec"
UNIT = "game-steps/s"
N_POINTS, DIM, T_ROLLOUT, MAX_VALUE = 20, 3, 20, 20
GAMES_PER_GPU = 1 << 20
CPU_SAMPLE_GAMES = int(os.environ.get("HK_BENCH_CPU_SAMPLE", 1 << 19))  # bounded sample of the C2 workload for the C port (state 126 MB, ~1 s per 40 steps)
REF_SAMPLE_GAMES = int(os.environ.get("HK_BENCH_REF_SAMPLE", 1 << 14))  # games per step of the real reference (its [B,N,N,d] temporaries: 79 MB each)
MAX_RESIDENT_ROLLOUTS = 10  # distinct pre-generated batches; beyond K = 200 they are restored from pristine copies
DUMP_SAMPLE_GAMES = 1 << 17  # games whose state --dump-outputs writes (31.5 MB of float32)
BYTES_PER_GAME_STEP = 8 * N_POINTS * DIM + 13  # SURVEY.md 8(d): int32 state r+w, 2 x int32 action, u8 done, f32 reward
OPS_PER_GAME_STEP = N_POINTS * (N_POINTS - 1) * (DIM + 1) + 3 * N_POINTS * DIM + N_POINTS


def workload_config(n_gpus: int) -> dict:
    return {
        "workload": "C2: test/jax_config.yml shape (dim=3, max_num_points=20) random-play rollout, "
                    "random host vs random agent, JAX semantics with reposition",
        "games_per_gpu": GAMES_PER_GPU, "global_batch": GAMES_PER_GPU * n_gpus, "max_num_points": N_POINTS,
        "dimension": DIM, "rollout_length": T_ROLLOUT, "max_value": MAX_VALUE,
        "parallelism": f"batch-sharded x{n_gpus}, no collective on the step path",
        "l2_policy": "inputs larger than L2 (252 MB int32 state per GPU vs 126 MB L2); a new batch every 20 steps",
        "bytes_per_game_step": BYTES_PER_GAME_STEP, "int_ops_per_game_step": OPS_PER_GAME_STEP,
    }


def make_inputs(seed: int, B: int, n_rollouts: int):
    """Seeded CPU inputs: raw root points [R,B,N,d] int32 and action streams [R,T,B] int32."""
    rng = np.random.default_rng(seed)
    ncls = 2 ** DIM - DIM - 1
    pts = rng.integers(0, MAX_VALUE, size=(n_rollouts, B, N_POINTS, DIM), dtype=np.int32)
    ha = rng.integers(0, ncls, size=(n_rollouts, T_ROLLOUT, B), dtype=np.int32)
    ax = rng.integers(0, DIM, size=(n_rollouts, T_ROLLOUT, B), dtype=np.int32)
    return pts, ha, ax


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_per_launch():
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            return json.load(f).get("hk_sched_kernel_i32_20x3_bytes_per_launch_1Mi")
    except Exception:
        return None


# ---------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Polls NVML (SM clock + throttle reasons) from a thread while the timed region runs."""

    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int, uuid: str | None = None):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if uuid and not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for b, name in self.REASONS.items():
                    if bits & b and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self) -> dict:
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------- CPU arm
def cpu_rate(sample_games: int, steps: int, warmup: int, seed: int = 1234, threads: int | None = None):
    """Times the oracle's C port (all host threads) on a bounded sample of the same workload.
    This is the only place the bench executes oracle/ — as the measured CPU baseline."""
    from oracle import cport
    from oracle import hk_oracle as O
    if threads:
        cport.set_threads(threads)
    cores = cport.threads()
    n_roll = max(1, -(-(steps + warmup) // T_ROLLOUT))
    pts, ha, ax = make_inputs(seed, sample_games, n_roll)
    ops_step = O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON
    states = [cport.step(pts[r], None, None, O.OP_NEWTON | O.OP_REPOSITION, 0)[0] for r in range(n_roll)]
    out = np.empty_like(states[0])
    k = 0
    t0 = None
    for i in range(warmup + steps):
        if i == warmup:
            t0 = time.perf_counter()
        r, t = divmod(k, T_ROLLOUT)
        r %= n_roll
        cport.step(states[r], ha[r, t], ax[r, t], ops_step, O.F_ACT_DISCRETE, out=out)
        states[r], out = out, states[r]
        k += 1
    dt = time.perf_counter() - t0
    return sample_games * steps / dt, cores, dt


def reference_style_rate(games: int = 4096, steps: int = 10, seed: int = 77):
    """The NumPy restatement that keeps the reference's own algorithm shape — materialised
    [B,N,N,d] difference tensors per op, one array op per reference line (oracle/hk_oracle.py) —
    timed on one host thread.  Context for the C port's number: this is what the reference's
    array-library formulation costs on a CPU (BASELINE.md section 2 measured 7.6e4-9.1e4
    game-steps/s for the real torch reference on 8 threads)."""
    from oracle import hk_oracle as O
    rng = np.random.default_rng(seed)
    x = O.generate_pts(rng, (games, N_POINTS, DIM), MAX_VALUE, rescale=False, reposition=True)
    ncls = 2 ** DIM - DIM - 1
    t0 = time.perf_counter()
    for _ in range(steps):
        x, *_ = O.step(x, rng.integers(0, ncls, games), rng.integers(0, DIM, games),
                       O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, O.F_ACT_DISCRETE)
    return games * steps / (time.perf_counter() - t0)


def reference_baseline(steps: int, warmup: int):
    """The unmodified reference (baseline/_ref, hironaka.core.TensorPoints over hironaka/src/_torch_ops.py) on a
    bounded sample of the C2 workload, all host threads.  Returns the cpu_baseline dict, or None when
    baseline/_ref did not travel."""
    from baseline import reference_arm as R
    if not R.available():
        return None
    rate, cores, threads, dt = R.rate(make_inputs, REF_SAMPLE_GAMES, steps, warmup, T_ROLLOUT)
    return {"value": rate, "unit": UNIT, "cores": cores, "torch_threads": threads, "kind": "reference",
            "seconds": dt,
            "sample": f"{REF_SAMPLE_GAMES} games x {steps} steps of the C2 workload through the UNMODIFIED reference "
                      f"(honglu2875/hironaka 0.0.1 in baseline/_ref): HostActionEncoder.decode_tensor -> TensorPoints.shift "
                      f"-> reposition -> get_newton_polytope -> ended_batch_in_tensor -> reward, torch on {threads} threads of "
                      f"{cores} cores, time.perf_counter (the reference's Timer).  The reference's JAX step cannot be timed: "
                      f"jax is not installed in this image"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cpu = reference_baseline(args.steps, args.warmup)
    if cpu is None:  # baseline/_ref did not travel: the oracle's C port stands in (kind "port")
        rate, cores, dt = cpu_rate(CPU_SAMPLE_GAMES, args.steps, args.warmup)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "seconds": dt,
               "sample": f"{CPU_SAMPLE_GAMES} games x {args.steps} steps of the C2 workload, oracle/hk_oracle.c over "
                         f"{cores} pthreads (baseline/_ref is missing)"}
    rate, dt = cpu["value"], cpu["seconds"]
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "float32" if cpu["kind"] == "reference" else "int32", "data": "synthetic",
        "config": workload_config(args.gpus), "cpu_baseline": cpu,
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------- GPU arm
def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    import hironaka_b200 as hb
    from hironaka_b200 import GameBatch, constants as C, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the engine has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    B, K, W = GAMES_PER_GPU, args.steps, args.warmup
    n_roll = min(-(-K // T_ROLLOUT), MAX_RESIDENT_ROLLOUTS)
    n_warm = 1
    pts, ha, ax = make_inputs(1000 + rank, B, n_roll + n_warm)
    op_step = C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON
    flags = C.HK_F_ACT_DISCRETE
    # resident inputs: filtered root states (generate_pts: newton -> reposition) and action streams
    batches = []
    for r in range(n_roll + n_warm):
        gb = GameBatch(torch.from_numpy(pts[r]).to(dev), semantics="jax", reposition=True, initial_filter=True)
        batches.append(gb)
    wraps = K > n_roll * T_ROLLOUT
    pristine = [(b.points.clone(), b.census.clone()) for b in batches[:n_roll]] if wraps else None
    ha_d = torch.from_numpy(ha).to(dev)
    ax_d = torch.from_numpy(ax).to(dev)
    done = torch.empty(B, dtype=torch.uint8, device=dev)
    reward = torch.empty(B, dtype=torch.float32, device=dev)
    lib = hb._lib.lib()
    if args.no_pdl:
        lib.hk_debug_set_pdl(0)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def launch_step(r, t):
        st = batches[r].points
        rc = lib.hk_step_census(st.data_ptr(), ha_d[r, t].data_ptr(), ax_d[r, t].data_ptr(), done.data_ptr(), None,
                                reward.data_ptr(), None, batches[r].census.data_ptr(), None, None, B, N_POINTS, DIM,
                                C.HK_DTYPE_I32, op_step, flags, -1.0, 1e8, stream)
        if rc != 0:
            raise RuntimeError(f"hk_step_census failed: {rc}")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank, uuid=str(torch.cuda.get_device_properties(dev).uuid))
    # ---- warm-up (untimed) ----
    for i in range(max(W, 3)):
        r, t = divmod(i, T_ROLLOUT)
        launch_step(n_roll + (r % n_warm), t)
    barrier()
    # ---- timed region: EXACTLY K steps, device-timed on the launching stream ----
    sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    barrier()
    # Gate: the device spins for a moment while the host enqueues the K launches behind it, so that the timed
    # region (events on the launching stream, after the gate) holds K back-to-back steps and no host launch gap
    # (the first launch after a barrier + synchronize used to cost 0.1-0.15 ms more than the others).
    torch.cuda._sleep(int(min(K, 400) * 60000 + 400000))
    ev[0].record()
    for i in range(K):
        r, t = divmod(i, T_ROLLOUT)
        if r >= n_roll:  # K > 200: reuse a batch; its restore (two D2D copies) is charged to the timed region
            r %= n_roll
            if t == 0:
                batches[r].points.copy_(pristine[r][0])
                batches[r].census.copy_(pristine[r][1])
        launch_step(r, t)
        ev[i + 1].record()
    barrier()
    total_ms = ev[0].elapsed_time(ev[K])
    per_launch_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(K)]
    # what the last timed step returned (batch r), read back before the launches below overwrite done / reward
    outputs = last_step_outputs(torch, batches[r].points, done, reward) if args.dump_outputs and rank == 0 else None
    # keep the device busy a little longer so that NVML has samples under load
    t_end = time.perf_counter() + 0.4
    i = 0
    while time.perf_counter() < t_end:
        launch_step(n_roll + (i % n_warm), i % T_ROLLOUT)
        i += 1
        if i % 64 == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    clocks = sampler.stop()

    if world > 1:
        tmax = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        total_ms_max = float(tmax.item())
    else:
        total_ms_max = total_ms
    value = B * world * K / (total_ms_max * 1e-3)

    # ---- end-to-end through the public API with HOST buffers (pinned), copies inside the timed region ----
    e2e = None if args.no_e2e else measure_e2e(torch, dev, B, K, pts, ha, ax, n_roll, barrier, world, dist)
    collective = None
    if world > 1 and not args.no_collective:
        try:
            collective = measure_collective(torch, dist, lib, C, dev, world, rank)
        except Exception as e:
            collective = {"error": repr(e)}
    secondary = None
    if rank == 0 and world == 1 and not args.no_secondary:
        try:
            secondary = measure_secondary(torch, lib, C, dev)
        except Exception as e:  # context numbers must never take the headline down
            secondary = {"error": repr(e)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peak, peak_src = measured_peak()
    avg_launch_s = float(np.mean(per_launch_ms)) * 1e-3
    achieved = B * BYTES_PER_GAME_STEP / avg_launch_s / 1e9
    traffic = traffic_per_launch()
    roofline = {
        "bound": "hbm", "kernel": "hk::hk_sched_kernel<int,20,3>", "achieved": achieved, "peak": peak,
        "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
        # `achieved` uses SURVEY 8d's algorithmic bytes (every game read AND written every step).  The census step
        # neither reads the games at rest nor writes back unchanged games, so the bytes that really move
        # (`traffic`, ncu, mean over a rollout) are far fewer and `frac` exceeds 1; `physical` is the same launch
        # counted in moved bytes, and secondary.C2_write_back.store_all is the tile-ring kernel made to read and
        # write every game (HK_F_STORE_ALL), the like-for-like number for the algorithmic byte model.
        "physical": None if not traffic else {"bytes_per_launch": traffic, "gbps": traffic / avg_launch_s / 1e9,
                                              "frac": traffic / avg_launch_s / 1e9 / peak},
        "store_all_frac": None if not secondary or "store_all" not in secondary.get("C2_write_back", {}) else
        secondary["C2_write_back"]["store_all"]["hbm_frac_algorithmic"],
        "algorithmic_bytes_per_launch": B * BYTES_PER_GAME_STEP, "avg_launch_ms": avg_launch_s * 1e3,
        "min_launch_ms": float(np.min(per_launch_ms)), "max_launch_ms": float(np.max(per_launch_ms)),
        # Instruction issue, from EXECUTED instructions (ncu smsp__inst_executed.sum of the committed capture of this
        # kernel on this workload, mean over the 20 launches of a rollout) over the live launch time, against the
        # measured INT32 issue peak (profiles/int32_peak.json, lane-ops / 32).  The dense op count of SURVEY 8d is not
        # used: the kernel visits live rows of games in play only.
        "issue": executed_issue(avg_launch_s),
        # mean launch time by position in the 20-step rollout (live points thin out as play goes on)
        "launch_ms_by_rollout_step": [round(float(np.mean(per_launch_ms[t::T_ROLLOUT])), 5)
                                      for t in range(min(T_ROLLOUT, K))],
    }
    cpu = None
    if not args.no_cpu and world == 1:
        try:
            rate, cores, dt = cpu_rate(CPU_SAMPLE_GAMES, 80, 5)
            port = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                    "sample": f"{CPU_SAMPLE_GAMES} games x 80 steps of the C2 workload in {dt:.2f} s, oracle/hk_oracle.c "
                              f"(C port of the reference step) over {cores} pthreads"}
            cpu = reference_baseline(40, 2)  # ~10-30 s of the real reference
            if cpu is None:
                cpu = dict(port)
            cpu["port"] = port
        except Exception as e:  # the CPU baseline must never take the GPU line down
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(W, 3),
        "ms_per_step": total_ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic", "config": workload_config(world), "roofline": roofline,
        "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": K, "clocks": clocks,
        "library": os.path.relpath(hb.LIB_PATH, ROOT), "collective": collective, "secondary": secondary,
    }
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def last_step_outputs(torch, points, done, reward) -> dict:
    """What a caller of the timed step receives, as float32 host arrays for --dump-outputs: the per-game done
    flags and rewards in full, and the new state of a fixed, seeded sample of DUMP_SAMPLE_GAMES games with their
    indices (the whole state, 252 MB, exceeds the 64 MB a dump may take)."""
    games = np.sort(np.random.default_rng(0).choice(points.shape[0], DUMP_SAMPLE_GAMES, replace=False))
    sample = points.index_select(0, torch.from_numpy(games).to(points.device))
    out = {"points": sample.cpu().numpy().astype(np.float32), "points_games": games.astype(np.float64),
           "done": done.cpu().numpy().astype(np.float32), "reward": reward.cpu().numpy().astype(np.float32)}
    assert sum(a.nbytes for a in out.values()) <= 64_000_000
    return out


def executed_issue(avg_launch_s):
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            per = json.load(f)["instructions_per_launch_M"]
        inst = float(np.mean(per)) * 1e6
    except Exception:
        return None
    peak = int32_peak()[0] / 32.0
    return {"executed_warp_instructions_per_launch": inst, "achieved_per_s": inst / avg_launch_s, "peak_per_s": peak,
            "frac": inst / avg_launch_s / peak, "source": "profiles/r2c_step_census_ncu_full_summary.csv"}


def int32_peak():
    try:
        with open(os.path.join(ROOT, "profiles", "int32_peak.json")) as f:
            return float(json.load(f)["int32_peak_ops"]), "measured (profiles/int32_peak.json, tools/int32_peak.cu)"
    except Exception:
        return 148 * 128 * 1.965e9, "nominal 148 SM x 128 lanes x 1.965 GHz"


def measure_secondary(torch, lib, C, dev):
    """The other BASELINE.json configs, device-timed with CUDA events (rank 0, N = 1 only).
    They are parity-test cases first (tests/test_gpu_parity.py::test_baseline_sizes_bit_exact);
    the numbers here are context for DESIGN.md, not the headline."""
    stream = torch.cuda.current_stream(dev).cuda_stream
    peak_hbm, _ = measured_peak()
    peak_int, int_src = int32_peak()
    out = {}

    def timed(fn, n, warm=3):
        for _ in range(warm):
            fn(0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n  # ms per call

    def make(B, N, d, T, mv, seed, reposition):
        rng = np.random.default_rng(seed)
        ncls = 2 ** d - d - 1
        x = torch.from_numpy(rng.integers(0, mv, size=(B, N, d), dtype=np.int32)).to(dev)
        ha = torch.from_numpy(rng.integers(0, ncls, size=(T, B), dtype=np.int32)).to(dev)
        ax = torch.from_numpy(rng.integers(0, d, size=(T, B), dtype=np.int32)).to(dev)
        init = C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)
        rc = lib.hk_step(x.data_ptr(), x.data_ptr(), None, None, None, None, None, None, None, None, B, N, d,
                         C.HK_DTYPE_I32, init, 0, -1.0, 1e8, stream)
        assert rc == 0, rc
        return x, ha, ax

    def step_fn(x, ha, ax, B, N, d, T, ops_bits, flags, done, reward, pristine=None):
        def fn(i):
            t = i % T
            if t == 0 and pristine is not None and i > 0:
                x.copy_(pristine)
            rc = lib.hk_step(x.data_ptr(), x.data_ptr(), ha[t].data_ptr(), ax[t].data_ptr(), done.data_ptr(),
                             reward.data_ptr(), None, None, None, None, B, N, d, C.HK_DTYPE_I32, ops_bits, flags, -1.0,
                             1e8, stream)
            if rc != 0:
                raise RuntimeError(rc)
        return fn

    # C1: TensorPoints batch=1024, dim=3, max_num_points=10, torch semantics, T=10 (launch-latency bound)
    B, N, d, T = 1024, 10, 3, 10
    x, ha, ax = make(B, N, d, T, 21, 1, False)
    done, rew = torch.empty(B, dtype=torch.uint8, device=dev), torch.empty(B, dtype=torch.float32, device=dev)
    ms = timed(step_fn(x, ha, ax, B, N, d, T, C.HK_OP_SHIFT | C.HK_OP_NEWTON, C.TORCH_SEMANTICS | C.HK_F_ACT_DISCRETE,
                       done, rew, x.clone()), 200)
    out["C1"] = {"workload": "B=1024, N=10, d=3, torch semantics, T=10", "us_per_launch": ms * 1e3,
                 "game_steps_per_s": B / (ms * 1e-3), "bound": "launch latency (1024 games = 123 KB per launch)",
                 "hbm_frac": B * (8 * N * d + 13) / (ms * 1e-3) / 1e9 / peak_hbm}

    # C4: the ADE start configurations (N=5, d=3), B=4096, FusedGame semantics + replay-buffer append
    try:
        from hironaka_b200 import ReplayBuffer, ops as hops
        ade = np.array([[[3, 0, 0], [0, 5, 0], [0, 0, 2]], [[2, 0, 0], [0, 3, 0], [0, 0, 3]], [[2, 0, 0], [0, 3, 0], [0, 0, 4]],
                        [[2, 0, 0], [0, 2, 1], [0, 0, 5]], [[2, 0, 0], [0, 2, 0], [0, 0, 4]], [[3, 0, 0], [0, 5, 0], [0, 2, 2]]],
                       dtype=np.float32)
        B, N, d, T = 4096, 5, 3, 10
        rng = np.random.default_rng(4)
        x0 = -np.ones((B, N, d), np.float32)
        x0[:, :3] = ade[rng.integers(0, 6, B)]
        xs = torch.from_numpy(x0).to(dev)
        pristine = xs.clone()
        ha = torch.from_numpy(rng.integers(0, 4, size=(T, B), dtype=np.int32)).to(dev)
        ax = torch.from_numpy(rng.integers(0, d, size=(T, B), dtype=np.int32)).to(dev)
        buf = ReplayBuffer((N, d), 4, 1 << 16, dev)
        fl = C.TORCH_SEMANTICS | C.HK_F_ACT_DISCRETE | C.HK_F_OBS_SORT_COORD0

        def dqn_step(i):
            t = i % T
            if t == 0:
                xs.copy_(pristine)
            before = hops.features(xs, flags=C.HK_F_OBS_SORT_COORD0)
            skip = hops.dones(xs)[0]
            r = hops.step(xs, ha[t], ax[t], ops=C.HK_OP_SHIFT | C.HK_OP_NEWTON, flags=fl, inplace=True, want_done=True,
                          want_reward=True, want_obs=True)
            buf.add_masked(skip, before, ha[t], r.reward, r.done, r.obs)
        ms = timed(dqn_step, 200)
        out["C4"] = {"workload": "6 ADE starts (search.py:123-128) padded to N=5, B=4096, FusedGame semantics, T=10; per step: "
                                 "features + dones + fused step with features + order-preserving replay append (6 launches, "
                                 "no host sync)", "us_per_step": ms * 1e3, "game_steps_per_s": B / (ms * 1e-3),
                     "bound": "launch latency (Python-driven, 4096 games)"}
        # the same replay-buffer generation through the FusedGame drop-in with fixed players, eager and as a CUDA graph
        from hironaka_b200 import FusedGame, TensorPoints
        from hironaka_b200.players import AllCoordHostModule, ChooseFirstAgentModule
        game = FusedGame(AllCoordHostModule(d, N, dev), ChooseFirstAgentModule(d, N, dev), device=dev)
        pts4 = TensorPoints(pristine.clone(), device=dev)
        buf2 = ReplayBuffer((N, d), 4, 1 << 16, dev)
        graph = game.graphed_step_into(buf2, pts4, "host", scale_observation=True, exploration_rate=0.2)

        def eager(i):
            if i % T == 0:
                pts4.points.copy_(pristine)
            game.step_into(buf2, pts4, "host", scale_observation=True, exploration_rate=0.2)

        def graphed(i):
            if i % T == 0:
                pts4.points.copy_(pristine)
            graph.replay()
        out["C4"]["fused_game_step_into_us"] = {"eager": timed(eager, 100) * 1e3, "cuda_graph": timed(graphed, 300) * 1e3,
                                                "note": "FusedGame.step_into with AllCoord host / ChooseFirst agent modules, "
                                                        "exploration 0.2, scale_observation: nets, noise, fused step, "
                                                        "features, order-preserving append"}
    except Exception as e:
        out["C4"] = {**out.get("C4", {}), "error": repr(e)}

    # C5: dim=5, max_num_points=64, batch 256K, T=20 — the warp-per-game kernel, ALU-bound shape
    B, N, d, T = 1 << 18, 64, 5, 20
    x, ha, ax = make(B, N, d, T, 20, 5, True)
    done, rew = torch.empty(B, dtype=torch.uint8, device=dev), torch.empty(B, dtype=torch.float32, device=dev)
    pristine = x.clone()
    fn = step_fn(x, ha, ax, B, N, d, T, C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON, C.HK_F_ACT_DISCRETE, done,
                 rew, None)
    per = []
    for rep in range(3):
        x.copy_(pristine)
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(T + 1)]
        ev[0].record()
        for t in range(T):
            fn(t)
            ev[t + 1].record()
        torch.cuda.synchronize()
        if rep:
            per.append([ev[t].elapsed_time(ev[t + 1]) for t in range(T)])
    per = np.mean(np.array(per), axis=0)
    ms = float(per.mean())
    # the same rollout through hk_step_census: the games down to <= 8 live rows are stepped thread-per-game on their
    # live rows alone (hk_rows_kernel), games at rest are skipped, the rest goes warp-per-game (two launches a step)
    census5 = torch.zeros(lib.hk_census_bytes(B, N, d), dtype=torch.uint8, device=dev)
    per_c = []
    for rep in range(3):
        x.copy_(pristine)
        census5.zero_()
        rc = lib.hk_step_census(x.data_ptr(), None, None, None, None, None, None, census5.data_ptr(), None, None, B, N, d,
                                C.HK_DTYPE_I32, C.HK_OP_NEWTON | C.HK_OP_REPOSITION, 0, -1.0, 1e8, stream)  # fills the census
        assert rc == 0
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(T + 1)]
        ev[0].record()
        for t in range(T):
            rc = lib.hk_step_census(x.data_ptr(), ha[t].data_ptr(), ax[t].data_ptr(), done.data_ptr(), None, rew.data_ptr(),
                                    None, census5.data_ptr(), None, None, B, N, d, C.HK_DTYPE_I32,
                                    C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON, C.HK_F_ACT_DISCRETE, -1.0, 1e8, stream)
            assert rc == 0
            ev[t + 1].record()
        torch.cuda.synchronize()
        if rep:
            per_c.append([ev[t].elapsed_time(ev[t + 1]) for t in range(T)])
    per_c = np.mean(np.array(per_c), axis=0)
    ms_c = float(per_c.mean())
    ops5 = N * (N - 1) * (d + 1) + 3 * N * d + N
    bytes5 = 8 * N * d + 13
    # the same kernel on the ROOT filter (64 random live points per game = the dense worst case)
    xr = torch.from_numpy(np.random.default_rng(6).integers(0, 20, size=(B, N, d), dtype=np.int32)).to(dev)
    work = xr.clone()

    def root(i):
        work.copy_(xr)
        rc = lib.hk_step(work.data_ptr(), work.data_ptr(), None, None, None, None, None, None, None, None, B, N, d,
                         C.HK_DTYPE_I32, C.HK_OP_NEWTON, 0, -1.0, 1e8, stream)
        assert rc == 0

    def copy_only(i):
        work.copy_(xr)
    ms_root = timed(root, 10) - timed(copy_only, 10)
    out["C5"] = {"workload": "B=262144, N=64, d=5, random play T=20, JAX semantics with reposition",
                 "kernel": "hk::hk_generic_kernel<int,5,false>", "ms_per_step": ms, "game_steps_per_s": B / (ms * 1e-3),
                 "ms_by_rollout_step": [round(float(v), 4) for v in per],
                 "hbm_frac": B * bytes5 / (ms * 1e-3) / 1e9 / peak_hbm,
                 "int_ops_per_game_step_dense": ops5, "int32_peak": peak_int, "int32_peak_source": int_src,
                 "census": {"api": "hk_step_census: hk_rows_kernel (games with <= 8 live rows, thread-per-game on live rows) + "
                                   "hk_generic_kernel (the rest), games at rest skipped",
                            "ms_per_step": ms_c, "game_steps_per_s": B / (ms_c * 1e-3),
                            "ms_by_rollout_step": [round(float(v), 4) for v in per_c],
                            "hbm_frac": B * bytes5 / (ms_c * 1e-3) / 1e9 / peak_hbm},
                 "root_filter_ms": ms_root, "root_filter_int_frac": B * ops5 / (ms_root * 1e-3) / peak_int,
                 "note": "root_filter_int_frac: the root filter (64 live points per game) is the one launch that executes "
                         "the dense op count of SURVEY 8d, so dense ops / time / INT32 peak is meaningful there; steps of real "
                         "play visit live rows only, and their executed-instruction counts are in "
                         "profiles/r2a_c5_census_ncu_full_summary.csv"}
    # the same 20 steps as ONE launch (hk_rollout on the warp-per-game family: compact rows stay in registers)
    try:
        dcount5 = torch.zeros(T, dtype=torch.int32, device=dev)

        def roll5(i):
            x.copy_(pristine)
            rc = lib.hk_rollout(x.data_ptr(), x.data_ptr(), ha.data_ptr(), ax.data_ptr(), None, None, dcount5.data_ptr(),
                                None, B, N, d, T, C.HK_DTYPE_I32, C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON,
                                C.HK_F_ACT_DISCRETE, -1.0, stream)
            assert rc == 0

        def copy5(i):
            x.copy_(pristine)
        ms5 = timed(roll5, 6) - timed(copy5, 6)
        out["C5"]["rollout_fused_T20"] = {"ms_per_rollout": ms5, "game_steps_per_s": B * T / (ms5 * 1e-3)}
    except Exception as e:
        out["C5"]["rollout_fused_T20"] = {"error": repr(e)}

    # C2 with HK_F_STORE_ALL: every game written back every step (what the roofline's algorithmic bytes assume)
    try:
        B, N, d, T = GAMES_PER_GPU, N_POINTS, DIM, T_ROLLOUT
        x, ha, ax = make(B, N, d, T, MAX_VALUE, 12, True)
        done, rew = torch.empty(B, dtype=torch.uint8, device=dev), torch.empty(B, dtype=torch.float32, device=dev)
        pristine = x.clone()
        res = {}
        for name, extra in (("changed_games_only", 0), ("store_all", C.HK_F_STORE_ALL)):
            per = []
            for rep in range(4):
                x.copy_(pristine)
                torch.cuda.synchronize()
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(T + 1)]
                ev[0].record()
                for t in range(T):
                    rc = lib.hk_step(x.data_ptr(), x.data_ptr(), ha[t].data_ptr(), ax[t].data_ptr(), done.data_ptr(),
                                     rew.data_ptr(), None, None, None, None, B, N, d, C.HK_DTYPE_I32,
                                     C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON, C.HK_F_ACT_DISCRETE | extra,
                                     -1.0, 1e8, stream)
                    assert rc == 0
                    ev[t + 1].record()
                torch.cuda.synchronize()
                if rep:
                    per.append([ev[t].elapsed_time(ev[t + 1]) for t in range(T)])
            per = np.mean(np.array(per), axis=0)
            ms = float(per.mean())
            res[name] = {"ms_per_step": ms, "game_steps_per_s": B / (ms * 1e-3),
                         "hbm_frac_algorithmic": B * (8 * N * d + 13) / (ms * 1e-3) / 1e9 / peak_hbm,
                         "ms_by_rollout_step": [round(float(v), 4) for v in per]}
        res["workload"] = ("C2, 1 Mi games, one 20-step random-play rollout, in place: the default (only games that "
                           "changed are written back) against HK_F_STORE_ALL (every game rewritten every step)")
        out["C2_write_back"] = res
        del x, pristine
    except Exception as e:
        out["C2_write_back"] = {"error": repr(e)}

    # C2 with the fused host observation (kernel (c) of the north star): step + done/reward + features in one launch
    try:
        B, N, d, T = GAMES_PER_GPU, N_POINTS, DIM, T_ROLLOUT
        x, ha, ax = make(B, N, d, T, MAX_VALUE, 11, True)
        done, rew = torch.empty(B, dtype=torch.uint8, device=dev), torch.empty(B, dtype=torch.float32, device=dev)
        obs = torch.empty((B, N * d), dtype=torch.float32, device=dev)
        pristine = x.clone()
        oflags = C.HK_F_ACT_DISCRETE | C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE
        per = []
        for rep in range(4):
            x.copy_(pristine)
            torch.cuda.synchronize()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(T + 1)]
            ev[0].record()
            for t in range(T):
                rc = lib.hk_step(x.data_ptr(), x.data_ptr(), ha[t].data_ptr(), ax[t].data_ptr(), done.data_ptr(),
                                 rew.data_ptr(), None, obs.data_ptr(), None, None, B, N, d, C.HK_DTYPE_I32,
                                 C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON, oflags, -1.0, 1e8, stream)
                assert rc == 0
                ev[t + 1].record()
            torch.cuda.synchronize()
            if rep:
                per.append([ev[t].elapsed_time(ev[t + 1]) for t in range(T)])
        per = np.mean(np.array(per), axis=0)
        ms = float(per.mean())
        bytes_obs = 8 * N * d + 13 + 4 * N * d
        # the same through hk_step_census_obs: games at rest get their constant observation from the census byte
        census_o = torch.zeros(lib.hk_census_bytes(B, N, d), dtype=torch.uint8, device=dev)
        per_c = []
        for rep in range(4):
            x.copy_(pristine)
            census_o.zero_()
            rc = lib.hk_step_census(x.data_ptr(), None, None, None, None, None, None, census_o.data_ptr(), None, None, B, N, d,
                                    C.HK_DTYPE_I32, C.HK_OP_NEWTON | C.HK_OP_REPOSITION, 0, -1.0, 1e8, stream)
            assert rc == 0
            torch.cuda.synchronize()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(T + 1)]
            ev[0].record()
            for t in range(T):
                rc = lib.hk_step_census_obs(x.data_ptr(), ha[t].data_ptr(), ax[t].data_ptr(), done.data_ptr(), None, rew.data_ptr(),
                                            None, obs.data_ptr(), None, census_o.data_ptr(), None, None, B, N, d, C.HK_DTYPE_I32,
                                            C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON, oflags, -1.0, 1e8, stream)
                assert rc == 0
                ev[t + 1].record()
            torch.cuda.synchronize()
            if rep:
                per_c.append([ev[t].elapsed_time(ev[t + 1]) for t in range(T)])
        per_c = np.mean(np.array(per_c), axis=0)
        ms_c = float(per_c.mean())
        out["C2_step_with_features"] = {
            "workload": "C2, 1 Mi games, random play T=20; one launch per step = shift + reposition + newton + done/reward + "
                        "host observation (rescaled, lexicographically sorted f32 rows)",
            "kernel": "hk::hk_small_kernel<int,20,3,true>", "ms_per_step": ms, "game_steps_per_s": B / (ms * 1e-3),
            "bytes_per_game_step": bytes_obs, "hbm_frac": B * bytes_obs / (ms * 1e-3) / 1e9 / peak_hbm,
            "ms_by_rollout_step": [round(float(v), 4) for v in per],
            "census": {"api": "hk_step_census_obs (hk_sched_kernel<..., OBS>): the observation of a game at rest is a constant "
                              "written from its census byte; only the games in play run the feature code",
                       "ms_per_step": ms_c, "game_steps_per_s": B / (ms_c * 1e-3),
                       "hbm_frac": B * bytes_obs / (ms_c * 1e-3) / 1e9 / peak_hbm,
                       "ms_by_rollout_step": [round(float(v), 4) for v in per_c]}}
        del x, obs, pristine
    except Exception as e:
        out["C2_step_with_features"] = {"error": repr(e)}

    # C3: MCTS node expansion — latency per call at eval_batch_size 10/100/512 (N=20, d=3)
    lat = {}
    for B, N in ((10, 20), (100, 20), (512, 20), (10, 5), (512, 5)):
        d, T = 3, 20
        x, ha, ax = make(B, N, d, T, 20, 3, True)
        done, rew = torch.empty(B, dtype=torch.uint8, device=dev), torch.empty(B, dtype=torch.float32, device=dev)
        obs = torch.empty((B, N * d), dtype=torch.float32, device=dev)
        flags = C.HK_F_ACT_DISCRETE | C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE

        def one(i):
            rc = lib.hk_step(x.data_ptr(), x.data_ptr(), ha[i % T].data_ptr(), ax[i % T].data_ptr(), done.data_ptr(),
                             rew.data_ptr(), None, obs.data_ptr(), None, None, B, N, d, C.HK_DTYPE_I32,
                             C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON, flags, -1.0, 1e8, stream)
            assert rc == 0
        stream_us = timed(one, 2000) * 1e3
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            gs = torch.cuda.current_stream(dev).cuda_stream
            rc = lib.hk_step(x.data_ptr(), x.data_ptr(), ha[0].data_ptr(), ax[0].data_ptr(), done.data_ptr(),
                             rew.data_ptr(), None, obs.data_ptr(), None, None, B, N, d, C.HK_DTYPE_I32,
                             C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON, flags, -1.0, 1e8, gs)
            assert rc == 0
        graph_us = timed(lambda i: g.replay(), 2000) * 1e3
        lat[f"B={B},N={N}"] = {"stream_launch_us": stream_us, "graph_replay_us": graph_us}
    out["C3_step_with_features_us_per_call"] = lat

    # one-launch rollout (hk_rollout, T=20): the state is read and written once per 20 steps
    B, N, d, T = GAMES_PER_GPU, N_POINTS, DIM, T_ROLLOUT
    x, ha, ax = make(B, N, d, T, MAX_VALUE, 9, True)
    pristine = x.clone()
    dcount = torch.zeros(T, dtype=torch.int32, device=dev)

    def roll(i):
        x.copy_(pristine)
        rc = lib.hk_rollout(x.data_ptr(), x.data_ptr(), ha.data_ptr(), ax.data_ptr(), None, None, dcount.data_ptr(), None,
                            B, N, d, T, C.HK_DTYPE_I32, C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON,
                            C.HK_F_ACT_DISCRETE, -1.0, stream)
        assert rc == 0

    def copy2(i):
        x.copy_(pristine)
    ms = timed(roll, 10) - timed(copy2, 10)
    out["rollout_fused_T20"] = {"workload": "C2, 1 Mi games, hk_rollout: 20 steps in one launch", "ms_per_rollout": ms,
                                "game_steps_per_s": B * T / (ms * 1e-3),
                                "bytes_per_game_step": (8 * N * d) / T + 8 + 0.0}
    return out


def measure_e2e(torch, dev, B, K, pts, ha, ax, n_roll, barrier, world, dist, repeats: int = 5):
    """The same K steps through the host-buffer C-ABI (hk_session_rollout_bits / _ex via HostSession.rollout): the
    state of each rollout batch is resident; EVERY step copies that step's actions from pinned host memory and
    brings back the step's per-game done flags and the finished-game count.  Three streams inside the session
    (uploads, steps, read-backs); a repeated call replays as one CUDA graph.  The K steps are repeated
    `repeats` times from the same start and the MEDIAN is reported (a single ~1 ms window is noisy).
    Headline: the compact transport — two games' actions per byte up (HK_F_ACT_NIBBLE), the done flags as a bit
    mask down.  `bytes_variant`: one action byte per game up (HK_F_ACT_PACKED), one done byte per game down."""
    from hironaka_b200 import HostSession, constants as C
    op_step = C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON
    root_ops = C.HK_OP_NEWTON | C.HK_OP_REPOSITION
    nwords = (B + 31) // 32
    nib_pin = torch.from_numpy(HostSession.pack_actions_nibble(ha[:n_roll], ax[:n_roll])).pin_memory()
    bits_pin = torch.empty((n_roll, T_ROLLOUT, nwords), dtype=torch.int32).pin_memory()
    ha_pin = torch.from_numpy(HostSession.pack_actions(ha[:n_roll], ax[:n_roll])).pin_memory()
    done_pin = torch.empty((n_roll, T_ROLLOUT, B), dtype=torch.uint8).pin_memory()
    sessions, starts = [], []
    for r in range(n_roll):
        s = HostSession(pts[r], device=dev.index)
        s.step(None, None, root_ops, 0)  # root filter (generate_pts), untimed
        sessions.append(s)
        starts.append(s.get_state())

    def rollout(r, T, compact):
        if compact:
            return sessions[r].rollout(nib_pin[r, :T].numpy(), None, op_step, C.HK_F_ACT_DISCRETE | C.HK_F_ACT_NIBBLE,
                                       done_bits=bits_pin[r, :T].numpy().view(np.uint32))
        return sessions[r].rollout(ha_pin[r, :T].numpy(), None, op_step, C.HK_F_ACT_DISCRETE | C.HK_F_ACT_PACKED,
                                   done=done_pin[r, :T].numpy())

    def one_pass(compact):
        barrier()
        t0 = time.perf_counter()
        total_done, done_steps, i = 0, 0, 0
        while done_steps < K:
            r = i % n_roll
            if i >= n_roll:  # reuse of a batch beyond K = 200 (charged to the timed region)
                sessions[r].set_state(starts[r])
            T = min(T_ROLLOUT, K - done_steps)
            counts = rollout(r, T, compact)
            total_done += int(counts.sum())
            done_steps += T
            i += 1
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3  # host-blocking API: wall clock is the device time plus the copies
        r = (i - 1) % n_roll  # the flags of the last step did reach the host
        check = int(HostSession.unpack_done_bits(bits_pin[r, T - 1].numpy().view(np.uint32), B).sum()) if compact \
            else int(done_pin[r, T - 1].sum())
        return ms, total_done, check, int(counts[-1])

    def measure(compact):
        times, total_done = [], 0
        for rep in range(repeats + 1):  # (the first pass runs eagerly and is not counted: graphs are captured on the second)
            for r in range(n_roll):  # back to the same start; the root filter is replayed (idempotent) to fill the census
                sessions[r].set_state(starts[r])
                sessions[r].step(None, None, root_ops, 0)
            ms, total_done, check, last = one_pass(compact)
            assert check == last, (check, last)
            if world > 1:
                tt = torch.tensor([ms], device=dev, dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                ms = float(tt.item())
            if rep:
                times.append(ms)
        return float(np.median(times)), times, total_done

    ms, times, total_done = measure(True)
    ms_b, times_b, _ = measure(False)
    for s in sessions:
        s.close()
    return {"value": B * world * K / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": (B + 1) // 2,
            "d2h_bytes_per_step": nwords * 4 + 4, "ms_per_step": ms / K, "repeats": repeats,
            "ms_per_step_all": [round(t / K, 5) for t in times],
            "api": "hk_session_rollout_bits (HostSession.rollout): per step H2D of half a byte per game (two games' discrete "
                   "host id | axis << 2 per byte, HK_F_ACT_NIBBLE) from pinned memory, one hk_step_census launch, D2H of "
                   "the per-game done flags as a bit mask (pinned) and of the finished-game count; CUDA-graph replay; "
                   "median of the repeats after one untimed eager pass",
            "bytes_variant": {"value": B * world * K / (ms_b * 1e-3), "ms_per_step": ms_b / K, "h2d_bytes_per_step": B,
                              "d2h_bytes_per_step": B + 4, "ms_per_step_all": [round(t / K, 5) for t in times_b],
                              "api": "hk_session_rollout_ex: one packed action byte per game up (HK_F_ACT_PACKED), one "
                                     "done byte per game down"},
            "checksum_done": int(total_done)}


def measure_collective(torch, dist, lib, C, dev, world, rank, games: int = 1 << 16):
    """The one collective of the path: the all-gather (NCCL over NVLink) that assembles per-rank rollout buffers
    for training, hironaka_b200.engine.gather_rollout — the analogue of the leading device axis pmap returns in
    JAXTrainer.simulate (hironaka/jax/jax_trainer.py:316-320,558-592).  Each rank plays a real T-step rollout of
    `games` games with the fused observation, producing obs [games*T, N*d] f32, policy logits [games*T, A] f32
    and values [games*T] f32 (the last two are placeholders of the right size: the nets are out of scope), then
    all ranks gather them.  Timed three ways on the device: the gather alone, the next rollout alone, and both
    together (gather on a side stream) — the overlap fraction says how much of the gather hides behind play."""
    from hironaka_b200.engine import gather_rollout
    N, d, T = N_POINTS, DIM, T_ROLLOUT
    A = 2 ** d - d - 1
    rng = np.random.default_rng(500 + rank)
    stream = torch.cuda.current_stream(dev).cuda_stream
    x0 = torch.from_numpy(rng.integers(0, MAX_VALUE, size=(games, N, d), dtype=np.int32)).to(dev)
    ha = torch.from_numpy(rng.integers(0, A, size=(T, games), dtype=np.int32)).to(dev)
    ax = torch.from_numpy(rng.integers(0, d, size=(T, games), dtype=np.int32)).to(dev)
    obs = torch.empty((T, games, N * d), dtype=torch.float32, device=dev)
    policy = torch.zeros((games * T, A), dtype=torch.float32, device=dev)
    value = torch.zeros(games * T, dtype=torch.float32, device=dev)
    oflags = C.HK_F_ACT_DISCRETE | C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE | C.HK_F_RESCALE_EPS
    x = x0.clone()

    def rollout():
        x.copy_(x0)
        rc = lib.hk_step(x.data_ptr(), x.data_ptr(), None, None, None, None, None, None, None, None, games, N, d,
                         C.HK_DTYPE_I32, C.HK_OP_NEWTON | C.HK_OP_REPOSITION, 0, -1.0, 1e8, stream)
        for t in range(T):
            rc |= lib.hk_step(x.data_ptr(), x.data_ptr(), ha[t].data_ptr(), ax[t].data_ptr(), None, None, None,
                              obs[t].data_ptr(), None, None, games, N, d, C.HK_DTYPE_I32,
                              C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON, oflags, -1.0, 1e8, stream)
        assert rc == 0

    def gather():
        return gather_rollout((obs.view(games * T, N * d), policy, value))

    def timed(fn, n=5):
        fn()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / n], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    rollout()
    out = gather()
    torch.cuda.synchronize()
    ok = bool(torch.equal(out[0][rank], obs.view(games * T, N * d)))  # this rank's slice came back intact
    side = torch.cuda.Stream(dev)

    def both():
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            gather()
        rollout()
        torch.cuda.current_stream(dev).wait_stream(side)

    ms_g, ms_r, ms_b = timed(gather), timed(rollout), timed(both)
    sent = obs.numel() * 4 + policy.numel() * 4 + value.numel() * 4
    recv = sent * (world - 1)
    return {"what": "all_gather_into_tensor of one rollout's obs/policy/value per rank (engine.gather_rollout, NCCL)",
            "games_per_rank": games, "steps": T, "bytes_sent_per_rank": sent, "bytes_received_per_rank": recv,
            "gather_ms": ms_g, "bus_gbps": recv / (ms_g * 1e-3) / 1e9,
            "nvlink_ref_gbps": 770.0, "bus_frac_of_measured_peer_copy": recv / (ms_g * 1e-3) / 1e9 / 770.0,
            "rollout_with_features_ms": ms_r, "overlapped_ms": ms_b,
            "overlap_fraction": max(0.0, min(1.0, (ms_g + ms_r - ms_b) / max(1e-9, min(ms_g, ms_r)))),
            "own_slice_intact": ok}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer end-to-end leg (profiling runs)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg (profiling runs)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the other BASELINE configs (profiling runs)")
    ap.add_argument("--no-pdl", action="store_true", help="disable programmatic dependent launch (A/B tuning)")
    ap.add_argument("--no-collective", action="store_true", help="skip the rollout all-gather leg (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed on rank 0 (done, reward, a seeded sample of the "
                         "new states) as DIR/<name>.npy, to compare builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be >= 1")
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the GPU arm's outputs; --impl reference has none")
        return run_reference_arm(args)
    return run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
