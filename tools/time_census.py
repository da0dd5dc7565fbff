"""Per-step device times of a C2 (or C5) random-play rollout: hk_step (tile ring) against hk_step_census
(census-scheduled).  python tools/time_census.py [c2|c5] [reps] [census]"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hironaka_b200 import constants as C  # noqa: E402
from hironaka_b200._lib import lib  # noqa: E402

which = sys.argv[1] if len(sys.argv) > 1 else "c2"
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 4
B, N, d, T = ((1 << 20, 20, 3, 20) if which == "c2" else (1 << 18, 64, 5, 20))
L = lib()
dev = torch.device("cuda")
rng = np.random.default_rng(3)
x0 = torch.from_numpy(rng.integers(0, 20, size=(B, N, d), dtype=np.int32)).to(dev)
ha = torch.from_numpy(rng.integers(0, 2 ** d - d - 1, size=(T, B), dtype=np.int32)).to(dev)
ax = torch.from_numpy(rng.integers(0, d, size=(T, B), dtype=np.int32)).to(dev)
done = torch.empty(B, dtype=torch.uint8, device=dev)
rew = torch.empty(B, dtype=torch.float32, device=dev)
stream = torch.cuda.current_stream().cuda_stream
OPS = C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON
ROOT = C.HK_OP_NEWTON | C.HK_OP_REPOSITION


root_ms = []


def run(census_mode):
    root_ms.clear()
    per = []
    final = None
    for rep in range(reps):
        x = x0.clone()
        census = torch.zeros(L.hk_census_bytes(B, N, d), dtype=torch.uint8, device=dev)
        cp = census.data_ptr() if census_mode else None
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        if census_mode:
            rc = L.hk_step_census(x.data_ptr(), None, None, None, None, None, None, cp, None, None, B, N, d, C.HK_DTYPE_I32, ROOT, 0,
                                  -1.0, 1e8, stream)
        else:
            rc = L.hk_step(x.data_ptr(), x.data_ptr(), None, None, None, None, None, None, None, None, B, N, d,
                           C.HK_DTYPE_I32, ROOT, 0, -1.0, 1e8, stream)
        assert rc == 0, rc
        r1.record()
        torch.cuda.synchronize()
        if rep:
            root_ms.append(r0.elapsed_time(r1))
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(T + 1)]
        ev[0].record()
        for t in range(T):
            if census_mode:
                rc = L.hk_step_census(x.data_ptr(), ha[t].data_ptr(), ax[t].data_ptr(), done.data_ptr(), None, rew.data_ptr(), None,
                                      cp, None, None, B, N, d, C.HK_DTYPE_I32, OPS, C.HK_F_ACT_DISCRETE, -1.0, 1e8, stream)
            else:
                rc = L.hk_step(x.data_ptr(), x.data_ptr(), ha[t].data_ptr(), ax[t].data_ptr(), done.data_ptr(),
                               rew.data_ptr(), None, None, None, None, B, N, d, C.HK_DTYPE_I32, OPS, C.HK_F_ACT_DISCRETE,
                               -1.0, 1e8, stream)
            assert rc == 0, rc
            ev[t + 1].record()
        torch.cuda.synchronize()
        if rep:
            per.append([ev[t].elapsed_time(ev[t + 1]) for t in range(T)])
        final = x
    per = np.mean(np.array(per), axis=0)
    return per, final


out = {}
only = sys.argv[3] if len(sys.argv) > 3 else ""
if only.startswith("census"):  # profiling runs: one mode only
    per, _ = run(True)
    print(json.dumps({only: [round(float(v), 4) for v in per]}))
    sys.exit(0)
base, xb = run(False)
out["hk_step"] = {"mean_ms": float(base.mean()), "by_step": [round(float(v), 4) for v in base], "root_filter_ms": round(float(np.mean(root_ms)), 4)}
per, xc = run(True)
assert os.environ.get("HK_NOASSERT") or torch.equal(xc, xb), "census rollout differs from hk_step rollout"
out["hk_step_census"] = {"mean_ms": float(per.mean()), "by_step": [round(float(v), 4) for v in per], "root_filter_ms": round(float(np.mean(root_ms)), 4)}
out["workload"] = f"{which}: B={B} N={N} d={d} T={T}"
print(json.dumps(out))
