"""CPU-only checks of the boundary and the host-side logic (no compute calls: there is no GPU
here and the product has no CPU path)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "hironaka_b200.h")


def header_text():
    return open(HEADER).read()


def declared_functions():
    txt = re.sub(r"/\*.*?\*/", "", header_text(), flags=re.S)
    return sorted(set(re.findall(r"\b(hk_[a-z_0-9]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    import hironaka_b200
    from hironaka_b200 import _lib
    if not os.path.exists(hironaka_b200.LIB_PATH):
        pytest.skip("library not built in this checkout (run python -m hironaka_b200.build)")
    L = ctypes.CDLL(hironaka_b200.LIB_PATH)
    names = declared_functions()
    assert len(names) >= 18
    for n in names:
        assert hasattr(L, n), f"{n} declared in the header but not exported"
    assert sorted(_lib.SIGNATURES) == names, "python binding and header disagree on the symbol list"
    lib = _lib.lib()
    assert lib.hk_version() == hironaka_b200.HK_VERSION
    assert lib.hk_error_string(0) == b"ok" and b"unsupported" in lib.hk_error_string(-2)
    assert lib.hk_kernel_class(20, 3) == 1 and lib.hk_kernel_class(64, 5) == 0
    assert lib.hk_kernel_class(2000, 3) < 0 and lib.hk_kernel_class(4, 11) < 0


def test_constants_match_header():
    from hironaka_b200 import constants as C
    txt = header_text()
    defs = dict(re.findall(r"#define\s+(HK_[A-Z_0-9]+)\s+(\(?[-0-9a-zA-Z<< u]+\)?)", txt))
    checked = 0
    for name, expr in defs.items():
        if not hasattr(C, name):
            continue
        val = eval(expr.replace("u", ""))
        assert getattr(C, name) == val, name
        checked += 1
    assert checked >= 20


def test_no_fallback_when_library_missing(tmp_path):
    """The product must fail loudly without the CUDA extension, and on CPU tensors."""
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "import hironaka_b200._lib as L\n"
        "L.LIB_PATH = %r\n"
        "try:\n"
        "    L.lib()\n"
        "    print('LOADED')\n"
        "except L.HironakaB200Error as e:\n"
        "    print('RAISED', 'no fallback' in str(e).lower())\n"
    ) % (ROOT, str(tmp_path / "missing.so"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert "RAISED True" in out.stdout, out.stdout + out.stderr
    import torch
    from hironaka_b200 import HironakaB200Error, ops
    with pytest.raises(HironakaB200Error):
        ops.step(torch.zeros(2, 5, 3, dtype=torch.int32), ops=4)
    with pytest.raises(HironakaB200Error):
        from hironaka_b200 import TensorPoints
        TensorPoints(torch.zeros(1, 2, 3), device="cpu")


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "hironaka_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.lower(), f"{f} mentions the oracle"
                assert "/root/reference" not in txt


def test_host_action_closed_form_and_encoder():
    from hironaka_b200.host_action import (HostActionEncoder, action_masks, batch_encode, batch_encode_one_hot,
                                           decode_id, decode_table, encode_mask, get_batch_decode)
    from oracle import hk_oracle as O
    from tests import kat as K
    import torch
    for d in range(2, 11):
        masks = action_masks(d)
        assert len(masks) == 2 ** d - d - 1
        for i, m in enumerate(masks):
            assert decode_id(i) == m and encode_mask(m) == i  # the kernel's closed form == the table
        assert np.array_equal(decode_table(d).numpy(), O.decode_table(d))
    enc = HostActionEncoder(3)
    assert enc.encode([0, 1]) == 0 and enc.decode(0) == [0, 1] and enc.decode(3) == [0, 1, 2]
    assert enc.decode_tensor(torch.tensor([0, 1])).tolist() == [[1, 1, 0], [1, 0, 1]]
    assert enc.encode_tensor(torch.tensor(K.ENCODE_IN)).tolist() == K.ENCODE_OUT.tolist()
    assert batch_encode(torch.tensor(K.ENCODE_IN)).tolist() == K.ENCODE_OUT.tolist()
    assert np.array_equal(batch_encode_one_hot(torch.tensor(K.ENCODE_IN)).numpy(), K.ENCODE_ONE_HOT_OUT)
    assert np.array_equal(get_batch_decode(3)(torch.tensor(K.ENCODE_OUT)).numpy(), K.ENCODE_IN)


def test_golden_tables_match_host_action(golden_dir):
    from hironaka_b200.host_action import decode_table
    g = np.load(os.path.join(golden_dir, "ref_tables.npz"))
    for d in range(2, 8):
        assert np.array_equal(decode_table(d).numpy(), g[f"decode_{d}"].astype(np.int32))


def test_coords_to_mask_cpu():
    import torch
    from hironaka_b200.ops import coords_to_mask
    assert coords_to_mask([[1, 2], [0, 2, 3]], 4, "cpu").tolist() == [0b0110, 0b1101]
    assert coords_to_mask(torch.tensor([[0., 1., 1., 0.], [1., 0., 1., 1.]]), 4, "cpu").tolist() == [0b0110, 0b1101]
    with pytest.raises(ValueError):
        coords_to_mask([[4]], 4, "cpu")


def test_shard_range_partitions():
    from hironaka_b200.engine import shard_range
    for total in (0, 1, 7, 8, 1000, 1 << 20):
        for world in (1, 2, 3, 4, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(10, 2, 2)


def test_rho_from_counts():
    import torch
    from hironaka_b200.engine import GameBatch
    # 10 games: 2 done at entry, then 3 / 6 / 6 finished after steps 1..3
    rho = GameBatch.rho(2, torch.tensor([3, 6, 7]), 10)
    # details (compute_rho, jax_trainer.py:519-555): [2, 1, 3, 10-7=3] -> rho = (1+3+3) / (1*1 + 2*3 + 3*3)
    assert abs(rho - 7 / 16) < 1e-12


def test_bench_reference_arm_runs_on_cpu():
    """`bench.py --impl reference` is the CPU arm — the unmodified reference from baseline/_ref when it is there
    (kind "reference"), the oracle's C port otherwise (kind "port"): it must run without a GPU and print one
    JSON line with the contract's keys."""
    import json
    from baseline import reference_arm as R
    env = dict(os.environ, HK_BENCH_CPU_SAMPLE="4096", HK_BENCH_REF_SAMPLE="512")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3",
                          "--warmup", "1"], capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "game_steps_per_sec" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == ("reference" if R.available() else "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["config"]["workload"].startswith("C2")
    for k in ("unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data"):
        assert k in line


def test_reference_arm_matches_the_oracle(golden_dir):
    """Parity gate of the reference arm (BASELINE.md section 3): what bench.py times as "the reference" — the
    unmodified hironaka.core.TensorPoints playing C2 random games, shift -> reposition -> newton ->
    ended_batch_in_tensor -> reward — gives, step by step, the states, done flags and rewards of the oracle's torch
    flavour on the same inputs (the GPU arm is held to the same oracle by tests/test_gpu_parity.py, and to this arm
    directly by test_reference_arm_matches_the_gpu).  The reference's side is stored: ref_rollout_c2_20x3*.npz,
    recorded from the unmodified reference by oracle/gen_golden.py (rollout_torch plays that composition), tiled
    here to 1024 games.  Where baseline/_ref is installed, the live reference also plays the bench's own inputs."""
    from baseline import reference_arm as R
    from oracle import cport, hk_oracle as O
    flags = O.F_NOOP_INVALID | O.F_FREEZE_ENDED | O.F_ACT_DISCRETE
    for name in ("c2_20x3", "c2_20x3_repos"):
        g = np.load(os.path.join(golden_dir, f"ref_rollout_{name}.npz"))
        _, B, _, _, T, _, _, repos = g["meta"].tolist()
        reps = -(-1024 // B)

        def tile(a):
            return np.tile(a, (reps,) + (1,) * (a.ndim - 1))
        ops = O.OP_SHIFT | O.OP_NEWTON | (O.OP_REPOSITION if repos else 0)
        o = cport.step(tile(g["init"]).astype(np.int32), None, None, O.OP_NEWTON, 0)[0]
        assert np.array_equal(o.astype(np.float32), tile(g["states"][0])), name
        for t in range(T):
            o, od, orw, _ = cport.step(o, tile(g["host_ids"][t]), tile(g["axes"][t]), ops, flags)
            assert np.array_equal(o.astype(np.float32), tile(g["states"][t + 1])), (name, t)
            assert np.array_equal(od.astype(bool), tile(g["dones"][t + 1])), (name, t)
            assert np.array_equal(orw, tile(g["dones"][t + 1] & ~g["dones"][t]).astype(np.float32)), (name, t)
    if not R.available():
        return
    sys.path.insert(0, ROOT)
    import bench
    torch, TensorPoints, HostActionEncoder = R.import_reference()
    B, T = 1024, 12
    pts, ha, ax = bench.make_inputs(99, B, 1)
    tp = R.root_states(TensorPoints, torch, pts[0], True)
    o = cport.step(pts[0], None, None, O.OP_NEWTON | O.OP_REPOSITION, 0)[0]
    assert np.array_equal(tp.points.numpy(), o.astype(np.float32))
    rec = []
    counts = R.play(tp, HostActionEncoder(3), torch, ha[0, :T], ax[0, :T], True, record=rec)
    for t in range(T):
        o, od, orw, _ = cport.step(o, ha[0, t], ax[0, t], O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, flags)
        assert np.array_equal(rec[t][0], o.astype(np.float32)), t
        assert np.array_equal(rec[t][1], od.astype(bool)) and np.array_equal(rec[t][2], orw), t
        assert counts[t] == int(od.sum())


def test_policy_glue_of_functional():
    """get_value_est_fn / apply_agent_action_mask / action_wrapper / rollout_sanity_tests
    (hironaka/jax/util.py:152-169,287-327,395-423): tensor plumbing, runs anywhere."""
    torch = pytest.importorskip("torch")
    from hironaka_b200 import functional as F
    est = F.get_value_est_fn("agent")(torch.zeros(3), torch.tensor([0, 2, 5]))
    assert torch.allclose(est, torch.tensor([-1.0, -0.5, -0.2]))
    n, d = 4, 3
    obs = torch.zeros(2, (n + 1) * d)
    obs[0, -d:] = torch.tensor([1.0, 0.0, 1.0])
    obs[1, -d:] = torch.tensor([0.0, 1.0, 1.0])

    def policy(x):
        return torch.tensor([[0.1, 5.0, 0.3], [2.0, 0.1, 0.3]]), torch.zeros(2)
    masked, _ = F.apply_agent_action_mask(policy, d)(obs)
    assert masked[0].tolist() == [pytest.approx(0.1), float("-inf"), pytest.approx(0.3)]
    act = F.action_wrapper(policy, d)(obs)
    assert act.tolist() == [[0.0, 0.0, 1.0], [0.0, 0.0, 1.0]]
    assert F.rollout_sanity_tests((obs, masked, torch.zeros(2)), (n, d))
    assert not F.rollout_sanity_tests((obs, policy(obs)[0], torch.zeros(2)), (n, d))  # mask not applied
    soft = torch.softmax(torch.randn(2, 3), dim=-1)
    assert not F.rollout_sanity_tests((torch.zeros(2, n * d), soft, torch.zeros(2)), (n, d))  # already a softmax


@pytest.mark.parametrize("n", [5, 10, 20])
def test_committed_sorting_networks_sort(n):
    """hk_sortnet.inc (generated by tools/gen_sortnet.py) is what the features kernel sorts row keys
    with: the comparator lists of the instantiated sizes must sort every 0/1 input (0-1 principle)."""
    import re
    src = open(os.path.join(ROOT, "hironaka_b200", "csrc", "hk_sortnet.inc")).read()
    m = re.search(r"if constexpr \(N == %d\) \{(.*?)\n\}" % n, src, re.S)
    assert m, f"no network for n = {n}"
    ces = [(int(a), int(b)) for a, b in re.findall(r"HK_CE\((\d+), (\d+)\)", m.group(1))]
    assert ces and all(0 <= a < b < n for a, b in ces)
    x = np.arange(1 << n, dtype=np.uint32)
    bits = [(x >> i) & 1 for i in range(n)]
    for a, b in ces:  # HK_CE(i, j): k[i] = max, k[j] = min (descending)
        bits[a], bits[b] = np.maximum(bits[a], bits[b]), np.minimum(bits[a], bits[b])
    assert all(bool(np.all(bits[i] >= bits[i + 1])) for i in range(n - 1))
