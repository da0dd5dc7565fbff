"""GPU parity tests: the CUDA path (through the C-ABI) against the oracle, bit-exact.

Run on a B200 with ``pytest -m gpu``.  Sources of truth, in order:
  * the reference's known-answer vectors (tests/kat.py),
  * outputs of the real reference (tests/golden/ref_*.npz),
  * the oracle (oracle/hk_oracle.py for small cases, oracle/cport.py = C port for large ones)
    on seeded random inputs, including BASELINE.json's full sizes.
Both kernel families (thread-per-game and warp-per-game) are exercised on every small shape via
the hk_debug_force_generic test hook.
"""
import glob
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import cport  # noqa: E402
from oracle import hk_oracle as O  # noqa: E402
from tests import kat as K  # noqa: E402

pytestmark = pytest.mark.gpu

TORCH_FLAGS = O.F_NOOP_INVALID | O.F_FREEZE_ENDED


@pytest.fixture(scope="module")
def hb():
    import hironaka_b200
    from hironaka_b200 import ops
    assert os.path.exists(hironaka_b200.LIB_PATH), "CUDA library not built"
    ops.force_generic(False)
    return hironaka_b200


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def run_step(hb, x_np, ha, ax, ops_bits, flags, pad=-1.0, want_obs=False, obs_coord=None):
    from hironaka_b200 import ops
    def call(x, inplace):
        return ops.step(x, None if ha is None else dev(ha.astype(np.int32)),
                        None if ax is None else dev(ax.astype(np.int32)), ops=ops_bits, flags=flags, padding_value=pad,
                        inplace=inplace, want_done=True, want_reward=True, want_num_points=True, want_obs=want_obs,
                        obs_coord=None if obs_coord is None else dev(obs_coord.astype(np.int32)))
    r = call(dev(x_np), False)
    out = (r.state.cpu().numpy(), r.done.cpu().numpy(), r.reward.cpu().numpy(), r.num_points.cpu().numpy(),
           None if r.obs is None else r.obs.cpu().numpy())
    # the same call in place (out == in) takes other routes through the library (changed games / rows
    # only are written back; large games go to the compacting kernel): it must give the same answers
    xi = dev(x_np)
    ri = call(xi, True)
    same = np.array_equal(xi.cpu().numpy().view(np.int32), out[0].view(np.int32))
    assert same, "in-place state differs from out-of-place"
    assert np.array_equal(ri.done.cpu().numpy(), out[1]) and np.array_equal(ri.reward.cpu().numpy(), out[2])
    assert np.array_equal(ri.num_points.cpu().numpy(), out[3])
    if want_obs:
        assert np.array_equal(ri.obs.cpu().numpy(), out[4])
    return out


@pytest.fixture(params=[False, True], ids=["family=auto", "family=generic"])
def family(request, hb):
    from hironaka_b200 import ops
    ops.force_generic(request.param)
    yield request.param
    ops.force_generic(False)


# ---------------------------------------------------------------- reference KATs


@pytest.mark.parametrize("dtype", [np.float32, np.int32])
def test_kat_ops(hb, family, dtype):
    x = K.R_IN.astype(dtype)
    n = run_step(hb, x, None, None, O.OP_NEWTON, 0)[0]
    assert np.array_equal(n, K.R.astype(dtype))
    s = run_step(hb, n, K.R_COORD_MASK, K.R_AXIS, O.OP_SHIFT, TORCH_FLAGS)[0]
    assert np.array_equal(s, K.R2.astype(dtype))
    r = run_step(hb, s, None, None, O.OP_REPOSITION, 0)[0]
    assert np.array_equal(r, K.R3.astype(dtype))
    f, done, rew, npts, _ = run_step(hb, n, K.R_COORD_MASK, K.R_AXIS, O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, 0)
    assert np.array_equal(f, K.R3.astype(dtype))
    assert done.tolist() == [False, False] and rew.tolist() == [0, 0] and npts.tolist() == [3, 2]
    q = run_step(hb, n, np.array([0b0010, 0b1101]), np.array(K.INVALID_AXIS), O.OP_SHIFT, TORCH_FLAGS)[0]
    assert np.array_equal(q, K.R.astype(dtype))
    e = run_step(hb, K.ENDED_P.astype(dtype), np.array([0b11]), np.array([1]), O.OP_SHIFT, TORCH_FLAGS)[0]
    assert np.array_equal(e, K.ENDED_P.astype(dtype))
    e = run_step(hb, K.ENDED_P.astype(dtype), np.array([0b11]), np.array([1]), O.OP_SHIFT, O.F_NOOP_INVALID)[0]
    assert np.array_equal(e, K.ENDED_Q.astype(dtype))
    o, done, rew, npts, _ = run_step(hb, K.ORIGIN20_IN.astype(dtype), None, None, O.OP_NEWTON, 0)
    assert np.array_equal(o, K.ORIGIN20_OUT.astype(dtype))
    assert done.tolist() == [True] and rew.tolist() == [1.0] and npts.tolist() == [1]
    assert np.array_equal(run_step(hb, K.REP_IN.astype(dtype), None, None, O.OP_NEWTON, 0)[0], K.REP_OUT.astype(dtype))
    assert np.array_equal(run_step(hb, K.REP_IN.astype(dtype), None, None, O.OP_DEDUPE, 0)[0], K.REP_OUT.astype(dtype))
    assert np.array_equal(run_step(hb, K.EXTREME_IN.astype(dtype), None, None, O.OP_NEWTON, 0)[0],
                          K.EXTREME_OUT.astype(dtype))


def test_kat_float(hb, family):
    assert np.array_equal(run_step(hb, K.R3, None, None, O.OP_RESCALE, 0)[0], K.RS)
    assert np.array_equal(run_step(hb, K.RESCALE_IN, None, None, O.OP_RESCALE, 0)[0], K.RESCALE_OUT)
    assert np.isfinite(run_step(hb, K.RESCALE0_IN, None, None, O.OP_RESCALE, 0)[0]).all()
    s = run_step(hb, K.FEAT_IN, np.array([0b110]), np.array([1]), O.OP_SHIFT, 0)[0]
    assert np.array_equal(s, K.FSHIFT_OUT)
    obs = run_step(hb, K.FEAT_IN, None, None, 0, O.F_OBS_SORT_LEX | O.F_OBS_RESCALE, want_obs=True)[4]
    assert np.array_equal(obs, K.FEAT_SORTED)
    pts = K.AGENT_FEAT_IN[:, :9].reshape(2, 3, 3).copy()
    cm = np.array([0b110, 0b101])
    for dt in (np.float32, np.int32):
        o = run_step(hb, pts.astype(dt), None, None, 0, O.F_OBS_SORT_LEX, want_obs=True, obs_coord=cm)[4]
        assert np.array_equal(o, K.AGENT_FEAT_NOSCALE)
        o = run_step(hb, pts.astype(dt), None, None, 0, O.F_OBS_SORT_LEX | O.F_OBS_RESCALE, want_obs=True, obs_coord=cm)[4]
        assert np.array_equal(o, K.AGENT_FEAT_SCALE)
    # take_actions composition with discrete ids (test/testJAX.py:461-488)
    s2 = run_step(hb, K.TA_HOST_OBS, np.array([2, 3]), np.array([1, 1]), O.OP_SHIFT | O.OP_NEWTON | O.OP_RESCALE,
                  O.F_ACT_DISCRETE)[0]
    ones = np.ones(2, np.float32)
    assert np.array_equal(s2.reshape(2, -1),
                          O.take_actions("host", (4, 3), K.TA_HOST_OBS.reshape(2, -1), K.TA_COORDS, ones, True, False))


# ---------------------------------------------------------------- real-reference goldens


@pytest.mark.parametrize("dtype", [np.float32, np.int32])
def test_golden_rollouts(hb, family, golden_dir, dtype):
    files = sorted(glob.glob(os.path.join(golden_dir, "ref_rollout_*.npz")))
    assert files
    for path in files:
        g = np.load(path)
        seed, B, N, d, T, mv, first, repos = g["meta"].tolist()
        ops_bits = O.OP_SHIFT | O.OP_NEWTON | (O.OP_REPOSITION if repos else 0)
        flags = TORCH_FLAGS | O.F_ACT_DISCRETE
        x, done, _, npts, _ = run_step(hb, g["init"].astype(dtype), None, None, O.OP_NEWTON, 0)
        assert np.array_equal(x.astype(np.float32), g["states"][0]), path
        assert np.array_equal(done, g["dones"][0]) and np.array_equal(npts, g["num_points"][0])
        for t in range(T):
            x, done, rew, npts, obs = run_step(hb, x, g["host_ids"][t], g["axes"][t], ops_bits,
                                               flags | O.F_OBS_SORT_COORD0, want_obs=True)
            assert np.array_equal(x.astype(np.float32), g["states"][t + 1]), (path, t)
            assert np.array_equal(done, g["dones"][t + 1]), (path, t)
            assert np.array_equal(npts, g["num_points"][t + 1]), (path, t)
            assert np.array_equal(rew, (g["dones"][t + 1] & ~g["dones"][t]).astype(np.float32)), (path, t)
            feat = obs.reshape(B, N, d)
            assert np.array_equal(feat[:, :, 0], g["features"][t][:, :, 0]), (path, t)
            if N <= 16:
                assert np.array_equal(feat, g["features"][t]), (path, t)
        # the same rollout as ONE launch (hk_rollout) must end in the same state
        from hironaka_b200 import ops
        st0 = dev(g["states"][0].astype(dtype))
        out, dn, rw, dcount, length = ops.rollout(st0, dev(g["host_ids"]), dev(g["axes"]), ops=ops_bits, flags=flags,
                                                  inplace=False, want_done=True, want_reward=True, want_length=True)
        assert np.array_equal(out.cpu().numpy().astype(np.float32), g["states"][T]), path
        assert np.array_equal(dn.cpu().numpy(), g["dones"][1:]), path
        assert np.array_equal(dcount.cpu().numpy(), g["dones"][1:].sum(1)), path
        first_done = np.where(g["dones"][0], 0, np.where(g["dones"][1:].any(0), g["dones"][1:].argmax(0) + 1, T + 1))
        assert np.array_equal(length.cpu().numpy(), first_done), path


@pytest.mark.parametrize("dtype", [np.float32, np.int32])
def test_golden_ops(hb, family, golden_dir, dtype):
    for path in sorted(glob.glob(os.path.join(golden_dir, "ref_ops_*.npz"))):
        g = np.load(path)
        x = g["points"].astype(dtype)
        B, N, d = x.shape
        hid, ax = g["host_ids"], g["axes"]
        c = lambda a: a.astype(np.float32)
        fl = O.F_ACT_DISCRETE
        assert np.array_equal(c(run_step(hb, x, hid, ax, O.OP_SHIFT, fl | TORCH_FLAGS)[0]), g["shift_ignore_ended"]), path
        assert np.array_equal(c(run_step(hb, x, hid, ax, O.OP_SHIFT, fl | O.F_NOOP_INVALID)[0]), g["shift_force_ended"]), path
        n = run_step(hb, x, None, None, O.OP_NEWTON, 0)[0]
        assert np.array_equal(c(n), g["newton"]), path
        assert np.array_equal(c(run_step(hb, x, None, None, O.OP_DEDUPE, 0)[0]), g["remove_repeated"]), path
        assert np.array_equal(c(run_step(hb, x, None, None, O.OP_REPOSITION, 0)[0]), g["reposition"]), path
        _, done0, _, npts0, _ = run_step(hb, x, None, None, 0, 0)
        assert np.array_equal(npts0, g["num_points"]) and np.array_equal(done0, g["ended"])
        obs = run_step(hb, n, None, None, 0, O.F_OBS_RESCALE, want_obs=True)[4]
        assert np.array_equal(obs.reshape(B, N, d), g["rescale_after_newton"]), path
        if dtype == np.float32:
            assert np.array_equal(run_step(hb, x, None, None, O.OP_RESCALE, 0)[0], g["rescale"]), path
            assert np.array_equal(run_step(hb, x, None, None, O.OP_NEWTON | O.OP_RESCALE, 0)[0],
                                  g["rescale_after_newton"]), path


# ---------------------------------------------------------------- seeded random vs oracle


def random_state(rng, B, N, d, max_value, dead_frac=0.2, dup_frac=0.2):
    x = rng.integers(0, max_value + 1, size=(B, N, d)).astype(np.int32)
    dead = rng.random((B, N)) < dead_frac
    x[dead] = -1
    for b in np.nonzero(rng.random(B) < dup_frac)[0]:
        i, j = rng.integers(0, N, 2)
        x[b, j] = x[b, i]
    return x


SHAPES = [(1, 5, 3), (7, 5, 3), (33, 10, 3), (257, 20, 3), (1000, 20, 3), (64, 2, 2), (50, 7, 2), (40, 16, 4),
          (37, 33, 3), (16, 64, 5), (5, 100, 3), (3, 300, 6), (9, 4, 10), (4, 1, 3), (2, 1024, 4)]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
def test_random_step_all_modes(hb, family, shape, dtype):
    B, N, d = shape
    rng = np.random.default_rng(B * 1000 + N * 10 + d)
    ncls = 2 ** d - d - 1
    for trial, (ops_bits, flags) in enumerate([
        (O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, 0),                                  # JAX step
        (O.OP_SHIFT | O.OP_NEWTON, TORCH_FLAGS),                                          # FusedGame step
        (O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, O.F_ACT_DISCRETE | O.F_ROLE_AGENT),  # discrete ids, agent reward
        (O.OP_SHIFT, O.F_FREEZE_ENDED),
        (O.OP_NEWTON, 0),
        (O.OP_REPOSITION | O.OP_DEDUPE, 0),
    ]):
        x = random_state(rng, B, N, d, max_value=int(rng.choice([1, 3, 20, 1000]))).astype(dtype)
        if flags & O.F_ACT_DISCRETE and ncls >= 1:
            ha = rng.integers(0, ncls, B)
        else:
            ha = rng.integers(0, 2 ** d, B)  # arbitrary masks, including empty and singletons
        ax = rng.integers(0, d, B)
        got = run_step(hb, x, ha, ax, ops_bits, flags)
        exp = cport.step(x, ha, ax, ops_bits, flags)
        assert np.array_equal(got[0], exp[0]), (trial, "state")
        assert np.array_equal(got[1], exp[1].astype(bool)), (trial, "done")
        assert np.array_equal(got[2], exp[2]), (trial, "reward")
        assert np.array_equal(got[3], exp[3]), (trial, "num_points")
        if B * N * N * d <= 2_000_000:  # NumPy restatement as a second, independent checker
            ref = O.step(x, ha, ax, ops_bits, flags)
            assert np.array_equal(got[0].astype(np.float32), ref[0]), (trial, "state/numpy")
            assert np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])


@pytest.mark.parametrize("shape", [(65, 20, 3), (33, 10, 3), (31, 5, 3), (12, 64, 5), (20, 16, 4), (6, 40, 2)],
                         ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
def test_random_features(hb, family, shape, dtype):
    B, N, d = shape
    rng = np.random.default_rng(N * 7 + d)
    x = random_state(rng, B, N, d, max_value=6, dead_frac=0.3).astype(dtype)  # small range => many key ties
    cm = rng.integers(0, 2 ** d, B)
    # the thread-per-game kernel ranks rows by packed integer keys while every live value is an integer
    # below 2^19 and by float compares otherwise: cover both, and the border between them
    variants = [x, np.where(x > 0, x * 80000, x).astype(dtype), np.where(x > 0, x * 100000, x).astype(dtype)]
    if dtype == np.float32:
        variants.append(np.where(x > 0, x + 0.5, x).astype(dtype))
        variants.append(np.where(x > 0, x / 8.0, x).astype(dtype))
    for vi, xv in enumerate(variants):
        for flags in (0, O.F_OBS_RESCALE, O.F_OBS_SORT_COORD0, O.F_OBS_SORT_LEX, O.F_OBS_SORT_LEX | O.F_OBS_RESCALE,
                      O.F_OBS_SORT_COORD0 | O.F_OBS_RESCALE, 1 << 12):  # 1 << 12 = HK_F_OBS_SORT_LEX_FIRST (C port only)
            for oc in (None, cm):
                got = run_step(hb, xv, None, None, 0, flags, want_obs=True, obs_coord=oc)[4]
                exp = cport.features(xv, flags, obs_coord=oc)
                assert np.array_equal(got, exp), (vi, flags, oc is None)
    # fused: features of the state AFTER the step
    ha, ax = rng.integers(0, 2 ** d, B), rng.integers(0, d, B)
    ops_bits = O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON
    got = run_step(hb, x, ha, ax, ops_bits, O.F_OBS_SORT_LEX | O.F_OBS_RESCALE, want_obs=True)
    exp_state = cport.step(x, ha, ax, ops_bits, 0)[0]
    assert np.array_equal(got[0], exp_state)
    assert np.array_equal(got[4], cport.features(exp_state, O.F_OBS_SORT_LEX | O.F_OBS_RESCALE))


@pytest.mark.parametrize("N", [5, 10, 20])
def test_rescale_with_empty_games_in_a_warp(hb, N):
    """Games without a live row sit next to live ones in the same warp: the per-game "anything to
    divide?" condition differs between lanes, the warp-wide choice of the division routine must not
    (regression: a vote taken under that condition let lanes run ahead of the obs-tile store)."""
    rng = np.random.default_rng(N)
    for B in (31, 64, 95):
        x = random_state(rng, B, N, 3, max_value=9, dead_frac=0.3).astype(np.float32)
        x[::3] = -1.0  # every third game is empty
        x[1::7, 1:] = -1.0  # and some have a single point
        for flags in (O.F_OBS_RESCALE, O.F_OBS_RESCALE | O.F_OBS_SORT_LEX, O.F_OBS_RESCALE | O.F_OBS_SORT_COORD0):
            for ops_bits in (0, O.OP_RESCALE, O.OP_NEWTON | O.OP_RESCALE):
                got = run_step(hb, x, None, None, ops_bits, flags, want_obs=True)
                exp_state = cport.step(x, None, None, ops_bits, 0)[0] if ops_bits else x
                assert np.array_equal(got[0], exp_state), (B, flags, ops_bits)
                assert np.array_equal(got[4], cport.features(exp_state, flags)), (B, flags, ops_bits)


@pytest.mark.parametrize("shape", [(1000, 20, 3), (333, 10, 3), (95, 5, 3), (300, 64, 5), (40, 16, 4)],
                         ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
def test_inplace_writes_only_changed_games(hb, family, shape, dtype):
    """In-place steps write back only the games that changed (most games of a long rollout sit at a
    fixed point).  The state must equal the oracle's after EVERY step, with and without
    HK_F_STORE_ALL, for both flavours, from a start whose dead rows hold arbitrary negative values
    (they must be normalised to the padding value) and whose ended games stay untouched."""
    from hironaka_b200 import ops
    B, N, d = shape
    rng = np.random.default_rng(B + N)
    T = 12
    x0 = random_state(rng, B, N, d, max_value=5, dead_frac=0.5, dup_frac=0.1).astype(dtype)
    junk = rng.random((B, N)) < 0.3  # dead rows that are not the padding value (still all-negative: well-formed)
    x0[(x0[:, :, 0] < 0) & junk] = -7
    x0[::5] = -1  # empty games
    x0[1::5, 1:] = -1  # single-point games
    x0[1::5, 0] = np.abs(x0[1::5, 0])
    ha = rng.integers(0, 2 ** d, size=(T, B)).astype(np.int32)
    ax = rng.integers(0, d, size=(T, B)).astype(np.int32)
    for ops_bits, flags in ((O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, 0), (O.OP_SHIFT | O.OP_NEWTON, TORCH_FLAGS),
                            (O.OP_SHIFT, TORCH_FLAGS), (O.OP_REPOSITION, 0)):
        o = x0.copy()
        g_sparse, g_all = dev(x0), dev(x0)
        for t in range(T):
            o = cport.step(o, ha[t], ax[t], ops_bits, flags)[0]
            ops.step(g_sparse, dev(ha[t]), dev(ax[t]), ops=ops_bits, flags=flags, inplace=True)
            ops.step(g_all, dev(ha[t]), dev(ax[t]), ops=ops_bits, flags=flags | (1 << 13), inplace=True)
            assert np.array_equal(g_sparse.cpu().numpy(), o), (ops_bits, flags, t)
            assert np.array_equal(g_all.cpu().numpy(), o), (ops_bits, flags, t, "store_all")


@pytest.mark.parametrize("shape", [(40003, 20, 3), (30001, 10, 3), (20001, 5, 3), (6011, 64, 5), (4001, 16, 4), (1003, 33, 3)],
                         ids=lambda s: "x".join(map(str, s)))
def test_changed_games_only_equals_store_all_under_caller_rewrites(hb, shape):
    """Long in-place rollouts, both dtypes and flavours, while the caller overwrites some games between
    steps (dead rows that are not the padding value included): the default write-back of changed games
    only and HK_F_STORE_ALL must stay identical in state and in every output.  The two kernel families
    are covered by the shapes."""
    from hironaka_b200 import constants as C, ops
    B, N, d = shape
    rng = np.random.default_rng(B)
    for dtype in (torch.int32, torch.float32):
        for ops_bits, flags in ((C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON, 0),
                                (C.HK_OP_SHIFT | C.HK_OP_NEWTON, C.TORCH_SEMANTICS)):
            x = rng.integers(0, 12, (B, N, d)).astype(np.int32)
            x[rng.random((B, N)) < 0.4] = -1
            a = torch.from_numpy(x).cuda().to(dtype)
            b = a.clone()
            for t in range(16):
                ha = torch.from_numpy(rng.integers(0, 2 ** d, B).astype(np.int32)).cuda()
                ax = torch.from_numpy(rng.integers(0, d, B).astype(np.int32)).cuda()
                ra = ops.step(a, ha, ax, ops=ops_bits, flags=flags, inplace=True, want_done=True, want_reward=True,
                              want_num_points=True)
                rb = ops.step(b, ha, ax, ops=ops_bits, flags=flags | C.HK_F_STORE_ALL, inplace=True, want_done=True,
                              want_reward=True, want_num_points=True)
                assert torch.equal(a, b), (dtype, ops_bits, t)
                assert torch.equal(ra.done, rb.done) and torch.equal(ra.reward, rb.reward), (dtype, ops_bits, t)
                assert torch.equal(ra.num_points, rb.num_points), (dtype, ops_bits, t)
                if t % 5 == 3:
                    idx = torch.from_numpy(rng.permutation(B)[:B // 40]).cuda()  # distinct games
                    fresh = rng.integers(-3, 9, (B // 40, N, d)).astype(np.int32)
                    dead = fresh[:, :, 0] < 0
                    fresh[dead] = -5                       # dead rows that are not the padding value
                    fresh[~dead] = np.maximum(fresh[~dead], 0)
                    fresh = torch.from_numpy(fresh).cuda().to(dtype)
                    a[idx] = fresh
                    b[idx] = fresh


F_ALL, F_ZEIL, F_FIRST, F_LAST = 1 << 8, 1 << 9, 1 << 10, 1 << 11


@pytest.mark.parametrize("shape", [(300, 20, 3), (200, 10, 3), (100, 5, 3), (64, 16, 4), (40, 64, 5), (30, 40, 2)],
                         ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
def test_fixed_players(hb, family, shape, dtype):
    """Hosts all_coord / Zeillinger and agents choose_first / choose_last evaluated in the kernel
    (hironaka/jax/players.py:42-105,156-212) against the C port, step by step and as one launch."""
    from hironaka_b200 import ops
    B, N, d = shape
    rng = np.random.default_rng(N + d)
    x0 = random_state(rng, B, N, d, 12, dead_frac=0.3, dup_frac=0.1).astype(dtype)
    ncls = 2 ** d - d - 1
    op_bits = O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON
    for pol in (F_ALL | F_FIRST, F_ALL | F_LAST, F_ZEIL | F_FIRST, F_ZEIL | F_LAST, F_ZEIL, F_FIRST, F_LAST):
        Tn = 5
        ha = rng.integers(0, ncls, (Tn, B)).astype(np.int32)
        ax = rng.integers(0, d, (Tn, B)).astype(np.int32)
        host_fixed, agent_fixed = pol & (F_ALL | F_ZEIL), pol & (F_FIRST | F_LAST)
        # JAX semantics, and the torch ones (invalid action = no-op, ended games frozen) on every other policy
        flags = pol | O.F_ACT_DISCRETE | (TORCH_FLAGS if (pol >> 8) % 2 else 0)
        o, g = x0, dev(x0)
        counts = []
        for t in range(Tn):
            o, od, orw, onp = cport.step(o, None if host_fixed else ha[t], None if agent_fixed else ax[t], op_bits, flags)
            r = ops.step(g, None if host_fixed else dev(ha[t]), None if agent_fixed else dev(ax[t]), ops=op_bits,
                         flags=flags, inplace=True, want_done=True, want_reward=True)
            assert np.array_equal(g.cpu().numpy(), o), (pol, t)
            assert np.array_equal(r.done.cpu().numpy(), od.astype(bool)) and np.array_equal(r.reward.cpu().numpy(), orw)
            counts.append(int(od.sum()))
        out, _, _, dcount, _ = ops.rollout(dev(x0), None if host_fixed else dev(ha), None if agent_fixed else dev(ax),
                                           ops=op_bits, flags=flags, inplace=False, steps=Tn)
        assert np.array_equal(out.cpu().numpy(), o) and dcount.tolist() == counts, pol


def test_zeillinger_kat(hb, family):
    """Zeillinger known answers of test/testJAX.py:232-268 through a kernel step: the chosen
    coordinates are read off the shifted point (x_a <- sum over the chosen set, agent = first)."""
    from hironaka_b200 import ops
    def chosen_mask(pts):
        p = pts.astype(np.float32)[None]
        got = ops.step(dev(p), ops=O.OP_SHIFT, flags=F_ZEIL | F_FIRST, inplace=False).state.cpu().numpy()[0]
        exp_oh = O.zeillinger_fn_slice(pts.astype(np.float32))
        mb = O.decode_table(pts.shape[1])[int(exp_oh.argmax())]
        a = int(np.argmax(mb))
        ref = pts.astype(np.float32).copy()
        live = ref[:, 0] >= 0
        ref[live, a] = (ref[live] * mb[None]).sum(1)
        assert np.array_equal(got, ref)
        return mb
    assert chosen_mask(K.ZEIL_PTS).tolist() == [1, 0, 1]                      # one-hot [0,1,0,0] = id 1 = {0,2}
    for pts, mb in zip(K.ZEIL_OBS2, K.ZEIL_OBS2_MB):
        assert chosen_mask(pts).tolist() == mb.tolist()
    assert chosen_mask(K.ZEIL_PTS3[0]).tolist() == [1, 0, 1]


def test_float_state_rescaled_rollout(hb, family):
    """DQN path with scale_observation: float state divided by its max every step
    (fused_game.py:160-162).  Values are non-integers; parity is exact because the kernel keeps
    the reference's left-to-right summation and IEEE division."""
    rng = np.random.default_rng(5)
    B, N, d = 200, 20, 3
    x = rng.integers(0, 21, size=(B, N, d)).astype(np.float32)
    ops_bits = O.OP_SHIFT | O.OP_NEWTON | O.OP_RESCALE
    flags = TORCH_FLAGS | O.F_ACT_DISCRETE
    g = run_step(hb, x, None, None, O.OP_NEWTON | O.OP_RESCALE, 0)[0]
    o = cport.step(x, None, None, O.OP_NEWTON | O.OP_RESCALE, 0)[0]
    assert np.array_equal(g, o)
    for t in range(6):
        ha, ax = rng.integers(0, 4, B), rng.integers(0, 3, B)
        g = run_step(hb, g, ha, ax, ops_bits, flags)[0]
        o = cport.step(o, ha, ax, ops_bits, flags)[0]
        assert np.array_equal(g, o), t


def test_padding_value_and_inplace(hb, family):
    from hironaka_b200 import ops
    rng = np.random.default_rng(11)
    x = random_state(rng, 70, 10, 3, 9).astype(np.float32)
    x[x < 0] = -1e-8  # padding used by test/testTrainer.py:77
    ha, ax = rng.integers(0, 8, 70), rng.integers(0, 3, 70)
    got = run_step(hb, x, ha, ax, O.OP_SHIFT | O.OP_NEWTON, TORCH_FLAGS, pad=-1e-8)[0]
    exp = cport.step(x, ha, ax, O.OP_SHIFT | O.OP_NEWTON, TORCH_FLAGS, padding_value=-1e-8)[0]
    assert np.array_equal(got, exp)
    t = dev(x)
    r = ops.step(t, dev(ha.astype(np.int32)), dev(ax.astype(np.int32)), ops=O.OP_SHIFT | O.OP_NEWTON,
                 flags=TORCH_FLAGS, padding_value=-1e-8, inplace=True)
    assert r.state.data_ptr() == t.data_ptr() and np.array_equal(t.cpu().numpy(), exp)
    # unaligned base pointer (4-byte aligned only): the non-TMA path must give the same answer
    buf = torch.zeros(70 * 30 + 1, dtype=torch.float32, device="cuda")
    view = buf[1:].view(70, 10, 3)
    view.copy_(dev(x))
    assert view.data_ptr() % 16 != 0
    ops.step(view, dev(ha.astype(np.int32)), dev(ax.astype(np.int32)), ops=O.OP_SHIFT | O.OP_NEWTON,
             flags=TORCH_FLAGS, padding_value=-1e-8, inplace=True)
    assert np.array_equal(view.cpu().numpy(), exp)


def test_exceed_flag_and_errors(hb):
    from hironaka_b200 import ops
    from hironaka_b200._lib import HironakaB200Error
    x = dev(np.array([[[1, 2, 3], [5, 0, 70000]]], dtype=np.int32))
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.step(x, ops=0, write_state=False, exceed_flag=flag, value_threshold=1e5)
    assert flag.item() == 0
    ops.step(x, ops=0, write_state=False, exceed_flag=flag, value_threshold=7e4)
    assert flag.item() == 1
    with pytest.raises(HironakaB200Error):
        ops.step(torch.zeros(2, 3, 3, dtype=torch.int32), ops=O.OP_NEWTON)  # CPU tensor: no fallback
    with pytest.raises(HironakaB200Error):
        ops.step(x, ops=O.OP_RESCALE)  # rescale is undefined on int32 state
    with pytest.raises(HironakaB200Error):
        ops.step(torch.zeros(1, 2, 11, dtype=torch.int32, device="cuda"), ops=O.OP_NEWTON)  # d > HK_MAX_DIM
    with pytest.raises(ValueError):
        ops.step(x, ops=O.OP_SHIFT)  # missing actions
    e = torch.zeros(0, 20, 3, dtype=torch.int32, device="cuda")
    assert ops.step(e, ops=O.OP_NEWTON, want_done=True).done.numel() == 0  # empty batch


def test_config4_ade_starts_dqn_replay(hb):
    """BASELINE config 4: the six ADE start configurations (search.py:123-128) padded to N = 5 and
    replicated to B = 4096 with independent action streams, FusedGame semantics (shift -> newton ->
    rescale; invalid action = no-op, ended games frozen), experiences of the games that were not over
    appended in order to a replay buffer — state, done, reward and buffer contents vs the oracle."""
    from hironaka_b200 import ReplayBuffer, ops
    B, N, d, Tn = 4096, 5, 3, 10
    rng = np.random.default_rng(44)
    x = -np.ones((B, N, d), np.float32)
    x[:, :3] = K.ADE_STARTS[rng.integers(0, 6, B)]
    for scale in (False, True):
        op_bits = O.OP_SHIFT | O.OP_NEWTON | (O.OP_RESCALE if scale else 0)
        flags = TORCH_FLAGS | O.F_ACT_DISCRETE
        o = cport.step(x, None, None, O.OP_NEWTON | (O.OP_RESCALE if scale else 0), 0)[0]
        g = dev(x)
        ops.step(g, ops=O.OP_NEWTON | (O.OP_RESCALE if scale else 0), inplace=True)
        assert np.array_equal(g.cpu().numpy(), o)
        buf = ReplayBuffer((N, d), 4, 1 << 15, torch.device("cuda"))
        ref_obs, ref_act, ref_rew, ref_done, ref_next = [], [], [], [], []
        for t in range(Tn):
            ha = rng.integers(0, 4, B).astype(np.int32)
            ax = rng.integers(0, 3, B).astype(np.int32)
            obs_before = cport.features(o, O.F_OBS_SORT_COORD0).reshape(B, N, d)
            prev_done = O.ended_batch(o)
            feat_before = ops.features(g, flags=O.F_OBS_SORT_COORD0).view(B, N, d)
            skip = ops.dones(g)[0]
            r = ops.step(g, dev(ha), dev(ax), ops=op_bits, flags=flags, inplace=True, want_done=True, want_reward=True,
                         want_obs=True)
            o, od, orw, _ = cport.step(o, ha, ax, op_bits, flags)
            assert np.array_equal(g.cpu().numpy(), o), (scale, t)
            assert np.array_equal(r.done.cpu().numpy(), od.astype(bool)) and np.array_equal(r.reward.cpu().numpy(), orw)
            assert np.array_equal(skip.cpu().numpy(), prev_done)
            next_feat = ops.features(g, flags=O.F_OBS_SORT_COORD0).view(B, N, d)
            buf.add_masked(skip, feat_before, dev(ha), r.reward, r.done, next_feat)
            keep = ~prev_done
            ref_obs.append(obs_before[keep]); ref_act.append(ha[keep]); ref_rew.append(orw[keep])
            ref_done.append(od.astype(bool)[keep]); ref_next.append(cport.features(o, O.F_OBS_SORT_COORD0).reshape(B, N, d)[keep])
        n = sum(len(a) for a in ref_act)
        assert buf.pos == n and not buf.full and n > 0
        assert np.array_equal(buf.observations[:n].cpu().numpy(), np.concatenate(ref_obs))
        assert np.array_equal(buf.next_observations[:n].cpu().numpy(), np.concatenate(ref_next))
        assert np.array_equal(buf.actions[:n, 0].cpu().numpy(), np.concatenate(ref_act))
        assert np.array_equal(buf.rewards[:n, 0].cpu().numpy(), np.concatenate(ref_rew))
        assert np.array_equal(buf.dones[:n, 0].cpu().numpy(), np.concatenate(ref_done))


# ---------------------------------------------------------------- BASELINE sizes


@pytest.mark.parametrize("cfg", [
    dict(name="C2", B=1 << 20, N=20, d=3, T=20, mv=20, ops=O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, flags=O.F_ACT_DISCRETE),
    dict(name="C1", B=1024, N=10, d=3, T=10, mv=21, ops=O.OP_SHIFT | O.OP_NEWTON, flags=TORCH_FLAGS | O.F_ACT_DISCRETE),
    # exactly the configuration bench.py times for C5: the HOT instantiation of the warp-per-game kernel
    # (shift + reposition + newton, discrete ids), every resident warp playing ~55 games in a row
    dict(name="C5", B=1 << 18, N=64, d=5, T=20, mv=20, ops=O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, flags=O.F_ACT_DISCRETE),
    dict(name="C5-norepos", B=1 << 16, N=64, d=5, T=6, mv=20, ops=O.OP_SHIFT | O.OP_NEWTON, flags=O.F_ACT_DISCRETE),
    # the warp-per-game family on the (20,3) shape at a size where its game loop iterates many times
    dict(name="C2-generic", B=1 << 16, N=20, d=3, T=20, mv=20, ops=O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON,
         flags=O.F_ACT_DISCRETE, generic=True),
], ids=lambda c: c["name"])
def test_baseline_sizes_bit_exact(hb, cfg):
    """Full-size parity against the C port on identical seeded inputs (SURVEY.md section 8d)."""
    from hironaka_b200 import ops
    B, N, d, T = cfg["B"], cfg["N"], cfg["d"], cfg["T"]
    ops.force_generic(bool(cfg.get("generic")))
    rng = np.random.default_rng(2024)
    x = rng.integers(0, cfg["mv"], size=(B, N, d)).astype(np.int32)
    ncls = 2 ** d - d - 1
    ha = rng.integers(0, ncls, size=(T, B)).astype(np.int32)
    ax = rng.integers(0, d, size=(T, B)).astype(np.int32)
    init_ops = O.OP_NEWTON | (cfg["ops"] & O.OP_REPOSITION)
    o = cport.step(x, None, None, init_ops, 0)[0]
    g = dev(x)
    ops.step(g, ops=init_ops, inplace=True)
    assert np.array_equal(g.cpu().numpy(), o)
    g_roll = g.clone()
    odones = []
    for t in range(T):
        o, od, orw, _ = cport.step(o, ha[t], ax[t], cfg["ops"], cfg["flags"])
        r = ops.step(g, dev(ha[t]), dev(ax[t]), ops=cfg["ops"], flags=cfg["flags"], inplace=True, want_done=True,
                     want_reward=True)
        odones.append(od.astype(bool))
        assert np.array_equal(r.done.cpu().numpy(), od.astype(bool)), t
        assert np.array_equal(r.reward.cpu().numpy(), orw), t
        if t in (0, 1, T - 1) or t % 5 == 4:
            assert np.array_equal(g.cpu().numpy(), o), t
    # one-launch rollout ends in the same state with the same per-step finished counts
    _, _, _, dcount, _ = ops.rollout(g_roll, dev(ha), dev(ax), ops=cfg["ops"], flags=cfg["flags"], inplace=True)
    assert np.array_equal(g_roll.cpu().numpy(), o)
    assert np.array_equal(dcount.cpu().numpy(), np.stack(odones).sum(1))
    # size-independent properties: the filter is idempotent; survivors are pairwise incomparable
    g2 = g.clone()
    ops.step(g2, ops=O.OP_NEWTON, inplace=True)
    assert torch.equal(g2, g)
    ops.force_generic(False)


# ---------------------------------------------------------------- the reference's own JAX sources


@pytest.mark.parametrize("dtype", [np.float32, np.int32])
def test_jax_golden_rollouts(hb, family, golden_dir, dtype):
    """Rollouts produced by EXECUTING the reference's JAX sources (hironaka/src/_jax_ops.py,
    hironaka/jax/util.py; oracle/gen_golden_jax.py): take_actions -> get_dones -> reward_fn -> feature_fn,
    host and agent roles, with / without reposition, rescaled float states, step by step and as one launch."""
    from hironaka_b200 import ops
    files = sorted(glob.glob(os.path.join(golden_dir, "ref_jax_rollout_*.npz")))
    assert len(files) >= 8
    for path in files:
        g = np.load(path)
        seed, B, N, d, T, mv, agent, repos, resc = g["meta"].tolist()
        if resc and dtype == np.int32:
            continue
        ops_bits = O.OP_SHIFT | O.OP_NEWTON | (O.OP_REPOSITION if repos else 0) | (O.OP_RESCALE if resc else 0)
        flags = O.F_ACT_DISCRETE | O.F_RESCALE_EPS | (O.F_ROLE_AGENT if agent else 0)
        root = O.OP_NEWTON | (O.OP_REPOSITION if repos else 0) | (O.OP_RESCALE if resc else 0)
        x, done, _, _, _ = run_step(hb, g["raw"].astype(dtype), None, None, root, flags)
        assert np.array_equal(x.astype(np.float32), g["states"][0]), path
        assert np.array_equal(done, g["dones"][0]), path
        x0 = x
        for t in range(T):
            hid, ax = g["host_ids"][t], g["axes"][t]
            x, done, rew, npts, obs = run_step(hb, x, hid, ax, ops_bits, flags | O.F_OBS_SORT_LEX | O.F_OBS_RESCALE,
                                               want_obs=True)
            assert np.array_equal(x.astype(np.float32), g["states"][t + 1]), (path, t)
            assert np.array_equal(done, g["dones"][t + 1]), (path, t)
            assert np.array_equal(rew, g["rewards"][t]), (path, t)
            assert np.array_equal(obs, g["feat_host"][t]), (path, t)
            raw = run_step(hb, x, None, None, 0, flags | O.F_OBS_SORT_LEX, want_obs=True)[4]
            assert np.array_equal(raw, g["feat_host_raw"][t]), (path, t)
            fa = run_step(hb, x, None, None, 0, flags | O.F_OBS_SORT_LEX | O.F_OBS_RESCALE, want_obs=True, obs_coord=hid)[4]
            assert np.array_equal(fa, g["feat_agent"][t]), (path, t)
        out, dn, rw, dcount, _ = ops.rollout(dev(x0), dev(g["host_ids"]), dev(g["axes"]), ops=ops_bits, flags=flags,
                                             inplace=False, want_done=True, want_reward=True)
        assert np.array_equal(out.cpu().numpy().astype(np.float32), g["states"][T]), path
        assert np.array_equal(dn.cpu().numpy(), g["dones"][1:]), path
        assert np.array_equal(rw.cpu().numpy(), g["rewards"]), path
        assert np.array_equal(dcount.cpu().numpy(), g["dones"][1:].sum(1)), path


def test_jax_golden_functional_api(hb, golden_dir):
    """The same goldens through the drop-in functional API (hironaka_b200.functional = hironaka/jax/util.py)."""
    from hironaka_b200 import functional as F
    g = np.load(os.path.join(golden_dir, "ref_jax_rollout_c2_20x3.npz"))
    seed, B, N, d, T, *_ = g["meta"].tolist()
    take = F.get_take_actions("host", (N, d), False, True)
    feat = F.get_feature_fn("host", (N, d), True)
    afeat = F.get_feature_fn("agent", (N, d), True)
    rewf = F.get_reward_fn("host")
    decode = F.get_batch_decode(d)
    x = dev(g["states"][0])
    prev = F.get_dones(x)
    for t in range(T):
        coords = decode(dev(g["host_ids"][t]))
        nxt = take(F.flatten(x), coords, dev(g["axes"][t]))
        assert np.array_equal(nxt.cpu().numpy(), g["states"][t + 1].reshape(B, -1)), t
        x = nxt.reshape(B, N, d)
        dn = F.get_dones(x)
        assert np.array_equal(dn.cpu().numpy(), g["dones"][t + 1]), t
        assert np.array_equal(rewf(dn, prev).cpu().numpy(), g["rewards"][t]), t
        assert np.array_equal(feat(nxt).cpu().numpy(), g["feat_host"][t]), t
        aobs = F.make_agent_obs(x, coords)
        assert np.array_equal(afeat(aobs).cpu().numpy(), g["feat_agent"][t]), t
        assert np.array_equal(F.get_done_from_flatten(aobs, "agent", d).cpu().numpy(), g["done_from_flatten"][t][1]), t
        prev = dn
    # the agent role reads its coordinates from the observation (util.py:66-75)
    ga = np.load(os.path.join(golden_dir, "ref_jax_rollout_c2_20x3_agent.npz"))
    _, B, N, d, T, *_ = ga["meta"].tolist()
    take_a = F.get_take_actions("agent", (N, d), False, True)
    x = dev(ga["states"][0])
    for t in range(T):
        coords = decode(dev(ga["host_ids"][t]))
        ax = dev(ga["axes"][t])
        nxt = take_a(F.make_agent_obs(x, coords), ax, ax)
        assert np.array_equal(nxt.cpu().numpy(), ga["states"][t + 1].reshape(B, -1)), t
        x = nxt.reshape(B, N, d)
    # select_sample_after_sim: the deterministic part is the reference's, the random part keeps its contract
    gs = np.load(os.path.join(golden_dir, "ref_jax_select_after_sim.npz"))
    for role, key in (("host", "host_obs"), ("agent", "agent_obs")):
        ro = (dev(gs[key]), None, None)
        und = F.select_sample_after_sim(role, ro, 3, mix_random_terminal_states=False)
        assert np.array_equal(und.cpu().numpy(), gs[f"undone_{role}"])
        gen = torch.Generator(device="cuda").manual_seed(3)
        sel = F.select_sample_after_sim(role, ro, 3, mix_random_terminal_states=True, generator=gen)
        assert bool((sel | ~und).all()) and int(sel.sum()) <= 2 * int(und.sum())
        assert int(sel.sum()) >= int(und.sum())


@pytest.mark.parametrize("dtype", [np.float32, np.int32])
def test_jax_golden_ops(hb, family, golden_dir, dtype):
    for path in sorted(glob.glob(os.path.join(golden_dir, "ref_jax_ops_*.npz"))):
        g = np.load(path)
        x = g["points"].astype(dtype)
        B, N, d = x.shape
        cm = (g["coord"].astype(np.int64) * (1 << np.arange(d))).sum(1).astype(np.int32)
        c = lambda a: a.astype(np.float32)
        assert np.array_equal(c(run_step(hb, x, cm, g["axes"], O.OP_SHIFT, 0)[0]), g["shift"]), path
        assert np.array_equal(c(run_step(hb, x, None, None, O.OP_REPOSITION, 0)[0]), g["reposition"]), path
        assert np.array_equal(c(run_step(hb, x, None, None, O.OP_DEDUPE, 0)[0]), g["remove_repeated"]), path
        assert np.array_equal(c(run_step(hb, x, None, None, O.OP_NEWTON, 0)[0]), g["newton"]), path
        if dtype == np.float32:
            assert np.array_equal(run_step(hb, x, None, None, O.OP_RESCALE, O.F_RESCALE_EPS)[0], g["rescale"]), path
            # calculate_rescale's eps rule (_jax_ops.py:93-98): maxima <= 1e-8 leave the game alone
            tiny = g["tiny_points"]
            assert np.array_equal(run_step(hb, tiny, None, None, O.OP_RESCALE, O.F_RESCALE_EPS)[0], g["tiny_rescale"]), path
            obs = run_step(hb, tiny, None, None, 0, O.F_OBS_RESCALE | O.F_RESCALE_EPS, want_obs=True)[4]
            assert np.array_equal(obs.reshape(B, N, d), g["tiny_rescale"]), path
            assert np.array_equal(run_step(hb, tiny, None, None, O.OP_RESCALE, 0)[0],
                                  cport.step(tiny, None, None, O.OP_RESCALE, 0)[0]), path


@pytest.mark.parametrize("N", [5, 10, 20])
def test_features_pack_borders(hb, family, N):
    """The observation kernel packs a whole row into one 32-bit key while every live value is an integer
    below 2^9 (d = 3), into a 64-bit key below 2^19, and compares floats beyond: values that straddle
    511/512 and 2^19 - 1 / 2^19, alone and mixed inside one warp tile, with ties on every coordinate."""
    rng = np.random.default_rng(N)
    B, d = 96, 3
    for lo, hi in ((509, 514), (0, 513), ((1 << 19) - 3, (1 << 19) + 3), (510, (1 << 19) + 2)):
        base = rng.integers(lo, hi, size=(B, N, d))
        pick = rng.random((B, N, d)) < 0.5
        x = np.where(pick, base, rng.integers(0, 4, size=(B, N, d))).astype(np.int32)
        x[rng.random((B, N)) < 0.3] = -1
        x[::7] = np.where(x[::7] >= 0, np.minimum(x[::7], 511), -1)       # games that stay packable next to ones that do not
        x[3::11, :, 2] = np.where(x[3::11, :, 0] >= 0, 512, -1)           # the border value in the primary sort column
        for dtype in (np.int32, np.float32):
            xv = x.astype(dtype)
            for flags in (O.F_OBS_SORT_LEX, O.F_OBS_SORT_LEX | O.F_OBS_RESCALE, O.F_OBS_SORT_COORD0, 1 << 12,
                          O.F_OBS_SORT_COORD0 | O.F_OBS_RESCALE):
                got = run_step(hb, xv, None, None, 0, flags, want_obs=True)[4]
                assert np.array_equal(got, cport.features(xv, flags)), (lo, hi, dtype, flags)


# ---------------------------------------------------------------- the census step


CENSUS_FLAVOURS = {
    "jax": (O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, O.F_ACT_DISCRETE),
    "torch-agent": (O.OP_SHIFT | O.OP_NEWTON, TORCH_FLAGS | O.F_ACT_DISCRETE | O.F_ROLE_AGENT),
    "no-reposition": (O.OP_SHIFT | O.OP_NEWTON, O.F_ACT_DISCRETE),
}


def census_rollout_inputs(B, N, d, dtype, T=14):
    """The start state and, per flavour of CENSUS_FLAVOURS (in that order), the T steps' actions and the games the
    caller rewrites after steps 2, 6 and 10 (None elsewhere): all drawn from one generator seeded with B + N."""
    rng = np.random.default_rng(B + N)
    x0 = random_state(rng, B, N, d, max_value=9, dead_frac=0.45, dup_frac=0.1).astype(dtype)
    junk = rng.random((B, N)) < 0.3
    x0[(x0[:, :, 0] < 0) & junk] = -7
    x0[::5] = -1
    x0[1::5, 1:] = -1
    x0[1::5, 0] = np.abs(x0[1::5, 0])
    ncls = 2 ** d - d - 1
    steps = {}
    for name in CENSUS_FLAVOURS:
        steps[name] = []
        for t in range(T):
            ha = rng.integers(0, ncls, B).astype(np.int32)
            ax = rng.integers(0, d, B).astype(np.int32)
            rewrite = None
            if t % 4 == 2:
                idx = rng.permutation(B)[:max(1, B // 30)]
                fresh = random_state(rng, len(idx), N, d, max_value=7, dead_frac=0.3).astype(dtype)
                fresh[(fresh[:, :, 0] < 0) & (rng.random((len(idx), N)) < 0.5)] = -3
                rewrite = (idx, fresh)
            steps[name].append((ha, ax, rewrite))
    return x0, steps


@pytest.mark.parametrize("shape", [(40003, 20, 3), (2500, 10, 3), (1111, 5, 3), (31, 20, 3), (3000, 64, 5), (700, 16, 4),
                                   (5003, 33, 3), (900, 40, 2), (300, 100, 3)],
                         ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
@pytest.mark.parametrize("flavour", list(CENSUS_FLAVOURS))
def test_census_step_equals_oracle(hb, shape, dtype, flavour):
    """hk_step_census over whole rollouts: games at rest are answered from their census byte, games in play
    are reordered by live count — state, done, reward, num_points and the finished count must equal the
    oracle's after EVERY step, for both flavours, from starts with junk in dead rows, empty games and
    lone points, with the caller rewriting games (and zeroing their census bytes) along the way.  The three
    flavours of a shape and dtype share one input stream (census_rollout_inputs), each case plays its part."""
    from hironaka_b200 import ops
    B, N, d = shape
    ops_bits, flags = CENSUS_FLAVOURS[flavour]
    x0, steps = census_rollout_inputs(B, N, d, dtype)
    o = x0.copy()
    g = dev(x0)
    census = ops.new_census(g)
    for t, (ha, ax, rewrite) in enumerate(steps[flavour]):
        o, od, orw, onp = cport.step(o, ha, ax, ops_bits, flags)
        dc = torch.zeros(1, dtype=torch.int32, device="cuda")
        r = ops.step(g, dev(ha), dev(ax), ops=ops_bits, flags=flags, inplace=True, want_done=True, want_reward=True,
                     want_num_points=True, census=census, done_count=dc)
        assert np.array_equal(g.cpu().numpy(), o), (ops_bits, flags, t)
        assert np.array_equal(r.done.cpu().numpy(), od.astype(bool)), (ops_bits, flags, t)
        assert np.array_equal(r.reward.cpu().numpy().view(np.int32), orw.view(np.int32)), (ops_bits, flags, t)
        assert np.array_equal(r.num_points.cpu().numpy(), onp), (ops_bits, flags, t)
        assert int(dc.item()) == int(od.sum()), (ops_bits, flags, t)
        if rewrite is not None:  # the caller rewrites some games and zeroes their census bytes
            idx, fresh = rewrite
            o[idx] = fresh
            ti = torch.from_numpy(idx).cuda()
            g[ti] = dev(fresh)
            census[ti] = 0
    c = census.cpu().numpy()[:B]
    live = (o[:, :, 0] >= 0).sum(1)
    known = c != 0
    assert np.array_equal(np.where(c[known] & 0x80, c[known] & 1, c[known]), live[known]), "census counts"
    if hb.ops.kernel_class(N, d) == 1:
        assert known.all()
    if census.numel() > B:  # large padded shape: the live masks of the known games name exactly the live rows
        masks = census.cpu().numpy()[(B + 7) // 8 * 8:].view(np.uint64)
        want = ((o[:, :, 0] >= 0).astype(np.uint64) << np.arange(N, dtype=np.uint64)[None, :]).sum(1, dtype=np.uint64)
        assert np.array_equal(masks[known], want[known]), "census masks"


def test_census_step_baseline_size(hb):
    """C2 at full size (1 Mi games, 20 steps) through hk_step_census against the C port, root filter included;
    in a reposition rollout every finished game ends at rest, so the last steps read almost nothing."""
    from hironaka_b200 import ops
    B, N, d, T = 1 << 20, 20, 3, 20
    rng = np.random.default_rng(77)
    x = rng.integers(0, 20, size=(B, N, d)).astype(np.int32)
    ha = rng.integers(0, 4, size=(T, B)).astype(np.int32)
    ax = rng.integers(0, d, size=(T, B)).astype(np.int32)
    step_ops = O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON
    o = cport.step(x, None, None, O.OP_NEWTON | O.OP_REPOSITION, 0)[0]
    g = dev(x)
    census = ops.new_census(g)
    ops.step(g, ops=O.OP_NEWTON | O.OP_REPOSITION, inplace=True, census=census)
    assert np.array_equal(g.cpu().numpy(), o)
    for t in range(T):
        o, od, orw, _ = cport.step(o, ha[t], ax[t], step_ops, O.F_ACT_DISCRETE)
        r = ops.step(g, dev(ha[t]), dev(ax[t]), ops=step_ops, flags=O.F_ACT_DISCRETE, inplace=True, want_done=True,
                     want_reward=True, census=census)
        assert np.array_equal(r.done.cpu().numpy(), od.astype(bool)), t
        assert np.array_equal(r.reward.cpu().numpy(), orw), t
        if t in (0, 1, 7, T - 1):
            assert np.array_equal(g.cpu().numpy(), o), t
    c = census.cpu().numpy()[:B]
    at_rest = (c & 0x82) == 0x82
    assert np.array_equal(at_rest, od.astype(bool)) and at_rest.mean() > 0.99


@pytest.mark.parametrize("shape", [(20011, 20, 3), (3001, 10, 3), (777, 5, 3), (31, 20, 3)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
def test_census_step_with_observation(hb, shape, dtype):
    """hk_step_census_obs: the census step with the fused observation.  Games at rest get their constant
    observation from the census byte, games in play run the feature code — every row of `obs` must equal the
    oracle's features of the new state after EVERY step of a whole rollout, for the three sorted modes, host and
    agent form (coordinates appended), with and without rescaling, with caller rewrites in between."""
    from hironaka_b200 import ops
    from hironaka_b200._lib import HironakaB200Error
    B, N, d = shape
    rng = np.random.default_rng(B + 7)
    T = 12
    x0 = random_state(rng, B, N, d, max_value=9, dead_frac=0.4, dup_frac=0.1).astype(dtype)
    x0[::5] = -1
    x0[1::5, 1:] = -1
    x0[1::5, 0] = np.abs(x0[1::5, 0])
    ncls = 2 ** d - d - 1
    op_bits = O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON
    for fflags, with_coord in ((O.F_OBS_SORT_LEX | O.F_OBS_RESCALE, False), (O.F_OBS_SORT_LEX | O.F_OBS_RESCALE, True),
                               (O.F_OBS_SORT_COORD0, False), (1 << 12, True)):
        flags = O.F_ACT_DISCRETE | fflags
        o = x0.copy()
        g = dev(x0)
        census = ops.new_census(g)
        for t in range(T):
            ha = rng.integers(0, ncls, B).astype(np.int32)
            ax = rng.integers(0, d, B).astype(np.int32)
            oc = rng.integers(0, ncls, B).astype(np.int32) if with_coord else None
            o, od, orw, _ = cport.step(o, ha, ax, op_bits, flags)
            r = ops.step(g, dev(ha), dev(ax), ops=op_bits, flags=flags, inplace=True, want_done=True, want_reward=True,
                         want_obs=True, obs_coord=None if oc is None else dev(oc), census=census)
            assert np.array_equal(g.cpu().numpy(), o), (fflags, t)
            assert np.array_equal(r.done.cpu().numpy(), od.astype(bool)) and np.array_equal(r.reward.cpu().numpy(), orw)
            assert np.array_equal(r.obs.cpu().numpy(), cport.features(o, flags, obs_coord=oc)), (fflags, with_coord, t)
            if t == 5:
                idx = rng.permutation(B)[:max(1, B // 20)]
                fresh = random_state(rng, len(idx), N, d, max_value=600, dead_frac=0.3).astype(dtype)  # values past the pack border
                o[idx] = fresh
                ti = torch.from_numpy(idx).cuda()
                g[ti] = dev(fresh)
                census[ti] = 0
    with pytest.raises(HironakaB200Error):  # an unsorted observation of a game at rest is not a constant
        ops.step(dev(x0), dev(np.zeros(B, np.int32)), dev(np.zeros(B, np.int32)), ops=op_bits, flags=O.F_ACT_DISCRETE,
                 inplace=True, want_obs=True, census=ops.new_census(dev(x0)))


@pytest.mark.parametrize("shape", [(3001, 20, 3), (1001, 10, 3), (600, 64, 5)], ids=lambda s: "x".join(map(str, s)))
def test_census_step_unaligned_buffers(hb, shape):
    """The census step on a state that is only 4-byte aligned and a census that is only 1-byte aligned: the bulk /
    cp.async fast paths must step aside for the word and byte copies, with the same results."""
    from hironaka_b200 import ops
    from hironaka_b200._lib import check, lib
    B, N, d = shape
    rng = np.random.default_rng(B)
    x0 = random_state(rng, B, N, d, max_value=9, dead_frac=0.4).astype(np.int32)
    buf = torch.zeros(B * N * d + 1, dtype=torch.int32, device="cuda")
    g = buf[1:].view(B, N, d)
    g.copy_(dev(x0))
    assert g.data_ptr() % 16 != 0
    nbytes = lib().hk_census_bytes(B, N, d)
    cbuf = torch.zeros(nbytes + 9, dtype=torch.uint8, device="cuda")
    off = 1 if nbytes == B else 8  # (the live masks after the bytes need their 8-byte alignment)
    census = cbuf[off:off + nbytes]
    o = x0
    ncls = 2 ** d - d - 1
    op_bits = O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON
    for t in range(10):
        ha = rng.integers(0, ncls, B).astype(np.int32)
        ax = rng.integers(0, d, B).astype(np.int32)
        o, od, orw, _ = cport.step(o, ha, ax, op_bits, O.F_ACT_DISCRETE)
        dn = torch.empty(B, dtype=torch.uint8, device="cuda")
        rw = torch.empty(B, dtype=torch.float32, device="cuda")
        ha_d, ax_d = dev(ha), dev(ax)  # (kept alive: a temporary's block would be handed to the next temporary)
        check(lib().hk_step_census(g.data_ptr(), ha_d.data_ptr(), ax_d.data_ptr(), dn.data_ptr(), None, rw.data_ptr(), None,
                                   census.data_ptr(), None, None, B, N, d, 0, op_bits, O.F_ACT_DISCRETE, -1.0, 1e8,
                                   torch.cuda.current_stream().cuda_stream))
        assert np.array_equal(g.cpu().numpy(), o), t
        assert np.array_equal(dn.cpu().numpy(), od) and np.array_equal(rw.cpu().numpy(), orw), t


@pytest.mark.parametrize("N", [5, 10, 20])
def test_packed_tier_borders(hb, N):
    """Single steps of int32 state take the packed tiers of the thread-per-game kernels while every live value of a
    warp's games fits one field after the shift (<= 255 for d = 3) and the exact tiers otherwise: values that
    straddle that border warp by warp and game by game, sums that land on 255 / 256, duplicates of every
    multiplicity, negative entries in live rows (never packed; filter-only calls), games with 0 / 1 / all rows live, junk in dead
    rows, both flavours, with and without reposition, with the exceed flag and with the census."""
    from hironaka_b200 import ops
    B, d = 4099, 3
    rng = np.random.default_rng(255 + N)
    ncls = 2 ** d - d - 1
    for trial, (ops_bits, flags) in enumerate([
        (O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, O.F_ACT_DISCRETE),
        (O.OP_SHIFT | O.OP_NEWTON, TORCH_FLAGS | O.F_ACT_DISCRETE | O.F_ROLE_AGENT),
        (O.OP_SHIFT | O.OP_NEWTON, 0),
        (O.OP_REPOSITION | O.OP_NEWTON, 0),
        (O.OP_NEWTON, 0),
    ]):
        x = np.empty((B, N, d), np.int32)
        # per warp of 32 games a value scale: tiny, just below the border (85 * 3 = 255), just above, large
        scale = np.repeat(rng.choice([3, 20, 85, 86, 128, 255, 256, 300, 70000], (B + 31) // 32), 32)[:B]
        x[:] = rng.integers(0, scale[:, None, None] + 1, (B, N, d))
        x[rng.random(B) < 0.3] //= 7                                  # small games inside large-valued warps
        hi = rng.random(B) < 0.15                                     # whole rows at the scale itself: sums on the border
        x[hi, : max(1, N // 2)] = scale[hi, None, None]
        dup = rng.integers(0, N, (B, 4))
        for k in range(3):                                            # duplicates, up to four copies of a row
            x[np.arange(B), dup[:, k + 1]] = x[np.arange(B), dup[:, 0]]
        dead = rng.random((B, N)) < rng.choice([0.0, 0.3, 0.7, 0.95], B)[:, None]
        x[dead] = -1
        x[dead & (rng.random((B, N)) < 0.2)] = -9                     # junk in dead rows
        x[::97] = -1                                                  # empty games
        if not ops_bits & O.OP_SHIFT:                                 # a negative entry in a live row (a shift could make
            neg = np.arange(B) % 53 == 7                              # coordinate 0 negative: not a state of the game)
            x[neg, 0, 0] = 4
            x[neg, 0, 1] = -2
        if flags & O.F_ACT_DISCRETE:
            ha = rng.integers(0, ncls, B)
        else:
            ha = rng.integers(0, 2 ** d, B)
        ax = rng.integers(0, d, B)
        got = run_step(hb, x, ha, ax, ops_bits, flags)
        exp = cport.step(x, ha, ax, ops_bits, flags)
        assert np.array_equal(got[0], exp[0]), (trial, "state")
        assert np.array_equal(got[1], exp[1].astype(bool)), (trial, "done")
        assert np.array_equal(got[2], exp[2]), (trial, "reward")
        assert np.array_equal(got[3], exp[3]), (trial, "num_points")
        # the exceed flag at a threshold inside the packed range, and the census route on the same inputs
        for thr in (40.0, 1e9):
            flag = torch.zeros(1, dtype=torch.int32, device="cuda")
            ops.step(dev(x), dev(ha.astype(np.int32)), dev(ax.astype(np.int32)), ops=ops_bits, flags=flags, inplace=True,
                     exceed_flag=flag, value_threshold=thr)
            live = exp[0][:, :, 0] >= 0
            assert bool(flag.item()) == bool((exp[0][live] >= thr).any()), (trial, thr)
        g = dev(x)
        census = ops.new_census(g)
        o = x
        for t in range(3):
            ha = rng.integers(0, ncls if flags & O.F_ACT_DISCRETE else 2 ** d, B).astype(np.int32)
            ax = rng.integers(0, d, B).astype(np.int32)
            o, od, orw, onp = cport.step(o, ha, ax, ops_bits, flags)
            r = ops.step(g, dev(ha), dev(ax), ops=ops_bits, flags=flags, inplace=True, want_done=True, want_reward=True,
                         want_num_points=True, census=census)
            assert np.array_equal(g.cpu().numpy(), o), (trial, t, "census state")
            assert np.array_equal(r.done.cpu().numpy(), od.astype(bool)) and np.array_equal(r.num_points.cpu().numpy(), onp)
            assert np.array_equal(r.reward.cpu().numpy().view(np.int32), orw.view(np.int32))
