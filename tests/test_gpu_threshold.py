"""Rollouts with a value threshold (hk_rollout_threshold) against the oracle's C port stepped once per step.

hk_rollout_threshold is hk_rollout_record that also follows every game against a value threshold: over_step[b] is 0
when a live entry of the input is already >= the threshold, t + 1 for the first step t after which one is, T + 1 when
none ever is; with stop_at_threshold a game that has crossed is not stepped again.  The expected trajectory is the C port
stepped once per step with a per-game freeze mask: a stopped game keeps its state (the input's with dead rows padded, or
the state after its crossing step), repeats its done flag, gets no reward, plays host mask 0 and axis -1.  For int32
states an int64 copy of every shift that is played bounds the values, so the reference itself stays exact.  Every output
is pre-filled with a sentinel and compared bit for bit; done_count is incremented from a nonzero start.

The tests without the gpu mark check the reference side: with nothing crossing it is the plain C-port trajectory, a
stopped rollout split in two is the same rollout, and at the int32 bound every stepped game stays below 2^30.
"""
import math

import numpy as np
import pytest

from hironaka_b200 import constants as C
from oracle import cport
from oracle import hk_oracle as O
from tests.test_gpu_record import (AGENT_FIXED, HOST_FIXED, RANDOM, agent_axes, mask_bits, oracle_record, replay_flags,
                                   zeillinger_masks)
from tests.test_gpu_rollout import (DONE_COUNT_BASE, F_ALL, F_FIRST, F_LAST, F_ZEIL, FUSED_STEP, INT32_BOUND, JAX_STEP,
                                    SEED, SENTINEL_REWARD, SENTINEL_WORD, STEP_OFFSET, SWEEP_SHAPES, TORCH_FLAGS, _dev,
                                    _filled, _stream, bits, decode_ids, lib, random_actions, shift_i64, start_state)

gpu = pytest.mark.gpu
_ = lib  # the module's library fixture

NAMES = ("state", "obs", "host_mask", "axis", "done", "reward", "done_count", "length", "over_step")


# ---------------------------------------------------------------- reference side (no GPU)


def crossed(x, thr):
    """Games with a live entry >= thr, compared as float32 (hk_overflow with strict = 0)."""
    live = x[:, :, :1] >= 0
    return ((x.astype(np.float32) >= np.float32(thr)) & live).any((1, 2))


def padded(x, pad):
    return np.where(x[:, :, :1] >= 0, x, x.dtype.type(pad))


def oracle_threshold(x, ha, ax, ops, flags, T, thr, stop, pad=-1.0, agent_obs=False, seed=0, step_offset=0):
    """T steps of the C port with a freeze mask: (state, obs [T, B, OW], host masks [T, B], axes [T, B], done [T, B],
    reward [T, B], finished games per step [T], length [B], over_step [B]).  Arguments as oracle_record's, plus the
    threshold and the stop flag.  int32: every shift that is played is redone on an int64 copy and must stay below 2^30
    (the games that are not stepped need no such bound)."""
    B, N, d = x.shape
    if flags & RANDOM:
        rha, rax = O.random_player_actions(B, d, T, seed, step_offset)
        if flags & C.HK_F_HOST_RANDOM:
            ha = rha
        if flags & C.HK_F_AGENT_RANDOM:
            ax = rax
    step_flags = flags & ~RANDOM
    discrete = flags & (C.HK_F_ACT_DISCRETE | C.HK_F_HOST_RANDOM)
    if flags & C.HK_F_HOST_RANDOM:
        step_flags |= C.HK_F_ACT_DISCRETE
    o = np.ascontiguousarray(x)
    length = np.where((o[:, :, 0] >= 0).sum(1) < 2, 0, T + 1).astype(np.int32)
    over = np.where(crossed(o, thr), 0, T + 1).astype(np.int32)
    obs, masks, axes = [], [], []
    done = np.empty((T, B), np.uint8)
    reward = np.empty((T, B), np.float32)
    for t in range(T):
        frozen = (over <= t) if stop else np.zeros(B, bool)
        if flags & F_ALL:
            cm = np.full(B, (1 << d) - 1, np.int32)
        elif flags & F_ZEIL:
            cm = zeillinger_masks(o)
        else:
            cm = decode_ids(ha[t], d) if discrete else np.asarray(ha[t], np.int32)
        a = agent_axes(cm, d, flags) if flags & AGENT_FIXED else np.asarray(ax[t], np.int32)
        played = np.where((o[:, :, 0] >= 0).any(1), cm, 0).astype(np.int32) if flags & HOST_FIXED else cm
        if not ops & C.HK_OP_SHIFT:
            played, a = np.zeros(B, np.int32), np.zeros(B, np.int32)
        played = np.where(frozen, 0, played).astype(np.int32)
        a = np.where(frozen, -1, a).astype(np.int32)
        f = cport.features(padded(o, pad), flags, padding_value=pad)
        obs.append(np.concatenate([f, mask_bits(played, d)], 1) if agent_obs else f)
        masks.append(played)
        axes.append(a)
        if o.dtype == np.int32 and ops & C.HK_OP_SHIFT:
            s = shift_i64(o[~frozen], cm[~frozen], a[~frozen], step_flags, pad)
            assert (np.where(s[:, :, :1] >= 0, s, 0) < INT32_BOUND).all(), ("int64 guard", t)
        n, dn, rw, _ = cport.step(o, None if ha is None else ha[t], None if ax is None else ax[t], ops, step_flags,
                                  padding_value=pad)
        n[frozen] = padded(o, pad)[frozen]
        dn[frozen] = ((o[frozen, :, 0] >= 0).sum(1) < 2).astype(np.uint8)
        rw[frozen] = -0.0 if flags & C.HK_F_ROLE_AGENT else 0.0
        o, done[t], reward[t] = n, dn, rw
        length[(length == T + 1) & (done[t] != 0)] = t + 1
        over[(over == T + 1) & crossed(o, thr)] = t + 1
    return (o, np.stack(obs), np.stack(masks), np.stack(axes), done, reward, done.sum(1).astype(np.int32), length, over)


def bound(d):
    """The largest float32 threshold <= floor(2^30 / d), the int32 bound of hk_rollout_threshold."""
    b = (1 << 30) // d
    f = np.float32(b)
    return float(np.nextafter(f, np.float32(0)) if int(f) > b else f)


def above_bound(d):
    return float(np.nextafter(np.float32(bound(d)), np.float32(np.inf)))


def near_bound_state(rng, B, N, d):
    """int32 games whose entries reach just below floor(2^30 / d) in some games and stay small in others: in a big game
    every live row holds one such entry, in a coordinate of its own choosing, so that the filter keeps several of them."""
    x = start_state(rng, B, N, d, np.int32, 30)
    big = rng.random(B) < 0.5
    hi = int(bound(d))
    vals = rng.integers(hi - hi // 4, hi, size=(B, N)).astype(np.int32)
    coord = rng.integers(0, d, size=(B, N))
    b, n = np.nonzero(big[:, None] & (x[:, :, 0] >= 0))
    x[b, n, coord[b, n]] = vals[b, n]
    return x


def test_reference_without_crossings_is_the_cport_trajectory():
    rng = np.random.default_rng(21)
    for (B, N, d) in ((40, 7, 2), (33, 10, 3), (20, 16, 4)):
        for dtype in (np.int32, np.float32):
            x = start_state(rng, B, N, d, dtype, 9)
            for ops, base in ((JAX_STEP, C.HK_F_ACT_DISCRETE), (FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE)):
                ha, ax = random_actions(rng, 6, B, d, base)
                rec = oracle_record(x, ha, ax, ops, base, 6, agent_obs=True)
                for stop in (False, True):
                    got = oracle_threshold(x, ha, ax, ops, base, 6, math.inf, stop, agent_obs=True)
                    for k in range(8):
                        assert np.array_equal(bits(got[k]), bits(rec[k])), (B, N, d, dtype, stop, k)
                    assert (got[8] == 7).all()


def test_reference_split_at_a_stop_is_one_rollout():
    rng = np.random.default_rng(22)
    B, N, d, T, T1 = 200, 10, 3, 12, 5
    x = start_state(rng, B, N, d, np.int32, 20)
    ops, flags = FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE
    ha, ax = random_actions(rng, T, B, d, flags)
    full = oracle_threshold(x, ha, ax, ops, flags, T, 300, True)
    a = oracle_threshold(x, ha[:T1], ax[:T1], ops, flags, T1, 300, True)
    b = oracle_threshold(a[0], ha[T1:], ax[T1:], ops, flags, T - T1, 300, True)
    assert 0 < (full[8] <= T).sum() < B
    assert np.array_equal(b[0], full[0])
    for k in (4, 5, 6):
        assert np.array_equal(bits(np.concatenate([a[k], b[k]])), bits(full[k])), k
    assert (b[8][a[8] <= T1] == 0).all()
    assert np.array_equal(np.where(a[8] <= T1, a[8], np.where(b[8] <= T - T1, b[8] + T1, T + 1)), full[8])


def test_reference_stays_exact_at_the_int32_bound():
    rng = np.random.default_rng(23)
    for d in (2, 3, 5, 10):
        x = near_bound_state(rng, 64, 8, d)
        flags = TORCH_FLAGS | C.HK_F_ACT_DISCRETE
        ha, ax = random_actions(rng, 6, 64, d, flags)
        r = oracle_threshold(x, ha, ax, FUSED_STEP, flags, 6, bound(d), True)  # the guard asserts inside
        assert (np.where(r[0][:, :, :1] >= 0, r[0], 0) < INT32_BOUND).all()
        assert (r[8] <= 6).any() and (r[8] == 7).any()


# ---------------------------------------------------------------- GPU helpers


def gpu_threshold(L, x, ha, ax, ops, flags, T, thr, stop, pad=-1.0, inplace=False, agent_obs=False, seed=0, step_offset=0,
                  record=False, want_over=True):
    """hk_rollout_threshold through the C-ABI, every output pre-filled with a sentinel (obs / actions only when
    `record`).  Returns (rc, state, obs, masks, axes, done, reward, done_count increments, length, over_step)."""
    import torch
    B, N, d = x.shape
    OW = N * d + (d if agent_obs else 0)
    xin = _dev(x)
    out = xin if inplace else _filled(x.shape, SENTINEL_WORD, xin.dtype)
    obs = _filled((T, B, OW), SENTINEL_WORD, torch.float32) if record else None
    hm = _filled((T, B), SENTINEL_WORD, torch.int32) if record else None
    axp = _filled((T, B), SENTINEL_WORD, torch.int32) if record else None
    done = torch.full((T, B), 0xAB, dtype=torch.uint8, device="cuda")
    reward = _filled((T, B), SENTINEL_REWARD, torch.float32)
    dcount = torch.full((T,), DONE_COUNT_BASE, dtype=torch.int32, device="cuda")
    length = _filled((B,), SENTINEL_WORD, torch.int32)
    over = _filled((B,), SENTINEL_WORD, torch.int32) if want_over else None
    ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    ha_d = None if ha is None else _dev(ha)
    ax_d = None if ax is None else _dev(ax)
    dt = C.HK_DTYPE_I32 if x.dtype == np.int32 else C.HK_DTYPE_F32
    rc = L.hk_rollout_threshold(xin.data_ptr(), out.data_ptr(), ptr(ha_d), ptr(ax_d), ptr(obs), 1 if agent_obs else 0,
                                ptr(hm), ptr(axp), done.data_ptr(), reward.data_ptr(), dcount.data_ptr(), length.data_ptr(),
                                B, N, d, T, dt, ops, flags, float(pad), seed & (2 ** 64 - 1), step_offset, float(thr),
                                1 if stop else 0, ptr(over), _stream())
    if rc != 0:
        return (rc,) + (None,) * 9
    cpu = lambda t: None if t is None else t.cpu().numpy()  # noqa: E731
    return (rc, cpu(out), cpu(obs), cpu(hm), cpu(axp), cpu(done), cpu(reward), cpu(dcount) - DONE_COUNT_BASE, cpu(length),
            cpu(over))


def assert_threshold(got, exp, what):
    assert got[0] == 0, (what, got[0])
    for name, g, e in zip(NAMES, got[1:], exp):
        if g is None:
            continue
        assert g.shape == e.shape, (what, name, g.shape, e.shape)
        if not np.array_equal(bits(g), bits(e)):
            bad = np.argwhere(bits(g) != bits(e))
            raise AssertionError((what, name, "first mismatch at", bad[0].tolist(), g[tuple(bad[0])], e[tuple(bad[0])]))


def check_families(L, x, ha, ax, ops, flags, T, thr, stop, exp, what, k=0, **kw):
    """Both kernel families; the k-th check of a test is run out of place on one family and in place on the other."""
    from hironaka_b200 import ops as hops
    for generic in (False, True):
        hops.force_generic(generic)
        try:
            inplace = (k + generic) % 2 == 1
            assert_threshold(gpu_threshold(L, x, ha, ax, ops, flags, T, thr, stop, inplace=inplace, **kw), exp,
                             (what, "generic" if generic else "auto", "in place" if inplace else "out of place"))
        finally:
            hops.force_generic(False)


MODES = [  # (name, ops, flags)
    ("jax", JAX_STEP, 0),
    ("fused", FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE),
    ("agent", JAX_STEP, C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT),
]


# ---------------------------------------------------------------- shapes x dtypes x stop


@gpu
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
@pytest.mark.parametrize("shape", SWEEP_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_threshold_sweep(lib, shape, dtype):
    """Low thresholds (tens to thousands) so that crossings are common, with and without the stop, in every op mode,
    plain and recorded: over_step, state, done_t, reward_t, length and done_count of both families."""
    B, N, d = shape
    rng = np.random.default_rng(B * 1000 + N * 10 + d + 31)
    k = 0
    for stop in (False, True):
        for name, ops, flags in MODES:
            T = int(rng.integers(5, 11))
            x = start_state(rng, B, N, d, dtype, max_value=int(rng.choice([5, 20, 200])))
            thr = float(rng.choice([10, 40, 300, 2000]))
            ha, ax = random_actions(rng, T, B, d, flags)
            exp = oracle_threshold(x, ha, ax, ops, flags, T, thr, stop)
            check_families(lib, x, ha, ax, ops, flags, T, thr, stop, exp, (name, thr, stop), k=k)
            record = k % 2 == 0
            if record:
                flags_o = flags | C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE
                exp = oracle_threshold(x, ha, ax, ops, flags_o, T, thr, stop, agent_obs=True)
                check_families(lib, x, ha, ax, ops, flags_o, T, thr, stop, exp, (name, thr, stop, "recorded"), k=k + 1,
                               record=True, agent_obs=True)
            k += 1


@gpu
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
@pytest.mark.parametrize("shape", [(65, 10, 3), (33, 20, 3), (40, 7, 4), (20, 64, 5)], ids=lambda s: "x".join(map(str, s)))
def test_long_rollouts(lib, shape, dtype):
    """The torch / FusedGame flavour without reposition over 40 steps (values keep growing: games stop), and the JAX
    flavour with reposition, with and without the stop."""
    B, N, d = shape
    rng = np.random.default_rng(N * 7 + d)
    T = 40
    crossings = 0
    for k, (ops, flags, thr, stop) in enumerate(((FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE, 20.0, True),
                                                  (FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE, 60.0, True),
                                                  (JAX_STEP, C.HK_F_ACT_DISCRETE, 15.0, True),
                                                  (JAX_STEP, C.HK_F_ACT_DISCRETE, 15.0, False))):
        x = start_state(rng, B, N, d, dtype, 12)
        ha, ax = random_actions(rng, T, B, d, flags)
        exp = oracle_threshold(x, ha, ax, ops, flags, T, thr, stop)
        crossings += int(((exp[8] > 0) & (exp[8] <= T)).sum())
        check_families(lib, x, ha, ax, ops, flags, T, thr, stop, exp, (ops, thr, stop), k=k)
    assert crossings > 0


@gpu
@pytest.mark.parametrize("d", [2, 3, 5, 10])
def test_int32_bound(lib, d):
    """value_threshold = floor(2^30 / d), starts just below it, with the stop: every written state equals the int64-guarded
    reference and stays below 2^30; a threshold one above the bound and NaN are refused."""
    rng = np.random.default_rng(d + 40)
    for k, (B, N) in enumerate(((97, 8), (33, 20))):
        x = near_bound_state(rng, B, N, d)
        flags = TORCH_FLAGS | C.HK_F_ACT_DISCRETE
        T = 8
        ha, ax = random_actions(rng, T, B, d, flags)
        for ops in (FUSED_STEP, JAX_STEP):
            exp = oracle_threshold(x, ha, ax, ops, flags, T, bound(d), True)
            check_families(lib, x, ha, ax, ops, flags, T, bound(d), True, exp, (d, N, ops), k=k)
            assert (np.where(exp[0][:, :, :1] >= 0, exp[0], 0) < INT32_BOUND).all()
    ha, ax = random_actions(rng, 2, 8, d, 0)
    x = start_state(rng, 8, 6, d, np.int32, 5)
    assert gpu_threshold(lib, x, ha, ax, JAX_STEP, 0, 2, above_bound(d), True)[0] == C.HK_ERR_BAD_ARG
    assert gpu_threshold(lib, x, ha, ax, JAX_STEP, 0, 2, math.nan, False)[0] == C.HK_ERR_BAD_ARG
    assert gpu_threshold(lib, x.astype(np.float32), ha, ax, JAX_STEP, 0, 2, math.nan, True)[0] == C.HK_ERR_BAD_ARG
    # a float32 state has no such bound
    assert gpu_threshold(lib, x.astype(np.float32), ha, ax, JAX_STEP, 0, 2, 1e12, True)[0] == 0


@gpu
@pytest.mark.parametrize("shape", [(129, 20, 3), (65, 10, 3), (40, 16, 4)], ids=lambda s: "x".join(map(str, s)))
def test_float32_thresholds_above_2_24(lib, shape):
    """float32 states with values around 2^24 .. 2^26 and thresholds above 2^24: the comparison is float32's."""
    B, N, d = shape
    rng = np.random.default_rng(N + d + 50)
    T = 8
    for k, stop in enumerate((True, False)):
        x = start_state(rng, B, N, d, np.float32, 10)
        live = x[:, :, :1] >= 0
        x = np.where(live & (rng.random((B, N, d)) < 0.3), rng.integers(1 << 23, 1 << 25, (B, N, d)), x).astype(np.float32)
        flags = TORCH_FLAGS | C.HK_F_ACT_DISCRETE
        ha, ax = random_actions(rng, T, B, d, flags)
        for j, thr in enumerate((float((1 << 24) + 2), float(1 << 25) + 4.0, 3.0e7)):
            exp = oracle_threshold(x, ha, ax, FUSED_STEP, flags, T, thr, stop)
            check_families(lib, x, ha, ax, FUSED_STEP, flags, T, thr, stop, exp, (thr, stop), k=k + j)


@gpu
@pytest.mark.parametrize("shape", [(97, 20, 3), (33, 10, 3), (50, 7, 2), (20, 64, 5)], ids=lambda s: "x".join(map(str, s)))
def test_crossing_at_entry(lib, shape):
    """Games over the threshold on entry: over_step 0, never stepped (state as read, dead rows padded), done repeated,
    no reward, length untouched; the others play on."""
    B, N, d = shape
    rng = np.random.default_rng(B + N + 60)
    T = 6
    for k, dtype in enumerate((np.int32, np.float32)):
        x = start_state(rng, B, N, d, dtype, 20)
        x[::3, 0] = 500  # row 0 live and over the threshold
        flags = C.HK_F_ACT_DISCRETE
        ha, ax = random_actions(rng, T, B, d, flags)
        exp = oracle_threshold(x, ha, ax, JAX_STEP, flags, T, 400.0, True)
        assert (exp[8][::3] == 0).all()
        assert np.array_equal(bits(exp[0][::3]), bits(padded(x, -1.0)[::3]))
        check_families(lib, x, ha, ax, JAX_STEP, flags, T, 400.0, True, exp, dtype.__name__, k=k)


@gpu
@pytest.mark.parametrize("shape", [(257, 20, 3), (33, 10, 3), (97, 5, 3), (50, 7, 2), (16, 64, 5)],
                         ids=lambda s: "x".join(map(str, s)))
def test_split_rollouts_and_random_players(lib, shape):
    """In-kernel random players across stops: one call of T equals T1 + (T - T1) with the step counter advanced; the
    second call reports 0 for the games stopped in the first, and every other game plays the draws it plays without
    the stop."""
    from hironaka_b200 import ops as hops
    B, N, d = shape
    rng = np.random.default_rng(B * 3 + N + 70)
    T, T1 = 12, 5
    for k, dtype in enumerate((np.int32, np.float32)):
        x = start_state(rng, B, N, d, dtype, 15)
        flags = RANDOM | TORCH_FLAGS | C.HK_F_ACT_DISCRETE
        thr = 20.0
        exp = oracle_threshold(x, None, None, FUSED_STEP, flags, T, thr, True, seed=SEED, step_offset=STEP_OFFSET)
        assert 0 < (exp[8] <= T).sum()
        check_families(lib, x, None, None, FUSED_STEP, flags, T, thr, True, exp, dtype.__name__, k=k, seed=SEED,
                       step_offset=STEP_OFFSET)
        for generic in (False, True):
            hops.force_generic(generic)
            try:
                a = gpu_threshold(lib, x, None, None, FUSED_STEP, flags, T1, thr, True, seed=SEED, step_offset=STEP_OFFSET)
                b = gpu_threshold(lib, a[1], None, None, FUSED_STEP, flags, T - T1, thr, True, seed=SEED,
                                  step_offset=STEP_OFFSET + T1, inplace=True)
                assert np.array_equal(bits(b[1]), bits(exp[0])), generic
                for i in (5, 6, 7):
                    assert np.array_equal(bits(np.concatenate([a[i], b[i]])), bits(exp[i - 1])), (generic, NAMES[i - 1])
                assert (b[9][a[9] <= T1] == 0).all()
                over = np.where(a[9] <= T1, a[9], np.where(b[9] <= T - T1, b[9] + T1, T + 1))
                assert np.array_equal(over, exp[8]), generic
            finally:
                hops.force_generic(False)


@gpu
@pytest.mark.parametrize("shape", [(40, 100, 3), (64, 7, 2), (96, 20, 3), (70, 10, 3)], ids=lambda s: "x".join(map(str, s)))
def test_fixed_players_and_replay(lib, shape):
    """The fixed players across stops, recorded: a stopped game's obs rows are the features of its frozen state, its
    host masks 0 and axes -1; the recorded actions replayed as streams with the same threshold and stop give the
    rollout back bit for bit."""
    B, N, d = shape
    rng = np.random.default_rng(N + d + 80)
    T = 8
    thr = 14.0
    stops = 0
    for dtype in (np.int32, np.float32):
        x = start_state(rng, B, N, d, dtype, 12)
        for k, pol in enumerate((F_ALL | F_FIRST, F_ZEIL | F_LAST, F_ZEIL, F_LAST, RANDOM)):
            ncls = 2 ** d - d - 1
            ha = None if pol & (HOST_FIXED | C.HK_F_HOST_RANDOM) else rng.integers(0, ncls, (T, B)).astype(np.int32)
            ax = None if pol & (AGENT_FIXED | C.HK_F_AGENT_RANDOM) else rng.integers(0, d, (T, B)).astype(np.int32)
            flags = pol | TORCH_FLAGS | C.HK_F_ACT_DISCRETE | C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE
            exp = oracle_threshold(x, ha, ax, FUSED_STEP, flags, T, thr, True, agent_obs=True, seed=SEED)
            stopped = exp[8] < T
            stops += int(stopped.sum())
            t_after = exp[8][stopped]
            assert (exp[3][t_after, np.nonzero(stopped)[0]] == -1).all()
            check_families(lib, x, ha, ax, FUSED_STEP, flags, T, thr, True, exp, (hex(pol), dtype.__name__), k=k,
                           record=True, agent_obs=True, seed=SEED)
            rep = gpu_threshold(lib, x, exp[2], exp[3], FUSED_STEP, replay_flags(flags), T, thr, True, record=True,
                                agent_obs=True)
            assert_threshold(rep, exp, ("replay", hex(pol), dtype.__name__))
    assert stops > 0


@gpu
@pytest.mark.parametrize("shape", [(101, 20, 3), (33, 10, 3), (50, 7, 2), (17, 64, 5)], ids=lambda s: "x".join(map(str, s)))
def test_infinite_threshold_is_the_recorded_rollout(lib, shape):
    """value_threshold = +inf: every output equals hk_rollout_record's and over_step is T + 1 everywhere, with and
    without the stop; without over_step the call is hk_rollout_record itself."""
    from tests.test_gpu_record import gpu_record
    B, N, d = shape
    rng = np.random.default_rng(B + N + 90)
    T = 7
    for k, dtype in enumerate((np.int32, np.float32)):
        x = start_state(rng, B, N, d, dtype, 1000)
        flags = C.HK_F_ACT_DISCRETE | C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE
        ha, ax = random_actions(rng, T, B, d, flags)
        ref = gpu_record(lib, x, ha, ax, JAX_STEP, flags, T, agent_obs=True)
        assert ref[0] == 0
        for stop in (False, True):
            for want_over in (True, False):
                got = gpu_threshold(lib, x, ha, ax, JAX_STEP, flags, T, math.inf, stop, record=True, agent_obs=True,
                                    want_over=want_over)
                assert got[0] == 0
                for i in range(1, 9):
                    assert np.array_equal(bits(got[i]), bits(ref[i])), (stop, want_over, NAMES[i - 1])
                if want_over:
                    assert (got[9] == T + 1).all()


@gpu
def test_game_batch_threshold(lib):
    """GameBatch(value_threshold=..., stop_at_threshold=True) with the random players, the torch flavour without
    reposition: rollout, record and step go through hk_rollout_threshold; `crossed` follows the games across calls and
    a stopped game stays stopped."""
    import torch
    from hironaka_b200.engine import GameBatch
    rng = np.random.default_rng(95)
    B, N, d = 300, 10, 3
    x = start_state(rng, B, N, d, np.int32, 20)
    thr = 150.0
    seed = 77
    gb = GameBatch(torch.from_numpy(x).cuda(), semantics="torch", reposition=False, host_policy="random",
                   agent_policy="random", seed=seed, value_threshold=thr, stop_at_threshold=True)
    flags = gb.flags
    ops = gb.ops
    exp = oracle_threshold(x, None, None, ops, flags, 12, thr, True, seed=seed)
    gb.rollout(steps=4)
    assert np.array_equal(gb.crossed.cpu().numpy(), exp[8] <= 4)
    traj = gb.record(steps=6, agent_obs=True)
    assert np.array_equal(gb.crossed.cpu().numpy(), exp[8] <= 10)
    mid = oracle_threshold(x, None, None, ops, flags, 4, thr, True, seed=seed)
    rec = oracle_threshold(mid[0], None, None, ops, flags | C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE, 6, thr, True,
                           agent_obs=True, seed=seed, step_offset=4)
    assert np.array_equal(traj.obs.cpu().numpy().view(np.int32), rec[1].view(np.int32))
    assert np.array_equal(traj.axis.cpu().numpy(), rec[3])
    for _ in range(2):
        done, reward = gb.step()
    assert np.array_equal(gb.points.cpu().numpy(), exp[0])
    assert np.array_equal(done.cpu().numpy(), exp[4][11] != 0)
    assert np.array_equal(reward.cpu().numpy().view(np.int32), exp[5][11].view(np.int32))
    assert np.array_equal(gb.crossed.cpu().numpy(), exp[8] <= 12)
    assert gb.crossed.any() and not gb.crossed.all()
