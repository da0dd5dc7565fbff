"""Recorded rollouts (hk_rollout_record) against the oracle's C port stepped once per step.

A recorded rollout is hk_rollout / hk_rollout_seeded that also writes what the players saw before every step (the
features of the state, hk_features' flags) and what they played (the coordinate bitmask and the axis of the shift).
The expected trajectory is the C port stepped once per step: cport.features of each state before its step, the played
actions from the streams (decoded), from oracle.random_player_actions, or from the fixed players (Zeillinger's host as
zeillinger_fn picks it, all coordinates, first / last agent).  Every output is pre-filled with a sentinel and compared
bit for bit; done_count is incremented from a nonzero start.

The tests without the gpu mark check the reference side: the played actions, replayed as bitmask streams without the
player flags, give the same C-port rollout.
"""
import numpy as np
import pytest

from hironaka_b200 import constants as C
from oracle import cport
from oracle import hk_oracle as O
from tests.test_gpu_rollout import (DONE_COUNT_BASE, F_ALL, F_FIRST, F_LAST, F_ZEIL, FUSED_STEP, JAX_STEP, SEED,
                                    SENTINEL_REWARD, SENTINEL_WORD, STEP_OFFSET, SWEEP_SHAPES, TORCH_FLAGS, _dev, _filled,
                                    _stream, bits, decode_ids, gpu_rollout, lib, oracle_rollout, pack_bytes, pack_nibbles,
                                    random_actions, start_state)

gpu = pytest.mark.gpu
_ = lib  # the module's library fixture

HOST_FIXED = F_ALL | F_ZEIL
AGENT_FIXED = F_FIRST | F_LAST
RANDOM = C.HK_F_HOST_RANDOM | C.HK_F_AGENT_RANDOM
PLAYERS = HOST_FIXED | AGENT_FIXED | RANDOM
FORMATS = C.HK_F_ACT_U8 | C.HK_F_ACT_PACKED | C.HK_F_ACT_NIBBLE


# ---------------------------------------------------------------- reference side (no GPU)


def zeillinger_masks(x):
    """zeillinger_fn (oracle) on every game at once, as coordinate bitmasks: among ordered pairs of rows without a
    negative entry whose difference is not constant, the smallest (max - min, #max + #min) in flat (i, j) order; its
    {argmin, argmax}, or decoded action 0 when there is no such pair or argmin == argmax."""
    B, N, d = x.shape
    p = x.astype(np.float32)
    ok_row = (p >= 0).all(2)
    diff = p[:, :, None, :] - p[:, None, :, :]
    mx, mn = diff.max(3), diff.min(3)
    ok = ok_row[:, :, None] & ok_row[:, None, :] & ~np.isclose(mx, mn)
    cmax, cmin = (diff == mx[..., None]).sum(3), (diff == mn[..., None]).sum(3)
    L = np.where(ok, mx - mn, np.inf).reshape(B, -1)
    S = np.where(ok, np.where(mx == mn, cmax, cmax + cmin), np.inf).reshape(B, -1)
    idx = np.lexsort((S, L), axis=-1)[:, 0]
    v = diff.reshape(B, N * N, d)[np.arange(B), idx]
    amin, amax = v.argmin(1), v.argmax(1)
    return np.where(amin == amax, 3, (1 << amin) | (1 << amax)).astype(np.int32)


def agent_axes(masks, d, flags):
    """choose_first_agent_fn / choose_last_agent_fn on coordinate bitmasks (an empty set: 0 / d - 1)."""
    m = np.asarray(masks, np.int64)
    sel = (m[:, None] >> np.arange(d)) & 1
    if flags & F_FIRST:
        return np.where(m == 0, 0, sel.argmax(1)).astype(np.int32)
    return np.where(m == 0, d - 1, d - 1 - sel[:, ::-1].argmax(1)).astype(np.int32)


def mask_bits(m, d):
    return ((np.asarray(m, np.int64)[:, None] >> np.arange(d)) & 1).astype(np.float32)


def oracle_record(x, ha, ax, ops, flags, T, pad=-1.0, agent_obs=False, seed=0, step_offset=0):
    """T steps of the C port with what each step saw and played: (state, obs [T, B, OW], host masks [T, B], axes [T, B],
    done [T, B], reward [T, B], finished games per step [T], length [B]).  ha / ax: int32 [T, B] streams (discrete ids
    with HK_F_ACT_DISCRETE), None for a fixed or random player.  `flags` carries the observation flags too."""
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
    obs, masks, axes = [], [], []
    done = np.empty((T, B), np.uint8)
    reward = np.empty((T, B), np.float32)
    for t in range(T):
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
        # the features read live rows only (a dead row is one with a negative coordinate 0); the C port's rescale would
        # also see what else a dead row of the start state holds, so it gets the state with dead rows padded
        f = cport.features(np.where((o[:, :, :1] >= 0), o, o.dtype.type(pad)), flags, padding_value=pad)
        obs.append(np.concatenate([f, mask_bits(played, d)], 1) if agent_obs else f)
        masks.append(played)
        axes.append(a)
        o, done[t], reward[t], _ = cport.step(o, None if ha is None else ha[t], None if ax is None else ax[t], ops,
                                              step_flags, padding_value=pad)
        length[(length == T + 1) & (done[t] != 0)] = t + 1
    return (o, np.stack(obs), np.stack(masks), np.stack(axes), done, reward, done.sum(1).astype(np.int32), length)


def replay_flags(flags):
    """The flags of a replay of recorded actions: bitmask and int32 axis streams, no players."""
    return flags & ~(PLAYERS | C.HK_F_ACT_DISCRETE | FORMATS)


def test_zeillinger_masks_match_zeillinger_fn():
    rng = np.random.default_rng(11)
    for (B, N, d) in ((40, 7, 2), (30, 10, 3), (20, 6, 4)):
        x = start_state(rng, B, N, d, np.int32, 5)
        exp = decode_ids(O.zeillinger_fn(x).argmax(1), d)
        assert np.array_equal(zeillinger_masks(x), exp), (B, N, d)


@pytest.mark.parametrize("shape", [(50, 7, 2), (33, 10, 3), (20, 16, 4)], ids=lambda s: "x".join(map(str, s)))
def test_replayed_actions_reproduce_oracle_rollout(shape):
    B, N, d = shape
    rng = np.random.default_rng(B + N + d)
    T = 8
    ncls = 2 ** d - d - 1
    for dtype in (np.int32, np.float32):
        x = start_state(rng, B, N, d, dtype, 9)
        for pol in (F_ALL | F_FIRST, F_ALL | F_LAST, F_ZEIL | F_FIRST, F_ZEIL | F_LAST, F_ZEIL, F_FIRST, F_LAST, RANDOM,
                    C.HK_F_HOST_RANDOM, C.HK_F_AGENT_RANDOM):
            for ops, base in ((JAX_STEP, C.HK_F_ACT_DISCRETE), (FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE)):
                flags = pol | base
                ha = None if pol & (HOST_FIXED | C.HK_F_HOST_RANDOM) else rng.integers(0, ncls, (T, B)).astype(np.int32)
                ax = None if pol & (AGENT_FIXED | C.HK_F_AGENT_RANDOM) else rng.integers(0, d, (T, B)).astype(np.int32)
                rec = oracle_record(x, ha, ax, ops, flags, T, seed=SEED, step_offset=STEP_OFFSET)
                replay = oracle_rollout(x, rec[2], rec[3], ops, replay_flags(flags))
                assert np.array_equal(bits(replay[0]), bits(rec[0])), (pol, ops)
                for k in range(1, 5):
                    assert np.array_equal(bits(replay[k]), bits(rec[k + 3])), (pol, ops, k)
                if pol & HOST_FIXED and not pol & AGENT_FIXED:  # the stream agent's axes are recorded as given
                    assert np.array_equal(rec[3], ax)


# ---------------------------------------------------------------- GPU helpers


def gpu_record(L, x, ha, ax, ops, flags, T, pad=-1.0, inplace=False, agent_obs=False, seed=0, step_offset=0,
               want_obs=True, want_actions=True):
    """hk_rollout_record through the C-ABI, every output pre-filled with a sentinel.  Returns (rc, state, obs, masks,
    axes, done, reward, done_count increments, length)."""
    import torch
    B, N, d = x.shape
    OW = N * d + (d if agent_obs else 0)
    xin = _dev(x)
    out = xin if inplace else _filled(x.shape, SENTINEL_WORD, xin.dtype)
    obs = _filled((T, B, OW), SENTINEL_WORD, torch.float32) if want_obs else None
    hm = _filled((T, B), SENTINEL_WORD, torch.int32) if want_actions else None
    axp = _filled((T, B), SENTINEL_WORD, torch.int32) if want_actions else None
    done = torch.full((T, B), 0xAB, dtype=torch.uint8, device="cuda")
    reward = _filled((T, B), SENTINEL_REWARD, torch.float32)
    dcount = torch.full((T,), DONE_COUNT_BASE, dtype=torch.int32, device="cuda")
    length = _filled((B,), SENTINEL_WORD, torch.int32)
    ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    ha_d = None if ha is None else _dev(ha)
    ax_d = None if ax is None else _dev(ax)
    dt = C.HK_DTYPE_I32 if x.dtype == np.int32 else C.HK_DTYPE_F32
    rc = L.hk_rollout_record(xin.data_ptr(), out.data_ptr(), ptr(ha_d), ptr(ax_d), ptr(obs), 1 if agent_obs else 0, ptr(hm),
                             ptr(axp), done.data_ptr(), reward.data_ptr(), dcount.data_ptr(), length.data_ptr(), B, N, d, T,
                             dt, ops, flags, float(pad), seed & (2 ** 64 - 1), step_offset, _stream())
    if rc != 0:
        return (rc,) + (None,) * 8
    cpu = lambda t: None if t is None else t.cpu().numpy()  # noqa: E731
    return (rc, cpu(out), cpu(obs), cpu(hm), cpu(axp), cpu(done), cpu(reward), cpu(dcount) - DONE_COUNT_BASE, cpu(length))


NAMES = ("state", "obs", "host_mask", "axis", "done", "reward", "done_count", "length")


def assert_record(got, exp, what):
    assert got[0] == 0, (what, got[0])
    for name, g, e in zip(NAMES, got[1:], exp):
        if g is None:
            continue
        assert g.shape == e.shape, (what, name, g.shape, e.shape)
        if not np.array_equal(bits(g), bits(e)):
            bad = np.argwhere(bits(g) != bits(e))
            raise AssertionError((what, name, "first mismatch at", bad[0].tolist(), g[tuple(bad[0])], e[tuple(bad[0])]))


def check_families(L, x, ha, ax, ops, flags, T, exp, what, k=0, **kw):
    """Both kernel families; the k-th check of a test is run out of place on one family and in place on the other."""
    from hironaka_b200 import ops as hops
    for generic in (False, True):
        hops.force_generic(generic)
        try:
            inplace = (k + generic) % 2 == 1
            assert_record(gpu_record(L, x, ha, ax, ops, flags, T, inplace=inplace, **kw), exp,
                          (what, "generic" if generic else "auto", "in place" if inplace else "out of place"))
        finally:
            hops.force_generic(False)


# ---------------------------------------------------------------- shapes x op modes x observation modes


OP_MODES = [  # (name, ops, flags, float32 only)
    ("jax", JAX_STEP, 0, False),
    ("fused", FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE, False),
    ("rescale", JAX_STEP | C.HK_OP_RESCALE, 0, True),
    ("rescale_eps", JAX_STEP | C.HK_OP_RESCALE, C.HK_F_RESCALE_EPS, True),
    ("dedupe", C.HK_OP_SHIFT | C.HK_OP_DEDUPE, C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT, False),
]
SORTS = [0, C.HK_F_OBS_SORT_COORD0, C.HK_F_OBS_SORT_LEX, C.HK_F_OBS_SORT_LEX_FIRST]
OBS_MODES = [(s | r, False) for s in SORTS for r in (0, C.HK_F_OBS_RESCALE)] + [(C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE, True)]


@gpu
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
@pytest.mark.parametrize("shape", SWEEP_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_record_modes(lib, shape, dtype):
    """Every observation mode (unsorted, coord0, lex, lex-first, each with and without HK_F_OBS_RESCALE, and the agent's
    view) under the op modes in turn; rescale on an int32 state is refused as hk_rollout refuses it."""
    B, N, d = shape
    rng = np.random.default_rng(B * 1000 + N * 10 + d + 7)
    modes = [m for m in OP_MODES if not m[3] or dtype == np.float32]
    for k, (obs_flags, agent_obs) in enumerate(OBS_MODES):
        name, ops, base, _ = modes[k % len(modes)]
        flags = base | obs_flags
        T = int(rng.integers(4, 9))
        x = start_state(rng, B, N, d, dtype, max_value=int(rng.choice([1, 3, 20, 1000])))
        ha, ax = random_actions(rng, T, B, d, flags)
        exp = oracle_record(x, ha, ax, ops, flags, T, agent_obs=agent_obs)
        check_families(lib, x, ha, ax, ops, flags, T, exp, (name, hex(obs_flags), agent_obs), k=k, agent_obs=agent_obs)
    if dtype == np.int32:
        ha, ax = random_actions(rng, 3, B, d, 0)
        x = start_state(rng, B, N, d, dtype, 5)
        assert gpu_record(lib, x, ha, ax, JAX_STEP | C.HK_OP_RESCALE, 0, 3)[0] == C.HK_ERR_UNSUPPORTED


@gpu
@pytest.mark.parametrize("shape", [(101, 20, 3), (33, 10, 3), (65, 5, 3), (31, 7, 2), (17, 64, 5)],
                         ids=lambda s: "x".join(map(str, s)))
def test_record_action_formats(lib, shape):
    """int32, uint8, packed and nibble streams (odd batch sizes): the recorded masks and axes are the unpacked, decoded
    actions, and the trajectory is the int32 stream's."""
    B, N, d = shape
    rng = np.random.default_rng(B + 5 * N + d)
    T = 6
    ncls = 2 ** d - d - 1
    for k, dtype in enumerate((np.int32, np.float32)):
        x = start_state(rng, B, N, d, dtype, 10)
        base = C.HK_F_ACT_DISCRETE | C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE
        hi = min(ncls, 4) if d <= 3 else ncls
        ha = rng.integers(0, hi, (T, B)).astype(np.int32)
        ax = rng.integers(0, d, (T, B)).astype(np.int32)
        ax[rng.random((T, B)) < 0.15] = 3 if d <= 3 else 7
        exp = oracle_record(x, ha, ax, JAX_STEP, base, T, agent_obs=True)
        streams = [("u8", ha.astype(np.uint8), ax.astype(np.uint8), base | C.HK_F_ACT_U8)]
        if d <= 5:
            streams.append(("packed", pack_bytes(ha, ax), None, base | C.HK_F_ACT_PACKED))
        if d <= 3:
            streams.append(("nibble", pack_nibbles(ha, ax), None, base | C.HK_F_ACT_NIBBLE))
        for j, (fmt, h, a, flags) in enumerate(streams):
            check_families(lib, x, h, a, JAX_STEP, flags, T, exp, (fmt, dtype.__name__), k=k + j, agent_obs=True)


@gpu
@pytest.mark.parametrize("shape", [(257, 20, 3), (33, 10, 3), (97, 5, 3), (50, 7, 2), (16, 64, 5)],
                         ids=lambda s: "x".join(map(str, s)))
def test_record_random_players(lib, shape):
    """In-kernel random players with a high seed and a step counter crossing 2^30: the recorded actions are
    oracle.random_player_actions decoded, in one call and in two calls split at T1 (step_offset advanced)."""
    import torch
    from hironaka_b200 import ops as hops
    B, N, d = shape
    rng = np.random.default_rng(B * 3 + N)
    T, T1 = 10, 4
    for k, dtype in enumerate((np.int32, np.float32)):
        x = start_state(rng, B, N, d, dtype, 15)
        flags = RANDOM | C.HK_F_ACT_DISCRETE | C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE
        exp = oracle_record(x, None, None, JAX_STEP, flags, T, agent_obs=True, seed=SEED, step_offset=STEP_OFFSET)
        check_families(lib, x, None, None, JAX_STEP, flags, T, exp, ("both random", dtype.__name__), k=k, agent_obs=True,
                       seed=SEED, step_offset=STEP_OFFSET)
        for generic in (False, True):
            hops.force_generic(generic)
            try:
                a = gpu_record(lib, x, None, None, JAX_STEP, flags, T1, agent_obs=True, seed=SEED, step_offset=STEP_OFFSET)
                b = gpu_record(lib, a[1], None, None, JAX_STEP, flags, T - T1, agent_obs=True, seed=SEED,
                               step_offset=STEP_OFFSET + T1, inplace=True)
                for i in range(1, 8):
                    got = b[i] if i == 1 else np.concatenate([a[i], b[i]])
                    assert np.array_equal(bits(got), bits(exp[i - 1])), (generic, NAMES[i - 1])
            finally:
                hops.force_generic(False)
        ax_s = rng.integers(0, d, (T, B)).astype(np.int32)
        flags = C.HK_F_HOST_RANDOM | TORCH_FLAGS | C.HK_F_OBS_SORT_COORD0
        exp = oracle_record(x, None, ax_s, FUSED_STEP, flags, T, seed=SEED, step_offset=STEP_OFFSET)
        check_families(lib, x, None, ax_s, FUSED_STEP, flags, T, exp, ("host random", dtype.__name__), k=k + 1,
                       seed=SEED, step_offset=STEP_OFFSET)
    torch.cuda.synchronize()


@gpu
@pytest.mark.parametrize("shape", [(40, 100, 3), (64, 7, 2), (96, 20, 3), (70, 10, 3)], ids=lambda s: "x".join(map(str, s)))
def test_record_fixed_players(lib, shape):
    """The seven fixed-player combinations: Zeillinger's choice and the agents' axes as the players pick them, 0 for
    a fixed host on a game without live rows."""
    B, N, d = shape
    rng = np.random.default_rng(N + d + 2)
    T = 6
    ncls = 2 ** d - d - 1
    for dtype in (np.int32, np.float32):
        x = start_state(rng, B, N, d, dtype, 12)
        for k, pol in enumerate((F_ALL | F_FIRST, F_ALL | F_LAST, F_ZEIL | F_FIRST, F_ZEIL | F_LAST, F_ZEIL, F_FIRST, F_LAST)):
            ha = None if pol & HOST_FIXED else rng.integers(0, ncls, (T, B)).astype(np.int32)
            ax = None if pol & AGENT_FIXED else rng.integers(0, d, (T, B)).astype(np.int32)
            flags = pol | C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT | (TORCH_FLAGS if k % 2 else 0) | C.HK_F_OBS_SORT_LEX
            exp = oracle_record(x, ha, ax, JAX_STEP, flags, T, agent_obs=True)
            check_families(lib, x, ha, ax, JAX_STEP, flags, T, exp, (pol, dtype.__name__), k=k, agent_obs=True)


# ---------------------------------------------------------------- self-consistency


@gpu
@pytest.mark.parametrize("shape", [(257, 20, 3), (33, 10, 3), (31, 5, 3), (40, 16, 4), (9, 4, 10)],
                         ids=lambda s: "x".join(map(str, s)))
def test_record_is_the_rollout(lib, shape):
    """With the recording outputs null and with them set, state / done / reward / done_count / length are those of
    hk_rollout (hk_rollout_seeded with random players); the recorded actions replayed as streams give the rollout
    again; T = 1 records hk_features of the start state."""
    import torch
    from hironaka_b200 import ops as hops
    B, N, d = shape
    rng = np.random.default_rng(B + N * d + 1)
    T = 9
    for dtype in (np.int32, np.float32):
        x = start_state(rng, B, N, d, dtype, 8)
        for generic in (False, True):
            hops.force_generic(generic)
            try:
                for ops, flags, seed in ((JAX_STEP, RANDOM | C.HK_F_ACT_DISCRETE, SEED),
                                         (FUSED_STEP, F_ZEIL | F_LAST | C.HK_F_ACT_DISCRETE | TORCH_FLAGS, None),
                                         (JAX_STEP, C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT, None)):
                    ha = None if flags & (HOST_FIXED | RANDOM) else random_actions(rng, T, B, d, flags)[0]
                    ax = None if flags & (AGENT_FIXED | RANDOM) else random_actions(rng, T, B, d, flags)[1]
                    kw = dict(seed=SEED, step_offset=STEP_OFFSET) if seed is not None else {}
                    ref = gpu_rollout(lib, x, ha, ax, ops, flags, T=T, **kw)
                    what = (dtype.__name__, generic, hex(flags))
                    for want in (False, True):
                        rec = gpu_record(lib, x, ha, ax, ops, flags | C.HK_F_OBS_SORT_LEX, T, want_obs=want,
                                         want_actions=want, **kw)
                        assert rec[0] == 0, what
                        for i, j in ((1, 1), (5, 2), (6, 3), (7, 4), (8, 5)):
                            assert np.array_equal(bits(rec[i]), bits(ref[j])), (what, want, NAMES[i - 1])
                    replay = gpu_rollout(lib, x, rec[3], rec[4], ops, replay_flags(flags), T=T)
                    for j in range(1, 6):
                        assert np.array_equal(bits(replay[j]), bits(ref[j])), (what, "replay", j)
                    # T = 1: the one recorded observation is hk_features of the start state
                    one = gpu_record(lib, x, ha if ha is None else ha[:1], ax if ax is None else ax[:1], ops,
                                     flags | C.HK_F_OBS_SORT_LEX_FIRST | C.HK_F_OBS_RESCALE, 1, **kw)
                    feats = hops.features(_dev(x), flags=C.HK_F_OBS_SORT_LEX_FIRST | C.HK_F_OBS_RESCALE).cpu().numpy()
                    assert np.array_equal(bits(one[2][0]), bits(feats)), what
                    assert np.array_equal(bits(one[1]), bits(gpu_rollout(lib, x, None if ha is None else ha[:1],
                                                                          None if ax is None else ax[:1], ops, flags, T=1,
                                                                          **kw)[1])), what
            finally:
                hops.force_generic(False)
    torch.cuda.synchronize()


@gpu
def test_record_refuses_what_rollout_refuses(lib):
    B, N, d, T = 33, 10, 3, 3
    rng = np.random.default_rng(5)
    x = start_state(rng, B, N, d, np.int32, 5)
    ha, ax = random_actions(rng, T, B, d, C.HK_F_ACT_DISCRETE)
    ax = np.clip(ax, 0, d - 1)
    cases = [  # (ops, flags, host actions, axes)
        (JAX_STEP | C.HK_OP_RESCALE, 0, ha, ax),                                  # rescale on int32
        (JAX_STEP, C.HK_F_ACT_PACKED | F_ZEIL, pack_bytes(ha % 4, ax), None),      # packed with a fixed player
        (JAX_STEP, C.HK_F_ACT_NIBBLE, pack_nibbles(ha % 4, ax), None),             # nibble without discrete ids
        (JAX_STEP, C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_SORT_COORD0, ha, ax),          # two sort modes
        (JAX_STEP, F_ZEIL | F_ALL, None, ax),                                      # two hosts
        (JAX_STEP, 0, None, ax),                                                   # a shift without host actions
    ]
    for ops, flags, h, a in cases:
        rc = gpu_record(lib, x, h, a, ops, flags, T)[0]
        ref = gpu_rollout(lib, x, h, a, ops, flags, T=T)[0]
        assert rc == ref and rc < 0, (ops, hex(flags), rc, ref)
    import torch
    obs = torch.empty((1, B, N * d), dtype=torch.float32, device="cuda")
    xin = _dev(x)
    assert lib.hk_rollout_record(xin.data_ptr(), xin.data_ptr(), _dev(ha).data_ptr(), _dev(ax).data_ptr(), obs.data_ptr(), 0,
                                 None, None, None, None, None, None, B, N, d, 0, C.HK_DTYPE_I32, JAX_STEP, 0, -1.0, 0, 0,
                                 _stream()) == C.HK_ERR_BAD_ARG
    assert lib.hk_rollout_record(xin.data_ptr(), xin.data_ptr(), _dev(ha).data_ptr(), _dev(ax).data_ptr(), None, 1, None, None,
                                 None, None, None, None, B, N, d, T, C.HK_DTYPE_I32, JAX_STEP, 0, -1.0, 0, 0,
                                 _stream()) == C.HK_ERR_BAD_ARG  # agent_obs without obs_t


# ---------------------------------------------------------------- a trajectory above 2^31 words


@gpu
def test_record_obs_beyond_2_31_words(lib):
    """C2 (1 Mi games of (20, 3)), 36 random-play steps: the obs buffer holds 36 * 2^20 * 60 > 2^31 words.  Steps 33, 34
    and 35 (row 34 starts below 2^31 words and ends above it) and a sample of the rest are compared on the device with
    hk_features of the states of single-step hk_rollout_seeded calls."""
    import torch
    from hironaka_b200 import ops as hops
    B, N, d, T = 1 << 20, 20, 3, 36
    OW = N * d
    assert T * B * OW > 2 ** 31 and 34 * B * OW < 2 ** 31 < 35 * B * OW
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randint(0, 12, (B, N, d), dtype=torch.int32, device="cuda", generator=g)
    x[torch.rand((B, N), device="cuda", generator=g) < 0.4] = -1
    flags = RANDOM | C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE
    traj = hops.rollout_record(x.clone(), T, ops=JAX_STEP, flags=flags, seed=SEED, step_offset=5, inplace=False,
                               want_actions=False, want_done=False, want_reward=False, want_length=False)
    s = x.clone()
    sample = torch.arange(0, B, 4099, device="cuda")
    for t in range(T):
        f = hops.features(s, flags=C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE)
        if t >= 33:
            assert torch.equal(traj.obs[t].view(torch.int32), f.view(torch.int32)), t
        else:
            assert torch.equal(traj.obs[t][sample].view(torch.int32), f[sample].view(torch.int32)), t
        hops.rollout_random(s, 1, SEED, ops=JAX_STEP, flags=RANDOM, step_offset=5 + t, inplace=True)
    assert torch.equal(traj.state, s)
    del traj
    torch.cuda.empty_cache()


# ---------------------------------------------------------------- GameBatch.record


@gpu
def test_game_batch_record():
    import torch
    from hironaka_b200 import ops as hops
    from hironaka_b200.engine import GameBatch
    rng = np.random.default_rng(9)
    x = torch.as_tensor(start_state(rng, 300, 20, 3, np.int32, 9)).cuda()
    gb = GameBatch(x.clone(), host_policy="random", agent_policy="random", seed=SEED, role="agent")
    a = gb.record(steps=5, agent_obs=True)
    b = gb.record(steps=4, scale_observation=False, sort="coord0")
    assert gb.steps_played == 9
    s = x.clone()
    ra = hops.rollout_record(s, 5, ops=gb.ops, flags=gb.flags | C.HK_F_OBS_SORT_LEX | C.HK_F_OBS_RESCALE, seed=SEED,
                             agent_obs=True)
    rb = hops.rollout_record(s, 4, ops=gb.ops, flags=gb.flags | C.HK_F_OBS_SORT_COORD0, seed=SEED, step_offset=5)
    for got, exp in ((a, ra), (b, rb)):
        for name, g_, e_ in zip(NAMES[1:], got[1:], exp[1:]):
            assert torch.equal(g_, e_), name
    assert torch.equal(gb.points, s)
    assert gb.census is None or not gb.census.any()
    assert a.obs.shape == (5, 300, 63) and b.obs.shape == (4, 300, 60)
    # stream players: the batch's flags, no step counter
    gs = GameBatch(x.clone(), semantics="torch")
    ha = torch.randint(0, 4, (3, 300), dtype=torch.int32, device="cuda")
    ax = torch.randint(0, 3, (3, 300), dtype=torch.int32, device="cuda")
    c = gs.record(host_actions=ha, axes=ax, sort="none")
    assert gs.steps_played == 0
    rc = hops.rollout_record(x.clone(), None, ha, ax, ops=gs.ops, flags=gs.flags | C.HK_F_OBS_RESCALE)
    for name, g_, e_ in zip(NAMES, c, rc):
        assert torch.equal(g_, e_), name
    assert torch.equal(c.host_mask, hops.coords_to_mask(torch.as_tensor(O.decode_table(3)).cuda(), 3, "cuda")[ha.long()])
