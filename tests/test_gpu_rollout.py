"""One-launch rollouts (hk_rollout, hk_rollout_seeded) against the oracle's C port applied step by step.

A rollout keeps the state on chip for T steps and has code of its own in both kernel families: the thread-per-game
kernel re-tiers its warps as games end and fetches the next step's actions ahead; the warp-per-game kernel keeps one
compact row per lane for all T steps and rebuilds that list once half its rows have died, while games with more than
32 live rows, or already ended at entry, take the padded route.  The tests call the C-ABI directly and fill every
output with a sentinel first, so that a game or a step the kernel never writes cannot pass unnoticed, and compare bit
for bit: the state (float32 states by their bits), done_t and reward_t after every step (rewards by their bits: the
agent role writes -0.0), length (0 if done at entry, T + 1 if never done) and done_count, which is incremented.

The tests without the gpu mark check this file's own reference side (action encoders, the int64 range guard, the
oracle rollout) and run anywhere.
"""
import numpy as np
import pytest

from hironaka_b200 import constants as C
from oracle import cport
from oracle import hk_oracle as O
from tests.test_gpu_parity import SHAPES

gpu = pytest.mark.gpu

TORCH_FLAGS = C.HK_F_NOOP_INVALID | C.HK_F_FREEZE_ENDED
JAX_STEP = C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON
FUSED_STEP = C.HK_OP_SHIFT | C.HK_OP_NEWTON
INT32_BOUND = 1 << 30  # int32 states are exact below this (Elem<int32_t>, hk_common.cuh)

SENTINEL_WORD = np.uint32(0xABABABAB)  # a negative int32 and a negative float32: reads as a dead row holding junk
SENTINEL_REWARD = np.uint32(0x7FC0DEAD)  # a quiet NaN
DONE_COUNT_BASE = 1000  # done_count is incremented: it starts here


# ---------------------------------------------------------------- reference side (no GPU)


def decode_ids(ids, d):
    """Discrete host ids -> coordinate bitmasks (decode_table, bit k <=> coordinate k)."""
    table = (O.decode_table(d).astype(np.int64) << np.arange(d)).sum(1)
    return table[np.asarray(ids)].astype(np.int32)


def host_masks(ha, d, flags):
    return decode_ids(ha, d) if flags & C.HK_F_ACT_DISCRETE else np.asarray(ha, dtype=np.int32)


def shift_i64(x, masks, axes, flags, pad=-1):
    """The shift in int64 arithmetic: x_a <- sum of the chosen coordinates on live rows, dead rows padded.  No sum can
    wrap, so its maximum bounds every entry of an int32 step (reposition and the filter only lower or remove)."""
    B, N, d = x.shape
    x64 = x.astype(np.int64)
    live = x64[:, :, 0] >= 0
    masks = np.asarray(masks, dtype=np.int64)
    axes = np.asarray(axes, dtype=np.int64)
    bits = (masks[:, None] >> np.arange(d)) & 1
    sums = (x64 * bits[:, None, :]).sum(2)
    apply = (axes >= 0) & (axes < d)
    if flags & C.HK_F_NOOP_INVALID:
        apply &= ((masks >> np.clip(axes, 0, 62)) & 1) == 1
    if flags & C.HK_F_FREEZE_ENDED:
        apply &= live.sum(1) >= 2
    out = x64.copy()
    b, n = np.nonzero(apply[:, None] & live)
    out[b, n, axes[b]] = sums[b, n]
    out[~live] = pad
    return out


def live_max_i64(x):
    """Largest live entry of a state, taken on an int64 copy."""
    x64 = x.astype(np.int64)
    live = x64[:, :, 0] >= 0
    return int(x64[live].max()) if live.any() else 0


def pack_bytes(ha, ax):
    """HK_F_ACT_PACKED: one byte per game-step, host action (< 32) in the low 5 bits, axis (< 8) in the high 3."""
    ha, ax = np.asarray(ha), np.asarray(ax)
    assert (ha >= 0).all() and (ha < 32).all() and (ax >= 0).all() and (ax < 8).all()
    return (ha.astype(np.uint8) | (ax.astype(np.uint8) << 5)).astype(np.uint8)


def pack_nibbles(ha, ax):
    """HK_F_ACT_NIBBLE: [T, B] ids (< 4) and axes (< 4) -> uint8 [T, ceil(B / 2)], game 2i in the low nibble of byte
    i of its step's row, game 2i + 1 in the high nibble (odd B: the last high nibble is unused)."""
    ha, ax = np.asarray(ha), np.asarray(ax)
    assert (ha >= 0).all() and (ha < 4).all() and (ax >= 0).all() and (ax < 4).all()
    T, B = ha.shape
    nib = np.zeros((T, 2 * ((B + 1) // 2)), np.uint8)
    nib[:, :B] = ha | (ax << 2)
    return (nib[:, 0::2] | (nib[:, 1::2] << 4)).astype(np.uint8)


def unpack_nibbles(buf, B, T):
    """The reading rule of load_actions: the byte of game g at step st is st * ((B + 1) >> 1) + (g >> 1) of the flat
    stream, its high nibble for odd g."""
    flat = np.ascontiguousarray(buf).reshape(-1)
    st, g = np.meshgrid(np.arange(T), np.arange(B), indexing="ij")
    byte = flat[st * ((B + 1) >> 1) + (g >> 1)].astype(np.int32)
    nib = np.where(g & 1, byte >> 4, byte & 15)
    return nib & 3, nib >> 2


def unpack_bytes(buf):
    b = np.asarray(buf).astype(np.int32)
    return b & 31, b >> 5


def oracle_rollout(x, ha, ax, ops, flags, pad=-1.0, T=None):
    """T steps of the C port: (state, done [T, B] uint8, reward [T, B] float32, finished games per step [T], length [B])."""
    T = T if T is not None else (ha if ha is not None else ax).shape[0]
    B = x.shape[0]
    o = np.ascontiguousarray(x)
    length = np.where((o[:, :, 0] >= 0).sum(1) < 2, 0, T + 1).astype(np.int32)
    done = np.empty((T, B), np.uint8)
    reward = np.empty((T, B), np.float32)
    for t in range(T):
        o, done[t], reward[t], _ = cport.step(o, None if ha is None else ha[t], None if ax is None else ax[t], ops, flags,
                                              padding_value=pad)
        length[(length == T + 1) & (done[t] != 0)] = t + 1
    return o, done, reward, done.sum(1).astype(np.int32), length


def start_state(rng, B, N, d, dtype, max_value, pad=-1.0):
    """Random games with junk in dead rows (negative coordinate 0, anything after it), empty games, lone points away
    from the origin and duplicated rows."""
    x = rng.integers(0, max_value + 1, size=(B, N, d)).astype(dtype)
    dead = rng.random((B, N)) < rng.choice([0.0, 0.2, 0.5, 0.8], size=(B, 1))
    x[dead] = pad
    junk = dead & (rng.random((B, N)) < 0.3)
    x[junk, 0] = -7 if dtype == np.int32 else -0.5
    if d > 1:
        x[junk & (rng.random((B, N)) < 0.5), 1] = 3
    for b in np.nonzero(rng.random(B) < 0.3)[0]:
        i, j = rng.integers(0, N, 2)
        x[b, j] = x[b, i]
    x[3::7] = pad  # empty games
    x[5::7, 1:] = pad  # lone points, away from the origin
    x[5::7, 0] = rng.integers(1, max_value + 2, size=(x[5::7].shape[0], d))
    return x


def bits(a):
    return a.view(np.int32) if a.dtype == np.float32 else a


def test_packed_and_nibble_encoders_round_trip():
    from hironaka_b200.session import HostSession
    rng = np.random.default_rng(1)
    for B in (1, 3, 33, 101):
        T = 5
        ha, ax = rng.integers(0, 4, (T, B)), rng.integers(0, 4, (T, B))
        nib = pack_nibbles(ha, ax)
        assert nib.shape == (T, (B + 1) // 2)
        assert np.array_equal(nib, HostSession.pack_actions_nibble(ha, ax))
        h2, a2 = unpack_nibbles(nib, B, T)
        assert np.array_equal(h2, ha) and np.array_equal(a2, ax), B
        if B > 1 and B % 2:  # the rows of an odd batch are (B + 1) / 2 bytes apart: B // 2 reads other bytes
            wrong = nib.reshape(-1)[np.arange(T)[:, None] * (B >> 1) + (np.arange(B) >> 1)]
            assert not np.array_equal(np.where(np.arange(B) & 1, wrong >> 4, wrong & 15) & 3, ha)
        ha, ax = rng.integers(0, 32, (T, B)), rng.integers(0, 8, (T, B))
        pk = pack_bytes(ha, ax)
        assert np.array_equal(pk, HostSession.pack_actions(ha, ax))
        h2, a2 = unpack_bytes(pk)
        assert np.array_equal(h2, ha) and np.array_equal(a2, ax), B


def test_int64_shift_guard_agrees_with_cport():
    rng = np.random.default_rng(2)
    for (B, N, d) in ((300, 7, 3), (200, 5, 4), (100, 4, 2), (50, 6, 5)):
        for flags in (0, C.HK_F_NOOP_INVALID, TORCH_FLAGS, C.HK_F_ACT_DISCRETE, C.HK_F_FREEZE_ENDED | C.HK_F_ACT_DISCRETE):
            x = start_state(rng, B, N, d, np.int32, (1 << 24) - 1)
            x[x[:, :, 0] < 0] = -1  # dead rows padded: every entry is then defined by the shift
            if flags & C.HK_F_ACT_DISCRETE:
                ha = rng.integers(0, 2 ** d - d - 1, B)
            else:
                ha = rng.integers(0, 2 ** d, B)
            ax = rng.integers(-1, d + 1, B)
            exp = cport.step(x, ha, ax, C.HK_OP_SHIFT, flags)[0]
            got = shift_i64(x, host_masks(ha, d, flags), ax, flags)
            assert np.array_equal(got, exp.astype(np.int64)), (B, N, d, flags)
            assert live_max_i64(exp) == live_max_i64(got)
    # above the int32 range the int64 copy keeps the sum that the int32 arithmetic would wrap
    x = np.full((1, 2, 3), (1 << 30) + 5, np.int32)
    assert live_max_i64(shift_i64(x, [7], [0], 0)) == 3 * ((1 << 30) + 5)


def test_oracle_rollout_composes_and_counts():
    rng = np.random.default_rng(3)
    B, N, d, T = 200, 10, 3, 14
    x = start_state(rng, B, N, d, np.int32, 6)
    ha, ax = rng.integers(0, 4, (T, B)).astype(np.int32), rng.integers(0, d, (T, B)).astype(np.int32)
    full = oracle_rollout(x, ha, ax, JAX_STEP, C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT)
    a = oracle_rollout(x, ha[:5], ax[:5], JAX_STEP, C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT)
    b = oracle_rollout(a[0], ha[5:], ax[5:], JAX_STEP, C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT)
    assert np.array_equal(full[0], b[0])
    assert np.array_equal(full[1], np.concatenate([a[1], b[1]])) and np.array_equal(full[2], np.concatenate([a[2], b[2]]))
    done_at_entry = (x[:, :, 0] >= 0).sum(1) < 2
    first = np.where(full[1].any(0), full[1].argmax(0) + 1, T + 1)
    assert np.array_equal(full[4], np.where(done_at_entry, 0, first))
    assert 0 < (full[4] == T + 1).sum() < B and (full[4] == 0).sum() > 0
    assert np.array_equal(full[3], full[1].sum(1))
    # the agent's reward is -0.0 where nothing happened: only a bitwise comparison tells it from +0.0
    r = full[2]
    assert (r.view(np.int32) == np.float32(-0.0).view(np.int32)).any() and (r == -1.0).any()


# ---------------------------------------------------------------- GPU helpers


def _dev(a):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def _filled(shape, word, dtype):
    import torch
    t = torch.empty(shape, dtype=torch.int32, device="cuda")
    t.fill_(int(np.uint32(word).view(np.int32)))
    return t.view(dtype)


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


@pytest.fixture(scope="module")
def lib():
    import torch
    from hironaka_b200 import ops
    from hironaka_b200._lib import lib as _lib
    assert torch.cuda.is_available()
    ops.force_generic(False)
    yield _lib()
    ops.force_generic(False)


FAMILIES = (False, True)  # the dispatcher's choice; the warp-per-game kernel forced onto every shape


def gpu_rollout(L, x, ha, ax, ops, flags, pad=-1.0, inplace=False, T=None, seed=None, step_offset=0):
    """hk_rollout (hk_rollout_seeded when `seed` is given) through the C-ABI with every output pre-filled with a
    sentinel.  Returns (rc, state, done [T, B], reward [T, B], done_count increments [T], length [B])."""
    import torch
    B, N, d = x.shape
    T = T if T is not None else (ha if ha is not None else ax).shape[0]
    xin = _dev(x)
    out = xin if inplace else _filled(x.shape, SENTINEL_WORD, xin.dtype)
    done = torch.full((T, B), 0xAB, dtype=torch.uint8, device="cuda")
    reward = _filled((T, B), SENTINEL_REWARD, torch.float32)
    dcount = torch.full((T,), DONE_COUNT_BASE, dtype=torch.int32, device="cuda")
    length = _filled((B,), SENTINEL_WORD, torch.int32)
    ha_d = None if ha is None else _dev(ha)
    ax_d = None if ax is None else _dev(ax)
    ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    dt = C.HK_DTYPE_I32 if x.dtype == np.int32 else C.HK_DTYPE_F32
    if seed is None:
        rc = L.hk_rollout(xin.data_ptr(), out.data_ptr(), ptr(ha_d), ptr(ax_d), done.data_ptr(), reward.data_ptr(),
                          dcount.data_ptr(), length.data_ptr(), B, N, d, T, dt, ops, flags, float(pad), _stream())
    else:
        rc = L.hk_rollout_seeded(xin.data_ptr(), out.data_ptr(), ptr(ha_d), ptr(ax_d), done.data_ptr(), reward.data_ptr(),
                                 dcount.data_ptr(), length.data_ptr(), B, N, d, T, dt, ops, flags, float(pad),
                                 seed & (2 ** 64 - 1), step_offset, _stream())
    if rc != 0:
        return rc, None, None, None, None, None
    return (rc, out.cpu().numpy(), done.cpu().numpy(), reward.cpu().numpy(), dcount.cpu().numpy() - DONE_COUNT_BASE,
            length.cpu().numpy())


def assert_rollout(got, exp, what):
    rc, state, done, reward, dcount, length = got
    o, odone, oreward, ocount, olength = exp
    assert rc == 0, (what, rc)
    assert np.array_equal(bits(state), bits(o)), (what, "state")
    for t in range(odone.shape[0]):
        assert np.array_equal(done[t], odone[t]), (what, "done_t", t)
        assert np.array_equal(reward[t].view(np.int32), oreward[t].view(np.int32)), (what, "reward_t", t)
    assert np.array_equal(dcount, ocount), (what, "done_count")
    assert np.array_equal(length, olength), (what, "length")


def check_both_families(L, x, ha, ax, ops, flags, exp, what, pad=-1.0, **kw):
    from hironaka_b200 import ops as hops
    for generic in FAMILIES:
        hops.force_generic(generic)
        try:
            for inplace in (False, True):
                assert_rollout(gpu_rollout(L, x, ha, ax, ops, flags, pad=pad, inplace=inplace, **kw), exp,
                               (what, "generic" if generic else "auto", "in place" if inplace else "out of place"))
        finally:
            hops.force_generic(False)


# ---------------------------------------------------------------- 1. shapes x modes


SWEEP_SHAPES = SHAPES + [(1, 20, 3), (1, 64, 5), (33, 20, 3), (65, 10, 3), (97, 5, 3), (129, 16, 4), (33, 2, 2)]

# (name, ops, flags, padding value of a float32 state, of an int32 state)
MODES = [
    ("jax", JAX_STEP, 0, -1.0, -1.0),
    ("fused", FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE, -1.0, -1.0),
    ("agent", JAX_STEP, C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT, -1.0, -1.0),
    ("shift_freeze", C.HK_OP_SHIFT, C.HK_F_FREEZE_ENDED, -1.0, -1.0),
    ("freeze_newton", FUSED_STEP, C.HK_F_FREEZE_ENDED | C.HK_F_ROLE_AGENT, -1.0, -1.0),
    ("noop_invalid", JAX_STEP, C.HK_F_NOOP_INVALID, -1.0, -1.0),
    ("newton", C.HK_OP_NEWTON, 0, -1.0, -1.0),
    ("repos_dedupe", C.HK_OP_REPOSITION | C.HK_OP_DEDUPE, 0, -1.0, -1.0),
    ("shift_dedupe", C.HK_OP_SHIFT | C.HK_OP_DEDUPE, C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT, -1.0, -1.0),
    ("reposition", C.HK_OP_REPOSITION, 0, -1.0, -1.0),
    ("observe", 0, 0, -1.0, -1.0),
    ("fused_rescale", FUSED_STEP | C.HK_OP_RESCALE, TORCH_FLAGS | C.HK_F_ACT_DISCRETE, -1.0, -1.0),
    ("jax_rescale_eps", JAX_STEP | C.HK_OP_RESCALE, C.HK_F_RESCALE_EPS, -1.0, -1.0),
    ("rescale", C.HK_OP_RESCALE, 0, -1.0, -1.0),
    ("fused_padding", FUSED_STEP, TORCH_FLAGS, -1e-8, -3.0),
]


def random_actions(rng, T, B, d, flags):
    """[T, B] streams: discrete ids or arbitrary bitmasks (empty sets and singletons included); about one axis in ten
    is out of range (-1 or d)."""
    ncls = 2 ** d - d - 1
    ha = rng.integers(0, ncls, (T, B)) if flags & C.HK_F_ACT_DISCRETE else rng.integers(0, 2 ** d, (T, B))
    ax = rng.integers(0, d, (T, B))
    bad = rng.random((T, B)) < 0.1
    ax[bad] = rng.choice([-1, d], size=int(bad.sum()))
    return ha.astype(np.int32), ax.astype(np.int32)


@gpu
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
@pytest.mark.parametrize("shape", SWEEP_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_rollout_modes(lib, shape, dtype):
    B, N, d = shape
    rng = np.random.default_rng(B * 1000 + N * 10 + d)
    for name, ops, flags, pad_f, pad_i in MODES:
        pad = pad_f if dtype == np.float32 else pad_i
        T = int(rng.integers(12, 25))
        x = start_state(rng, B, N, d, dtype, max_value=int(rng.choice([1, 3, 20, 1000])), pad=pad)
        ha, ax = random_actions(rng, T, B, d, flags)
        if ops & C.HK_OP_RESCALE and dtype == np.int32:  # rescale is not defined on an int32 state
            for inplace in (False, True):
                assert gpu_rollout(lib, x, ha, ax, ops, flags, pad=pad, inplace=inplace)[0] == C.HK_ERR_UNSUPPORTED, name
            continue
        exp = oracle_rollout(x, ha, ax, ops, flags, pad=pad)
        check_both_families(lib, x, ha, ax, ops, flags, exp, (name, T), pad=pad)


@gpu
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
def test_dedupe_rollout_ignores_rows_that_died_earlier(lib, dtype):
    """Regression: the remove_repeated pass of a multi-step rollout took a row's liveness from its data, and a row
    killed in an earlier step still holds its old values in the warp's game slot (dead rows are padded on the way
    out).  Row 1 duplicates row 0 and dies at step 1 holding (1, 2); at step 2 row 2 becomes (1, 2) and was killed
    as its copy."""
    x = np.array([[[1, 1], [1, 1], [1, 0], [-1, -1]]], dtype)
    x = np.concatenate([x, x[:, [0, 1, 3, 2]], x[:, ::-1]])  # the same game with its rows in other slots
    ha = np.full((2, 3), 0b11, np.int32)
    ax = np.ones((2, 3), np.int32)
    ops = C.HK_OP_SHIFT | C.HK_OP_DEDUPE
    exp = oracle_rollout(x, ha, ax, ops, 0)
    assert exp[0][0].tolist() == [[1, 3], [-1, -1], [1, 2], [-1, -1]]
    assert exp[1].tolist() == [[0, 0, 0], [0, 0, 0]]
    check_both_families(lib, x, ha, ax, ops, 0, exp, "dedupe")


def antichain_state(rng, B, N, d, total, dtype):
    """Games whose rows lie on the hyperplane sum = total: no row dominates another, so the filter keeps them all and
    more than 32 rows stay live for several steps."""
    x = np.empty((B, N, d), np.int64)
    for b in range(B):
        cuts = np.sort(rng.integers(0, total + 1, (N, d - 1)), axis=1)
        x[b] = np.diff(np.concatenate([np.zeros((N, 1), np.int64), cuts, np.full((N, 1), total)], axis=1), axis=1)
    x = x.astype(dtype)
    x[1::4, -3:] = -1
    x[2::4, rng.integers(0, N, 3)] = -9 if dtype == np.int32 else -0.25
    return x


@gpu
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
@pytest.mark.parametrize("shape", [(34, 40, 3), (33, 64, 5), (9, 100, 3), (12, 64, 4)], ids=lambda s: "x".join(map(str, s)))
def test_rollout_many_live_rows(lib, shape, dtype):
    """Games that start with more than 32 live rows take the warp-per-game kernel's padded route for every step."""
    B, N, d = shape
    rng = np.random.default_rng(N * 10 + d)
    for name, ops, flags, pad_f, pad_i in MODES:
        if name in ("observe", "reposition", "rescale") or (ops & C.HK_OP_RESCALE and dtype == np.int32):
            continue
        T = int(rng.integers(12, 25))
        x = antichain_state(rng, B, N, d, 4 * N, dtype)
        ha, ax = random_actions(rng, T, B, d, flags)
        exp = oracle_rollout(x, ha, ax, ops, flags)
        after1 = oracle_rollout(x, ha[:1], ax[:1], ops, flags)[0]
        assert ((after1[:, :, 0] >= 0).sum(1) > 32).any(), name  # the start does what it is for
        check_both_families(lib, x, ha, ax, ops, flags, exp, (name, T))


# ---------------------------------------------------------------- single steps: every output written


@gpu
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
@pytest.mark.parametrize("shape", [(70, 20, 3), (33, 10, 3), (31, 5, 3), (40, 16, 4), (5, 64, 5), (3, 40, 2)],
                         ids=lambda s: "x".join(map(str, s)))
def test_step_out_of_place_writes_unchanged_games(lib, shape, dtype):
    """hk_step out of place on games the step does not change (ended, frozen, invalid axis, at rest): every game of
    the output, and every done / reward / num_points entry, must be written."""
    import torch
    from hironaka_b200 import ops as hops
    B, N, d = shape
    rng = np.random.default_rng(B + N + d)
    x = start_state(rng, B, N, d, dtype, 9)
    for ops, flags in ((FUSED_STEP, TORCH_FLAGS), (JAX_STEP, C.HK_F_ROLE_AGENT)):
        root = C.HK_OP_NEWTON | (ops & C.HK_OP_REPOSITION)
        x0 = cport.step(x, None, None, root, 0)[0]  # filtered (and repositioned): twice, since the filter can remove
        x0 = cport.step(x0, None, None, root, 0)[0]  # the row that held a coordinate's minimum
        ended = (x0[:, :, 0] >= 0).sum(1) < 2
        ha = rng.integers(0, 2 ** d, B).astype(np.int32)
        ax = rng.integers(0, d, B).astype(np.int32)
        if flags & C.HK_F_NOOP_INVALID:  # the axis is not among the chosen coordinates: nothing moves
            ha = np.where((ha >> ax) & 1, ha & ~(1 << ax), ha).astype(np.int32)
        else:  # the axis is out of range: nothing moves
            ax = rng.choice([-1, d, 7], B).astype(np.int32)
        if not ops & C.HK_OP_REPOSITION:  # ended games are frozen whatever their action
            ha[ended] = (2 ** d) - 1
            ax[ended] = 0
        o, od, orw, onp = cport.step(x0, ha, ax, ops, flags)
        assert np.array_equal(bits(o), bits(x0)), "the inputs are meant to stay unchanged"
        for generic in FAMILIES:
            hops.force_generic(generic)
            try:
                xin = _dev(x0)
                out = _filled(x0.shape, SENTINEL_WORD, xin.dtype)
                done = torch.full((B,), 0xAB, dtype=torch.uint8, device="cuda")
                rew = _filled((B,), SENTINEL_REWARD, torch.float32)
                npts = _filled((B,), SENTINEL_WORD, torch.int32)
                ha_d, ax_d = _dev(ha), _dev(ax)
                rc = lib.hk_step(xin.data_ptr(), out.data_ptr(), ha_d.data_ptr(), ax_d.data_ptr(), done.data_ptr(),
                                 rew.data_ptr(), npts.data_ptr(), None, None, None, B, N, d,
                                 C.HK_DTYPE_I32 if dtype == np.int32 else C.HK_DTYPE_F32, ops, flags, -1.0, 1e8, _stream())
                assert rc == 0
                what = (ops, flags, generic)
                assert np.array_equal(bits(out.cpu().numpy()), bits(o)), what
                assert np.array_equal(done.cpu().numpy(), od), what
                assert np.array_equal(rew.cpu().numpy().view(np.int32), orw.view(np.int32)), what
                assert np.array_equal(npts.cpu().numpy(), onp), what
                # ops.step with out= (a caller-owned buffer that holds something else)
                dst = _filled(x0.shape, SENTINEL_WORD, xin.dtype)
                r = hops.step(xin, ha_d, ax_d, ops=ops, flags=flags, inplace=False, out=dst, want_done=True)
                assert r.state.data_ptr() == dst.data_ptr()
                assert np.array_equal(bits(dst.cpu().numpy()), bits(o)), what
            finally:
                hops.force_generic(False)


# ---------------------------------------------------------------- 2. composition


@gpu
@pytest.mark.parametrize("shape", [(257, 20, 3), (33, 10, 3), (40, 16, 4), (16, 64, 5), (3, 300, 6), (50, 7, 2)],
                         ids=lambda s: "x".join(map(str, s)))
def test_rollout_composes(lib, shape):
    """rollout(T) = rollout(T1) then rollout(T - T1) on the rest of the streams = T calls of hk_step.  T = 70 runs
    past the 64 steps whose finished counts the warp-per-game kernel gathers in registers."""
    import torch
    from hironaka_b200 import ops as hops
    B, N, d = shape
    rng = np.random.default_rng(B * 7 + N)
    for dtype in (np.int32, np.float32):
        for ops, flags, T in ((JAX_STEP, C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT, 70),
                              (FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE, 16)):
            x = start_state(rng, B, N, d, dtype, 12)
            ha, ax = random_actions(rng, T, B, d, flags)
            exp = oracle_rollout(x, ha, ax, ops, flags)
            for generic in FAMILIES:
                hops.force_generic(generic)
                try:
                    what = (dtype.__name__, ops, T, generic)
                    full = gpu_rollout(lib, x, ha, ax, ops, flags)
                    assert_rollout(full, exp, what)
                    for T1 in (1, T // 2 + 1, T - 1):
                        a = gpu_rollout(lib, x, ha[:T1], ax[:T1], ops, flags)
                        b = gpu_rollout(lib, a[1], ha[T1:], ax[T1:], ops, flags, inplace=True)
                        assert np.array_equal(bits(b[1]), bits(full[1])), (what, T1)
                        for k in (2, 3, 4):  # done_t, reward_t, done_count
                            assert np.array_equal(bits(np.concatenate([a[k], b[k]])), bits(full[k])), (what, T1, k)
                    g = _dev(x)
                    for t in range(T):
                        r = hops.step(g, _dev(ha[t]), _dev(ax[t]), ops=ops, flags=flags, inplace=True, want_done=True,
                                      want_reward=True)
                        assert np.array_equal(r.done.cpu().numpy(), full[2][t].astype(bool)), (what, t)
                        assert np.array_equal(r.reward.cpu().numpy().view(np.int32), full[3][t].view(np.int32)), (what, t)
                    assert np.array_equal(bits(g.cpu().numpy()), bits(full[1])), what
                finally:
                    hops.force_generic(False)
    torch.cuda.synchronize()


# ---------------------------------------------------------------- 3. action formats


@gpu
@pytest.mark.parametrize("shape", [(101, 20, 3), (33, 10, 3), (65, 5, 3), (31, 7, 2), (45, 16, 4), (17, 64, 5), (3, 33, 3),
                                   (1, 5, 3), (5, 9, 6)], ids=lambda s: "x".join(map(str, s)))
def test_rollout_action_formats(lib, shape):
    """int32, uint8 (HK_F_ACT_U8), one byte (HK_F_ACT_PACKED, d <= 5) and half a byte (HK_F_ACT_NIBBLE, d <= 3) per
    game-step, all with T > 1 and odd batch sizes: each stream gives exactly the int32 stream's rollout.  Out-of-range
    axes are written in each format's own way (-1 / d / 7 as int32, 255 as uint8, 7 packed, 3 in a nibble)."""
    B, N, d = shape
    rng = np.random.default_rng(B + 3 * N + d)
    T = 15
    ncls = 2 ** d - d - 1
    for dtype in (np.int32, np.float32):
        x = start_state(rng, B, N, d, dtype, 10)
        for ops, base in ((JAX_STEP, C.HK_F_ACT_DISCRETE), (JAX_STEP, 0), (FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE),
                          (FUSED_STEP, TORCH_FLAGS)):
            discrete = bool(base & C.HK_F_ACT_DISCRETE)
            nibble = discrete and d <= 3
            hi = (min(ncls, 4) if nibble else ncls) if discrete else 2 ** d
            ha = rng.integers(0, hi, (T, B)).astype(np.int32)
            ax = rng.integers(0, d, (T, B)).astype(np.int32)
            bad = rng.random((T, B)) < 0.15
            if nibble:  # an axis a nibble can carry and the game does not have
                ax[bad] = 3
            elif d <= 5:
                ax[bad] = 7
            else:
                ax[bad] = rng.choice([-1, d], int(bad.sum()))
            exp = oracle_rollout(x, ha, ax, ops, base)
            streams = [("int32", ha, ax, base)]
            u8_ax = np.where(ax < 0, 255, ax).astype(np.uint8)
            streams.append(("u8", ha.astype(np.uint8), u8_ax, base | C.HK_F_ACT_U8))
            if d <= 5:
                streams.append(("packed", pack_bytes(ha, ax), None, base | C.HK_F_ACT_PACKED))
            if nibble:
                streams.append(("nibble", pack_nibbles(ha, ax), None, base | C.HK_F_ACT_NIBBLE))
            for fmt, h, a, flags in streams:
                check_both_families(lib, x, h, a, ops, flags, exp, (fmt, dtype.__name__, ops, base), T=T)
            # where a format cannot carry the actions, the library refuses the call
            if d > 5:
                assert gpu_rollout(lib, x, pack_bytes(ha % 32, ax % 8), None, ops, base | C.HK_F_ACT_PACKED,
                                   T=T)[0] == C.HK_ERR_BAD_ARG
            if d > 3 or not discrete:
                assert gpu_rollout(lib, x, np.zeros((T, (B + 1) // 2), np.uint8), None, ops, base | C.HK_F_ACT_NIBBLE,
                                   T=T)[0] == C.HK_ERR_BAD_ARG


# ---------------------------------------------------------------- 4. value ranges


def order_sensitive_state(rng, B, N, d):
    """float32 games whose shifted sums depend on the order of summation: integers in [2^24, 2^26] (most with the
    lowest significand bit set) or mixed magnitudes (1e7 next to 0.375)."""
    big = rng.integers(1 << 24, 1 << 26, (B, N, d)).astype(np.float32)
    mixed = rng.choice(np.array([1e7, 0.375, 3.0, 12345.678, 2.5e6 + 0.5, 0.0], np.float32), (B, N, d))
    mixed = (mixed * rng.choice(np.array([1.0, 3.0, 0.5], np.float32), (B, N, d))).astype(np.float32)
    x = np.where(rng.random((B, 1, 1)) < 0.5, big, mixed).astype(np.float32)
    x[rng.random((B, N)) < 0.25] = -1.0
    x[::9] = -1.0
    return x


def wide_masks(rng, T, B, d):
    """Bitmasks with three or more coordinates where the dimension allows it."""
    full = (1 << d) - 1
    if d < 3:
        return np.full((T, B), full, np.int32)
    m = rng.integers(0, 1 << d, (T, B))
    pc = np.vectorize(lambda v: bin(int(v)).count("1"))(m)
    return np.where(pc >= 3, m, full).astype(np.int32)


@gpu
@pytest.mark.parametrize("shape", [(96, 20, 3), (64, 10, 3), (64, 5, 3), (40, 16, 4), (20, 64, 5), (33, 7, 4), (9, 4, 10)],
                         ids=lambda s: "x".join(map(str, s)))
def test_float32_summation_order(lib, shape):
    """The kernels sum the chosen coordinates left to right, as the reference does: single steps and rollouts with and
    without reposition on values where the order decides the result, and a long FusedGame-flavour rollout (no
    reposition, 40 steps) in which the values keep growing."""
    from hironaka_b200 import ops as hops
    B, N, d = shape
    rng = np.random.default_rng(N * 31 + d)
    x = order_sensitive_state(rng, B, N, d)
    for ops, flags in ((JAX_STEP, 0), (FUSED_STEP, TORCH_FLAGS), (C.HK_OP_SHIFT, 0)):
        T = 12
        ha, ax = wide_masks(rng, T, B, d), rng.integers(0, d, (T, B)).astype(np.int32)
        # single steps (hk_step) on the start state
        o = cport.step(x, ha[0], ax[0], ops, flags)[0]
        left_to_right = cport.step(x, ha[0], ax[0], C.HK_OP_SHIFT, 0)[0]
        for generic in FAMILIES:
            hops.force_generic(generic)
            try:
                g = hops.step(_dev(x), _dev(ha[0]), _dev(ax[0]), ops=ops, flags=flags, inplace=False).state.cpu().numpy()
                assert np.array_equal(bits(g), bits(o)), (ops, generic)
            finally:
                hops.force_generic(False)
        check_both_families(lib, x, ha, ax, ops, flags, oracle_rollout(x, ha, ax, ops, flags), (ops, flags, T))
    # the inputs do what they are for: another order of summation gives other sums
    live = x[:, :, 0] >= 0
    sel = (ha[0][:, None] >> np.arange(d)) & 1
    rev = np.zeros(x.shape[:2], np.float32)
    for k in reversed(range(d)):
        rev = np.where(sel[:, None, k] == 1, (rev + x[:, :, k]).astype(np.float32), rev)
    fwd = left_to_right[np.arange(B), :, ax[0]]
    assert (rev[live] != fwd[live]).any()
    # long FusedGame-flavour rollout: shift -> newton, no reposition, discrete ids, values growing
    if d <= 5:
        T = 40
        ncls = 2 ** d - d - 1
        ha = rng.integers(0, ncls, (T, B)).astype(np.int32)
        ax = rng.integers(0, d, (T, B)).astype(np.int32)
        flags = TORCH_FLAGS | C.HK_F_ACT_DISCRETE
        exp = oracle_rollout(x, ha, ax, FUSED_STEP, flags)
        assert np.isfinite(exp[0]).all() and exp[0].max() < 1e37
        check_both_families(lib, x, ha, ax, FUSED_STEP, flags, exp, ("long", T))


def tame_int32_actions(x, ha, ax, ops, flags):
    """Walk the oracle through the streams and turn the axis of any game-step whose shift would reach 2^30 into -1
    (no shift), asserting on int64 copies that every state stays inside int32's documented range."""
    d = x.shape[2]
    ax = ax.copy()
    o = x
    kept = 0
    for t in range(ha.shape[0]):
        s = shift_i64(o, host_masks(ha[t], d, flags), ax[t], flags)
        live = s[:, :, 0] >= 0
        over = (np.where(live[:, :, None], s, 0) >= INT32_BOUND).any((1, 2))
        ax[t, over] = -1
        kept += int((~over).sum())
        assert live_max_i64(shift_i64(o, host_masks(ha[t], d, flags), ax[t], flags)) < INT32_BOUND
        o = cport.step(o, ha[t], ax[t], ops, flags)[0]
        assert live_max_i64(o) < INT32_BOUND, t
    return ax, kept


@gpu
@pytest.mark.parametrize("shape", [(96, 20, 3), (64, 10, 3), (64, 5, 3), (40, 16, 4), (20, 64, 5), (33, 7, 2)],
                         ids=lambda s: "x".join(map(str, s)))
def test_int32_large_values(lib, shape):
    """int32 states with values in [2^24, 2^29]: exact integer arithmetic, single steps and rollouts, both families."""
    from hironaka_b200 import ops as hops
    B, N, d = shape
    rng = np.random.default_rng(N * 17 + d)
    T = 12
    for ops, flags in ((JAX_STEP, 0), (FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE), (JAX_STEP, C.HK_F_ACT_DISCRETE)):
        x = rng.integers(1 << 24, 1 << 29, (B, N, d)).astype(np.int32)
        x[rng.random((B, N)) < 0.3] = -1
        x[::6, :, 1:] //= 64  # one large coordinate next to smaller ones
        x[x[:, :, 0] < 0] = -1
        ncls = 2 ** d - d - 1
        ha = (rng.integers(0, ncls, (T, B)) if flags & C.HK_F_ACT_DISCRETE else rng.integers(0, 2 ** d, (T, B))).astype(np.int32)
        ax = rng.integers(0, d, (T, B)).astype(np.int32)
        ax, kept = tame_int32_actions(x, ha, ax, ops, flags)
        assert kept >= T * B // 4, kept  # most of the moves are played
        o = cport.step(x, ha[0], ax[0], ops, flags)[0]
        assert live_max_i64(o) >= 1 << 28
        for generic in FAMILIES:
            hops.force_generic(generic)
            try:
                g = hops.step(_dev(x), _dev(ha[0]), _dev(ax[0]), ops=ops, flags=flags, inplace=False).state.cpu().numpy()
                assert np.array_equal(g, o), (ops, flags, generic)
            finally:
                hops.force_generic(False)
        check_both_families(lib, x, ha, ax, ops, flags, oracle_rollout(x, ha, ax, ops, flags), (ops, flags))


# ---------------------------------------------------------------- 5. random and fixed players


SEED = 0xF1E2D3C4B5A69788  # high bits set: both key words matter
STEP_OFFSET = (1 << 30) - 7  # the step counter crosses 2^30 inside the rollout


@gpu
@pytest.mark.parametrize("shape", [(1, 5, 3), (33, 10, 3), (257, 20, 3), (64, 2, 2), (50, 7, 2), (9, 4, 10), (16, 64, 5),
                                   (5, 100, 3), (37, 33, 3)], ids=lambda s: "x".join(map(str, s)))
def test_seeded_rollout(lib, shape):
    """hk_rollout_seeded: players drawn in the kernel equal oracle.random_player_actions fed to the C port, with one or
    both players random, per step."""
    B, N, d = shape
    rng = np.random.default_rng(B + N * d)
    T = 14
    ha, ax = O.random_player_actions(B, d, T, SEED, STEP_OFFSET)
    assert ha.max() < 2 ** d - d - 1 and ax.max() < d
    for dtype in (np.int32, np.float32):
        x = start_state(rng, B, N, d, dtype, 15)
        for ops, flags in ((JAX_STEP, C.HK_F_ACT_DISCRETE), (FUSED_STEP, TORCH_FLAGS | C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT)):
            exp = oracle_rollout(x, ha, ax, ops, flags)
            kw = dict(T=T, seed=SEED, step_offset=STEP_OFFSET)
            check_both_families(lib, x, None, None, ops, flags | C.HK_F_HOST_RANDOM | C.HK_F_AGENT_RANDOM, exp,
                                ("both random", dtype.__name__), **kw)
            ax_s = rng.integers(0, d, (T, B)).astype(np.int32)
            check_both_families(lib, x, None, ax_s, ops, flags | C.HK_F_HOST_RANDOM,
                                oracle_rollout(x, ha, ax_s, ops, flags), ("host random", dtype.__name__), **kw)
            ha_s = rng.integers(0, 2 ** d - d - 1, (T, B)).astype(np.int32)
            check_both_families(lib, x, ha_s, None, ops, flags | C.HK_F_AGENT_RANDOM,
                                oracle_rollout(x, ha_s, ax, ops, flags), ("agent random", dtype.__name__), **kw)


F_ALL, F_ZEIL, F_FIRST, F_LAST = C.HK_F_HOST_ALL_COORD, C.HK_F_HOST_ZEILLINGER, C.HK_F_AGENT_FIRST, C.HK_F_AGENT_LAST


@gpu
@pytest.mark.parametrize("shape", [(40, 100, 3), (64, 7, 2), (96, 20, 3), (70, 10, 3)], ids=lambda s: "x".join(map(str, s)))
def test_fixed_players_rollout(lib, shape):
    """All-coordinates / Zeillinger hosts and first / last agents evaluated in the kernel, 12 steps in one launch:
    done_t and reward_t of every step, the finished counts, length and the state."""
    B, N, d = shape
    rng = np.random.default_rng(N + d + 1)
    T = 12
    ncls = 2 ** d - d - 1
    for dtype in (np.int32, np.float32):
        x = start_state(rng, B, N, d, dtype, 12)
        for pol in (F_ALL | F_FIRST, F_ALL | F_LAST, F_ZEIL | F_FIRST, F_ZEIL | F_LAST, F_ZEIL, F_FIRST, F_LAST):
            ha = rng.integers(0, ncls, (T, B)).astype(np.int32)
            ax = rng.integers(0, d, (T, B)).astype(np.int32)
            host_fixed, agent_fixed = pol & (F_ALL | F_ZEIL), pol & (F_FIRST | F_LAST)
            flags = pol | C.HK_F_ACT_DISCRETE | C.HK_F_ROLE_AGENT | (TORCH_FLAGS if (pol >> 8) % 2 else 0)
            h, a = None if host_fixed else ha, None if agent_fixed else ax
            exp = oracle_rollout(x, h, a, JAX_STEP, flags, T=T)
            check_both_families(lib, x, h, a, JAX_STEP, flags, exp, (pol, dtype.__name__), T=T)
