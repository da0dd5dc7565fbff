"""Float32 state at its edges, against the oracles (oracle/hk_oracle.py and the C port, oracle/hk_oracle.c).

The parity suites put small integers into float32 state.  Rescaled states (TensorPoints, FusedGame with
scale_observation, the gym hosts with Zeillinger's host) hold arbitrary floats in [0, 1], and the kernels have code that
only such values reach:
  * Zeillinger's host tests jnp.isclose(max, min): |max - min| <= 1e-8 + 1e-5 |min| in float32, the product and the sum
    each rounded.  An FMA rounds once; states whose |max - min| lies between the two results tell them apart.
  * -0.0: the reference treats it as 0 (a row whose coordinate 0 is -0.0 is live, a -0.0 / +0.0 pair is a duplicate);
    the kernels read liveness and dominance from sign bits and canonicalise -0.0 to +0.0 when they load a game.
  * The division by a game's maximum takes a reciprocal fast path when the maximum, the smallest positive entry and
    the maximum's significand are away from the ends of the float range; the choice is made once per warp.
  * Large (above 2^24) and fractional values, rows one ulp apart, and the borders of the packed sort keys of the
    features (2^(27/D) for the sorting network, 2^19 for the rolled sort).
The first half of the file runs without a GPU and checks that the constructed inputs really sit on their borders, so
that an edit to a generator cannot quietly turn these tests into ordinary ones.

inf and NaN are out of scope: a game's state is finite (the reference never produces either from a finite state).
"""
import os
from fractions import Fraction

import numpy as np
import pytest

from oracle import cport
from oracle import hk_oracle as O

f32 = np.float32
ATOL, RTOL = f32(1e-8), f32(1e-5)  # jnp.isclose's defaults, as float32
F_ZEIL, F_FIRST, F_LAST = 1 << 9, 1 << 10, 1 << 11
F_STORE_ALL = 1 << 13
TORCH_FLAGS = O.F_NOOP_INVALID | O.F_FREEZE_ENDED
JAX_STEP = O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON
FUSED_STEP = O.OP_SHIFT | O.OP_NEWTON
F_OBS_SORT_LEX_FIRST = 1 << 12
OBS_FLAGS = [0, O.F_OBS_SORT_COORD0, O.F_OBS_SORT_LEX, F_OBS_SORT_LEX_FIRST]
gpu = pytest.mark.gpu


def exact(v):
    return Fraction(float(v))


def rn32(v: Fraction) -> np.float32:
    """v rounded to the nearest float32, ties to even."""
    x = f32(float(v))
    cands = [np.nextafter(x, f32(-np.inf)), x, np.nextafter(x, f32(np.inf))]
    return min(cands, key=lambda t: (abs(exact(t) - v), int(np.array(t).view(np.uint32)) & 1))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ---------------------------------------------------------------- Zeillinger's closeness border


def isclose_bound(mn, fused):
    """1e-8 + 1e-5 |mn| in float32: the product and the sum rounded (the reference), or rounded once (an FMA)."""
    if fused:
        return rn32(exact(RTOL) * exact(abs(mn)) + exact(ATOL))
    return f32(ATOL + f32(RTOL * f32(abs(mn))))


def zeil_masks(x, fused=False):
    """zeillinger_fn (hironaka/jax/players.py:55-105) as coordinate bitmasks, with isclose_bound's two readings."""
    out = []
    for p in np.asarray(x, f32):
        N, d = p.shape
        diff = p[:, None, :] - p[None, :, :]
        mx, mn = diff.max(2), diff.min(2)
        if fused:
            bound = np.array([[isclose_bound(v, True) for v in row] for row in mn], f32)
        else:
            bound = ATOL + RTOL * np.abs(mn)
        ok = (p >= 0).all(1)
        adm = ok[:, None] & ok[None, :] & ~(np.abs(mx - mn) <= bound)
        cmax, cmin = (diff == mx[..., None]).sum(2), (diff == mn[..., None]).sum(2)
        L = np.where(adm, mx - mn, np.inf).ravel()
        S = np.where(adm, np.where(mx == mn, cmax, cmax + cmin), np.inf).ravel()
        v = diff.reshape(-1, d)[np.lexsort((S, L))[0]]
        amin, amax = int(v.argmin()), int(v.argmax())
        out.append(3 if amin == amax else (1 << amin) | (1 << amax))
    return np.array(out, np.int32)


def zeil_border_pairs(oracle_close):
    """(mn, mx) with 0 < mn < mx and mx - mn exact and equal to the larger of isclose_bound(mn)'s two readings, where
    they differ: the pair is close for the reference and not for an FMA (oracle_close) or the reverse.

    Construction: q = RN(1e-5 mn) is an odd multiple of 2^-51, so that 1e-8 + q (below 2^-26, where float32 steps by
    2^-50) is the midpoint M of two adjacent floats: rounded twice the sum ties and goes to the even neighbour, while
    the exact product, which lies off q, sends the single rounding to the side it lies on."""
    j = np.arange(21, 2001, 2, dtype=np.int64)
    q = j * 2.0 ** -51
    found = []
    for off in (-1, 0, 1):
        mn = ((q / np.float64(RTOL)).astype(f32).view(np.int32) + off).view(f32)
        prod = np.float64(RTOL) * mn.astype(np.float64)  # exact: 24 x 24 bits
        s = np.float64(ATOL) + q  # exact, a midpoint of the float32 grid
        two = s.astype(f32)  # ties to even
        other = np.where(two.astype(np.float64) > s, np.nextafter(two, f32(0)), np.nextafter(two, f32(1)))
        fused = np.where((prod > q) == (other > two), other, two)
        L = np.maximum(two, fused)
        mx = (mn.astype(np.float64) + L.astype(np.float64)).astype(f32)
        keep = ((prod.astype(f32).astype(np.float64) == q) & (prod != q) & (two != fused) & ((two > fused) == oracle_close)
                & (mx.astype(np.float64) - mn.astype(np.float64) == L.astype(np.float64)))
        found += [(mn[k], mx[k]) for k in np.nonzero(keep)[0]]
    found.sort()
    return found


def zeil_border_games(N, d, seed):
    """Games whose Zeillinger choice hangs on one ordered pair of rows (i, j): row i - row j = (mn .. mx), a pair at
    the closeness border.  Both directions, i before and after j, other live rows and dead rows around them.  The
    pair's coordinates {argmin, argmax} differ from {0, 1}, the set the game falls back to without it."""
    rng = np.random.default_rng(seed)
    games = []
    for oracle_close in (True, False):
        pairs = zeil_border_pairs(oracle_close)
        picks = [pairs[k] for k in np.linspace(0, len(pairs) - 1, 4).astype(int)]
        for mn, mx in picks:
            for i_first in (True, False):
                for _ in range(20):  # redraw the other rows until the pair decides the mask (d >= 3)
                    g = one_border_game(rng, N, d, mn, mx, i_first)
                    if d == 2 or zeil_masks(g[None])[0] != zeil_masks(g[None], fused=True)[0]:
                        break
                games.append(g)
    return np.stack(games)


def one_border_game(rng, N, d, mn, mx, i_first):
    diff = np.empty(d, f32)
    if d == 2:
        amin, amax = (1, 0) if rng.random() < 0.5 else (0, 1)
    else:
        amin, amax = rng.choice(np.arange(1, d), 2, replace=False) if rng.random() < 0.5 else (0, d - 1)
        if {amin, amax} == {0, 1}:
            amin, amax = 1, d - 1
    mid = [c for c in range(d) if c not in (amin, amax)]
    diff[amin], diff[amax] = mn, mx
    inner = np.linspace(float(mn), float(mx), len(mid) + 2)[1:-1].astype(f32)  # strictly inside, distinct
    diff[mid] = inner
    x = np.full((N, d), -1.0, f32)
    slots = rng.choice(N, 2, replace=False)
    si, sj = (min(slots), max(slots)) if i_first else (max(slots), min(slots))
    x[sj] = 0.0
    x[si] = diff
    others = [k for k in range(N) if k not in (si, sj)]
    for k in rng.permutation(others)[:min(len(others), 3)]:
        x[k] = rng.integers(1, 7, d)  # far from the pair: integer differences, L >= 1 or a constant vector
    assert np.array_equal(x[si] - x[sj], diff)
    return x


def test_zeillinger_border_pairs_sit_on_the_border():
    for oracle_close in (True, False):
        pairs = zeil_border_pairs(oracle_close)
        assert len(pairs) >= 4, oracle_close
        for mn, mx in pairs:
            two, one = isclose_bound(mn, False), isclose_bound(mn, True)
            assert two != one and (two > one) == oracle_close
            assert exact(mx) - exact(mn) == exact(max(two, one)) == exact(f32(mx - mn))
            p = exact(RTOL) * exact(mn)
            assert rn32(p) != p and 2 * (exact(ATOL) + exact(rn32(p))) == exact(two) + exact(one)  # the sum ties


@pytest.mark.parametrize("d", [2, 3, 4, 5, 6])
def test_zeillinger_border_games_split_the_oracles_from_an_fma(d):
    """The NumPy oracle, the C port and the restatement here agree on every border game; the same host with the bound
    rounded once picks another coordinate set on every one of them (d >= 3: with d = 2 there is one set only)."""
    for N in (5, 12):
        x = zeil_border_games(N, d, seed=N * 10 + d)
        masks = zeil_masks(x)
        assert np.array_equal(masks, zeil_masks_numpy_oracle(x))
        for agent in (F_FIRST, F_LAST):
            c, n = zeil_shift_cport(x, agent)
            assert np.array_equal(bits(c), bits(n)), (N, d, agent)
        if d >= 3:
            fused = zeil_masks(x, fused=True)
            assert (fused != masks).all(), (N, d, np.nonzero(fused == masks))


def zeil_masks_numpy_oracle(x):
    ids = O.zeillinger_fn(x).argmax(1)
    return (O.decode_table(x.shape[2])[ids] << np.arange(x.shape[2])).sum(1).astype(np.int32)


def zeil_shift_cport(x, agent):
    """A shift by Zeillinger's host and a fixed agent in the C port, and the same shift by the NumPy oracle's
    restatement from zeil_masks' sets: equal states mean equal sets (the pair's coordinates are distinct floats, so
    every set gives its own sums)."""
    masks = zeil_masks(x)
    sel = (masks[:, None] >> np.arange(x.shape[2])) & 1
    axis = sel.argmax(1) if agent == F_FIRST else x.shape[2] - 1 - sel[:, ::-1].argmax(1)
    return cport.step(x, None, None, O.OP_SHIFT, F_ZEIL | agent)[0], O.step(x, masks, axis, O.OP_SHIFT, 0)[0]


# ---------------------------------------------------------------- -0.0


def negzero_state(rng, B, N, d):
    """Small-integer games with many zeros, dead rows and duplicates, some zeros written as -0.0: -0.0 in coordinate 0
    of live rows, -0.0 / +0.0 twins in both slot orders, a -0.0 where a +0.0 row would dominate, and games made
    entirely of rows that hold -0.0."""
    x = rng.integers(0, 3, size=(B, N, d)).astype(f32)
    x[rng.random((B, N)) < 0.2] = -1.0
    for b in range(B):
        if N >= 2:
            i, j = rng.choice(N, 2, replace=False)
            x[b, i] = rng.integers(0, 3, d)
            x[b, j] = x[b, i]
            x[b, j, rng.integers(0, d)] = 0.0
            x[b, i, :] = x[b, j]
            (x[b, i] if b % 2 else x[b, j])[x[b, i] == 0] = -0.0  # twins, -0.0 in the lower or the higher slot
    neg = (x == 0) & (rng.random(x.shape) < 0.5)
    x[neg] = -0.0
    x[::5][x[::5] == 0] = -0.0  # games whose zeros are all -0.0
    x[2::5, :, 0] = np.where(x[2::5, :, 0] >= 0, -0.0, x[2::5, :, 0])  # every live row starts with -0.0
    assert (np.signbit(x) & (x == 0)).any()
    return x


def test_negzero_states_hold_negative_zeros():
    rng = np.random.default_rng(1)
    x = negzero_state(rng, 40, 6, 3)
    z = np.signbit(x) & (x == 0)
    assert z[:, :, 0].any() and z[::5].sum() == (x[::5] == 0).sum()
    # -0.0 is live and a twin of +0.0 for both oracles
    assert np.array_equal(O.get_num_points(x), (np.where(x[:, :, 0] == 0, 0, x[:, :, 0]) >= 0).sum(1))
    for ops_bits in (O.OP_NEWTON, O.OP_DEDUPE, JAX_STEP):
        assert np.array_equal(cport.step(x, np.full(40, 7), np.zeros(40), ops_bits, 0)[0],
                              O.step(x, np.full(40, 7), np.zeros(40), ops_bits, 0)[0])


# ---------------------------------------------------------------- the divider's fast-path border


def divider_games(N, d):
    """Games whose maximum b and smallest positive entry m sit at, and one ulp either side of, each condition of the
    fast path: b = 1e-30 and 1e30, m / b at 1e-30 (m = RN(b 1e-30)), significands of all ones, subnormal entries
    and entries near FLT_MAX.  Each returned game is tagged with the side of the conditions it is on."""
    up = lambda v: np.nextafter(f32(v), f32(np.inf))
    dn = lambda v: np.nextafter(f32(v), f32(0))
    cases = []
    for b0 in (f32(1e-30), f32(1e30)):
        for b in (dn(b0), b0, up(b0)):
            cases.append((b, b))
    for b in (f32(1.0), f32(3.0), f32(1e20)):
        m0 = f32(b * f32(1e-30))
        for m in (dn(m0), m0, up(m0)):
            cases.append((b, m))
    for b in (f32(16777215.0), f32(0.99999994), np.uint32(0x3fffffff).view(f32), np.uint32(0x7effffff).view(f32)):
        cases += [(b, b), (dn(b), dn(b)), (up(b), up(b))]
    for b in (f32(1.0), f32(5e-30)):
        cases.append((b, np.uint32(1).view(f32)))  # the smallest subnormal
        cases.append((b, np.uint32(0x007fffff).view(f32)))  # the largest subnormal
    fmax = np.finfo(f32).max
    cases += [(fmax, fmax), (fmax, f32(1.0)), (dn(fmax), f32(3e-8))]
    rng = np.random.default_rng(N * d)
    games = []
    for b, m in cases:
        x = np.full((N, d), -1.0, f32)
        live = max(2, N // 2)
        vals = np.clip(np.exp(rng.uniform(np.log(float(m)), np.log(float(b)), (live, d))), float(m), float(b)).astype(f32)
        vals[rng.random((live, d)) < 0.2] = 0.0
        vals[0, 0], vals[1, rng.integers(0, d)] = b, m
        x[rng.permutation(N)[:live]] = vals
        games.append(x)
    return np.stack(games)


def divider_safe(x):
    """make_divider's `safe`, from a game's maximum b and smallest positive live entry (in float32)."""
    live = x[:, :, 0] >= 0
    v = np.where(live[..., None], x, f32(-1))
    b = v.max((1, 2))
    pos = np.where(v > 0, v, f32(np.inf)).min((1, 2))
    sig_ones = (b.view(np.uint32) & 0x7fffff) == 0x7fffff
    return (b > f32(1e-30)) & (b < f32(1e30)) & (pos > f32(1e-30)) & (pos > b * f32(1e-30)) & ~sig_ones


def test_divider_games_straddle_every_condition():
    x = divider_games(5, 3)
    live = x[:, :, 0] >= 0
    v = np.where(live[..., None], x, f32(-1))
    b = v.max((1, 2))
    pos = np.where(v > 0, v, f32(np.inf)).min((1, 2))
    for edge in (f32(1e-30), f32(1e30)):
        assert (b == edge).any() and (b == np.nextafter(edge, f32(0))).any() and (b == np.nextafter(edge, f32(np.inf))).any()
    ratio = pos - b * f32(1e-30)
    assert (ratio < 0).any() and (ratio == 0).any() and (ratio > 0).any()
    # below b = 1e-8 the product b * 1e-30 leaves the normal range: a subnormal smallest entry passes the ratio test
    # and must still be turned away by its own bound
    tiny = (b * f32(1e-30) < np.finfo(f32).tiny) & (pos < np.finfo(f32).tiny) & (pos > b * f32(1e-30))
    assert tiny.any() and not divider_safe(x)[tiny].any()
    assert ((b.view(np.uint32) & 0x7fffff) == 0x7fffff).any()
    assert (pos < np.finfo(f32).tiny).any() and (b == np.finfo(f32).max).any()
    safe = divider_safe(x)
    assert safe.any() and (~safe).any()
    # the oracles agree with the correctly rounded quotient on every game
    exp = rescale_exact(x)
    assert np.array_equal(bits(cport.rescale(x)), bits(exp))
    assert np.array_equal(bits(O.rescale_torch(x)), bits(exp))


def rescale_exact(x, eps=False, pad=-1.0):
    """live entries / game maximum, correctly rounded (the float64 quotient of two floats rounds to float32 exactly:
    53 >= 2 * 24 + 2); a maximum of 0 (or <= 1e-8 with eps) divides by 1."""
    live = x[:, :, 0] >= 0
    b = x.max((1, 2))
    b = np.where((b == 0) | (eps & (b <= f32(1e-8))), f32(1), b)
    with np.errstate(over="ignore"):  # dead rows may overflow; they are padded below
        q = (x.astype(np.float64) / b.astype(np.float64)[:, None, None]).astype(f32)
    return np.where(live[..., None], q, f32(pad))


def divider_warps(N, d):
    """Warps of 32 games: border games that are all safe (the fast path), and the same games mixed with unsafe ones
    (the vote sends every lane down the slow path)."""
    x = divider_games(N, d)
    safe = divider_safe(x)
    s, u = x[safe], x[~safe]
    reps = lambda a, n: a[np.arange(n) % len(a)]
    all_safe = reps(s, 32)
    mixed = reps(s, 32).copy()
    mixed[5::7] = reps(u, len(mixed[5::7]))
    return np.concatenate([all_safe, mixed, reps(u, 32), x])


def below_parking(x):
    """The games whose entries are all below 3e38: the dominance filter parks dead rows there (DESIGN section 3), so
    a live row with every coordinate at or above it is not a state the filter takes."""
    return x[x.max((1, 2)) < f32(3e38)]


def eps_games(N, d):
    """HK_F_RESCALE_EPS: games whose maximum is 1e-8 and its two neighbours."""
    e = f32(1e-8)
    out = []
    for b in (np.nextafter(e, f32(0)), e, np.nextafter(e, f32(1))):
        x = np.full((N, d), -1.0, f32)
        x[0] = b
        x[1] = f32(b / 3)
        x[1, 0] = 0.0
        out.append(x)
    return np.stack(out)


def test_eps_games_straddle_the_cutoff():
    x = eps_games(5, 3)
    m = x.max((1, 2))
    assert (m < f32(1e-8)).sum() == 1 and (m == f32(1e-8)).sum() == 1 and (m > f32(1e-8)).sum() == 1
    exp = rescale_exact(x, eps=True)
    assert np.array_equal(bits(cport.step(x, None, None, O.OP_RESCALE, O.F_RESCALE_EPS)[0]), bits(exp))
    assert np.array_equal(bits(O.rescale_jax(x)), bits(exp))
    assert not np.array_equal(exp[2], x[2]) and np.array_equal(exp[1], x[1])


# ---------------------------------------------------------------- magnitudes


def magnitude_state(rng, B, N, d, kind):
    """'big': integers in [2^24, 2^26] (float32 steps by 2 and 4 there); 'frac': fractions of mixed scale; 'ulp':
    rows one ulp apart in one coordinate."""
    if kind == "big":
        x = rng.integers(2 ** 24, 2 ** 26, size=(B, N, d)).astype(f32)
    elif kind == "frac":
        x = (rng.random((B, N, d)) * 10.0 ** rng.integers(-3, 4, size=(B, 1, 1))).astype(f32)
    else:
        x = (rng.random((B, N, d)) + 0.5).astype(f32)
        for b in range(B):
            i, j = rng.choice(N, 2, replace=False)
            x[b, j] = x[b, i]
            c = rng.integers(0, d)
            x[b, j, c] = np.nextafter(x[b, i, c], f32(np.inf) if rng.random() < 0.5 else f32(0))
    x[rng.random((B, N)) < 0.25] = -1.0
    return x


def test_magnitude_states_need_float_rounding():
    rng = np.random.default_rng(3)
    x = magnitude_state(rng, 50, 8, 6, "big")
    live = x[:, :, 0] >= 0
    s = np.zeros(x.shape[:2], np.float64)
    s32 = np.zeros(x.shape[:2], f32)
    for c in range(6):
        s += x[:, :, c]
        s32 = s32 + x[:, :, c]
    assert ((s32.astype(np.float64) != s) & live).any()  # the sum rounds, so its order matters
    y = magnitude_state(rng, 50, 8, 3, "ulp")
    live = y[:, :, 0] >= 0
    steps = np.abs(y[:, :, None].view(np.int32).astype(np.int64) - y[:, None].view(np.int32))
    one_ulp = (steps.max(3) == 1) & live[:, :, None] & live[:, None]
    assert one_ulp.any(2).any(1).mean() > 0.5  # most games hold two live rows one ulp apart


# ================================================================ GPU


@pytest.fixture(scope="module")
def hb():
    import hironaka_b200
    from hironaka_b200 import ops
    assert os.path.exists(hironaka_b200.LIB_PATH), "CUDA library not built"
    ops.force_generic(False)
    return hironaka_b200


@pytest.fixture(params=[False, True], ids=["family=auto", "family=generic"])
def family(request, hb):
    from hironaka_b200 import ops
    ops.force_generic(request.param)
    yield request.param
    ops.force_generic(False)


def dev(a):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


def gpu_step(x, ha, ax, ops_bits, flags, want_obs=False, pad=-1.0):
    """hk_step out of place, in place and in place with HK_F_STORE_ALL: the three states must agree bit for bit, and
    so must the outputs.  Returns (state, done, reward, num_points, obs)."""
    from hironaka_b200 import ops
    h = None if ha is None else dev(np.asarray(ha, np.int32))
    a = None if ax is None else dev(np.asarray(ax, np.int32))
    res = []
    for inplace, extra in ((False, 0), (True, 0), (True, F_STORE_ALL)):
        g = dev(x)
        r = ops.step(g, h, a, ops=ops_bits, flags=flags | extra, inplace=inplace, padding_value=pad, want_done=True,
                     want_reward=True, want_num_points=True, want_obs=want_obs)
        res.append((host(r.state), host(r.done), host(r.reward), host(r.num_points),
                    None if r.obs is None else host(r.obs)))
    for k, what in ((1, "in place"), (2, "in place, HK_F_STORE_ALL")):
        assert np.array_equal(bits(res[k][0]), bits(res[0][0])), what
        for o in range(1, 5):
            assert (res[k][o] is None) or np.array_equal(res[k][o], res[0][o]), (what, o)
    return res[0]


def assert_step_matches_oracles(x, ha, ax, ops_bits, flags, what):
    got = gpu_step(x, ha, ax, ops_bits, flags)
    exp = cport.step(x, ha, ax, ops_bits, flags)
    assert np.array_equal(got[0], exp[0]), (what, "state")
    assert np.array_equal(got[1], exp[1].astype(bool)) and np.array_equal(got[2], exp[2]), (what, "done / reward")
    assert np.array_equal(got[3], exp[3]), (what, "num_points")
    return got


ZEIL_SHAPES = [(5, 3), (10, 3), (20, 3), (7, 2), (16, 4), (12, 5), (9, 6), (40, 3), (33, 4)]


@gpu
@pytest.mark.parametrize("shape", ZEIL_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_zeillinger_border(hb, family, shape):
    """Zeillinger's host on games at the closeness border: the policy, the step with first / last agents in both
    flavours, the one-launch rollout, the recorded host masks and the threshold rollout all play the reference's
    coordinate set."""
    from hironaka_b200 import ops
    N, d = shape
    x = zeil_border_games(N, d, seed=N * 10 + d)
    B = len(x)
    exp = zeil_masks(x)
    got = host(ops.host_policy(dev(x), "zeillinger"))
    assert np.array_equal(got, exp), f"{int((got != exp).sum())} of {B} games: got {got[got != exp]}, expected {exp[got != exp]}"
    for ops_bits, flavour in ((JAX_STEP, 0), (FUSED_STEP, TORCH_FLAGS)):
        for agent in (F_FIRST, F_LAST):
            flags = F_ZEIL | agent | flavour
            assert_step_matches_oracles(x, None, None, ops_bits, flags, (ops_bits, flags))
            T = 3
            o = x
            for _ in range(T):
                o = cport.step(o, None, None, ops_bits, flags)[0]
            out = ops.rollout(dev(x), None, None, ops=ops_bits, flags=flags, inplace=False, steps=T)[0]
            assert np.array_equal(host(out), o), ("rollout", flags)
            thr = ops.rollout(dev(x), None, None, ops=ops_bits, flags=flags, inplace=False, steps=T,
                              value_threshold=1e30)[0]
            assert np.array_equal(host(thr), o), ("threshold rollout", flags)
            tr = ops.rollout_record(dev(x), T, ops=ops_bits, flags=flags, inplace=False)
            assert np.array_equal(host(tr.host_mask)[0], exp), ("recorded host mask", flags)
            assert np.array_equal(host(tr.state), o), ("recorded rollout", flags)


NEGZERO_SHAPES = [(5, 3), (10, 3), (20, 3), (33, 3), (40, 2), (64, 5), (16, 4), (9, 10)]
NEGZERO_STEPS = [(O.OP_NEWTON, 0), (O.OP_DEDUPE, 0), (O.OP_SHIFT, TORCH_FLAGS), (O.OP_SHIFT, 0), (O.OP_REPOSITION, 0),
                 (O.OP_RESCALE, 0), (O.OP_NEWTON | O.OP_RESCALE, 0), (JAX_STEP, 0), (FUSED_STEP, TORCH_FLAGS)]


@gpu
@pytest.mark.parametrize("shape", NEGZERO_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_negative_zero_steps(hb, shape):
    """-0.0 is 0 to every op; the state a step writes holds no live -0.0 (a game that held one counts as changed, so
    the default write-back equals HK_F_STORE_ALL), and both kernel families write the same bits."""
    from hironaka_b200 import ops
    N, d = shape
    rng = np.random.default_rng(N + d)
    B = 70
    x = negzero_state(rng, B, N, d)
    ha, ax = rng.integers(0, 2 ** d, B), rng.integers(0, d, B)
    for ops_bits, flags in NEGZERO_STEPS:
        by_family = []
        for generic in (False, True):
            ops.force_generic(generic)
            try:
                got = assert_step_matches_oracles(x, ha, ax, ops_bits, flags, (ops_bits, flags, generic))
            finally:
                ops.force_generic(False)
            if N * N * d * B <= 2_000_000:
                ref = O.step(x, ha, ax, ops_bits, flags)
                assert np.array_equal(got[0], ref[0]), (ops_bits, flags, generic, "numpy")
            live = got[0][:, :, 0] >= 0
            assert not (np.signbit(got[0]) & (got[0] == 0) & live[..., None]).any(), (ops_bits, flags, generic)
            by_family.append(got[0])
        assert np.array_equal(bits(by_family[0]), bits(by_family[1])), (ops_bits, flags, "families")


@gpu
@pytest.mark.parametrize("shape", [(5, 3), (10, 3), (20, 3), (33, 3), (16, 4), (40, 2)], ids=lambda s: "x".join(map(str, s)))
def test_negative_zero_reads(hb, family, shape):
    """Features in every sort mode, with and without rescale; dones / num_points; overflow."""
    from hironaka_b200 import ops
    N, d = shape
    rng = np.random.default_rng(3 * N + d)
    x = negzero_state(rng, 64, N, d)
    g = dev(x)
    for sort in OBS_FLAGS:
        for resc in (0, O.F_OBS_RESCALE):
            got = host(ops.features(g, flags=sort | resc))
            assert np.array_equal(got, cport.features(x, sort | resc)), (sort, resc)
    done, npts = ops.dones(g, want_num_points=True)
    assert np.array_equal(host(done), O.get_dones(x)) and np.array_equal(host(npts), O.get_num_points(x))
    live = (x[:, :, 0] >= 0)[..., None]
    for thr, strict in ((0.0, False), (0.0, True), (1.0, False)):
        exp = (((x > thr) if strict else (x >= thr)) & live).any((1, 2))
        assert np.array_equal(host(ops.overflow(g, thr, strict)), exp), (thr, strict)


@gpu
@pytest.mark.parametrize("shape", [(5, 3), (10, 3), (20, 3), (33, 3), (40, 2), (64, 5)], ids=lambda s: "x".join(map(str, s)))
def test_negative_zero_census_and_rollouts(hb, shape):
    """Census steps from a state with -0.0 (the small shapes, and the shapes whose sparse games the rows kernel
    steps), with games rewritten by the caller between steps (census bytes zeroed), and one-launch rollouts."""
    from hironaka_b200 import ops
    N, d = shape
    rng = np.random.default_rng(5 * N + d)
    B, T = 96, 6
    x = negzero_state(rng, B, N, d)
    ha = rng.integers(0, 2 ** d, (T, B)).astype(np.int32)
    ax = rng.integers(0, d, (T, B)).astype(np.int32)
    for ops_bits, flags in ((JAX_STEP, 0), (FUSED_STEP, TORCH_FLAGS)):
        out = ops.rollout(dev(x), dev(ha), dev(ax), ops=ops_bits, flags=flags, inplace=False)[0]
        o = x
        for t in range(T):
            o = cport.step(o, ha[t], ax[t], ops_bits, flags)[0]
        assert np.array_equal(host(out), o), (ops_bits, "rollout")
        g = dev(x)
        census = ops.new_census(g)
        o = x
        for t in range(T):
            r = ops.step(g, dev(ha[t]), dev(ax[t]), ops=ops_bits, flags=flags, census=census, want_done=True,
                         want_reward=True, want_num_points=True)
            o, od, orw, onp = cport.step(o, ha[t], ax[t], ops_bits, flags)
            s = host(g)
            assert np.array_equal(s, o), (ops_bits, t)
            assert not (np.signbit(s) & (s == 0) & (s[:, :, :1] >= 0)).any(), (ops_bits, t)
            assert np.array_equal(host(r.done), od.astype(bool)) and np.array_equal(host(r.num_points), onp), (ops_bits, t)
            assert np.array_equal(host(r.reward), orw), (ops_bits, t)
            if t == 2:  # the caller rewrites some games, -0.0 included, and zeroes their census bytes
                idx = rng.permutation(B)[:B // 6]
                fresh = negzero_state(rng, len(idx), N, d)
                o = o.copy()
                o[idx] = fresh
                g[dev(idx)] = dev(fresh)
                census[dev(idx)] = 0


@gpu
@pytest.mark.parametrize("shape", [(5, 3), (10, 3), (20, 3), (16, 4), (33, 3)], ids=lambda s: "x".join(map(str, s)))
def test_divider_border(hb, family, shape):
    """Rescale of games at each border of the divider's fast path, in warps that are all safe and in warps that mix
    safe and unsafe games: OP_RESCALE, OP_NEWTON | OP_RESCALE, rescaled features, and HK_F_RESCALE_EPS at 1e-8."""
    from hironaka_b200 import ops
    N, d = shape
    x = divider_warps(N, d)
    exp = rescale_exact(x)
    got = gpu_step(x, None, None, O.OP_RESCALE, 0)[0]
    assert np.array_equal(bits(got), bits(exp)), np.nonzero((bits(got) != bits(exp)).any((1, 2)))[0][:8]
    assert np.array_equal(bits(got), bits(cport.step(x, None, None, O.OP_RESCALE, 0)[0]))
    xn = below_parking(x)
    n = cport.step(xn, None, None, O.OP_NEWTON, 0)[0]
    got = gpu_step(xn, None, None, O.OP_NEWTON | O.OP_RESCALE, 0)[0]
    assert np.array_equal(bits(got), bits(rescale_exact(n)))
    for sort in OBS_FLAGS:
        obs = host(ops.features(dev(x), flags=sort | O.F_OBS_RESCALE))
        assert np.array_equal(bits(obs), bits(cport.features(x, sort | O.F_OBS_RESCALE))), sort
        if sort == 0:
            assert np.array_equal(bits(obs), bits(exp.reshape(len(x), -1)))
        o = gpu_step(n, None, None, O.OP_NEWTON, sort | O.F_OBS_RESCALE, want_obs=True)[4]
        assert np.array_equal(bits(o), bits(cport.features(n, sort | O.F_OBS_RESCALE))), ("fused", sort)
    e = np.concatenate([eps_games(N, d)] * 11)
    for ops_bits in (O.OP_RESCALE, O.OP_NEWTON | O.OP_RESCALE):
        got = gpu_step(e, None, None, ops_bits, O.F_RESCALE_EPS)[0]
        assert np.array_equal(bits(got), bits(cport.step(e, None, None, ops_bits, O.F_RESCALE_EPS)[0])), ops_bits
    obs = host(ops.features(dev(e), flags=O.F_OBS_RESCALE | O.F_RESCALE_EPS))
    assert np.array_equal(bits(obs), bits(rescale_exact(e, eps=True).reshape(len(e), -1)))


@gpu
@pytest.mark.parametrize("N", [5, 10, 20])
def test_divider_border_census_observation(hb, N):
    """The census step with the fused rescaled observation on the divider's border games."""
    from hironaka_b200 import ops
    x = below_parking(divider_warps(N, 3))
    g = dev(x)
    census = ops.new_census(g)
    for sort in (O.F_OBS_SORT_COORD0, O.F_OBS_SORT_LEX):
        flags = sort | O.F_OBS_RESCALE
        r = ops.step(g, None, None, ops=O.OP_NEWTON, flags=flags, census=census, want_obs=True)
        exp = cport.step(x, None, None, O.OP_NEWTON, 0)[0]
        assert np.array_equal(host(g), exp)
        assert np.array_equal(bits(host(r.obs)), bits(cport.features(exp, flags))), sort
        x = exp


@gpu
@pytest.mark.parametrize("d", [2, 3, 4, 5, 6, 7, 8, 9, 10])
@pytest.mark.parametrize("kind", ["big", "frac", "ulp"])
def test_magnitudes(hb, family, d, kind):
    """Large, fractional and one-ulp-apart values through the step in both flavours, with shift masks of many bits:
    the shift's float32 sum runs in coordinate order, the dominance test sees one-ulp differences."""
    N = {3: 20}.get(d, 12)
    rng = np.random.default_rng(d * 7 + len(kind))
    B = 64
    x = magnitude_state(rng, B, N, d, kind)
    full = (1 << d) - 1
    ha = np.where(rng.random(B) < 0.6, full, rng.integers(3, 2 ** d, B)).astype(np.int32)
    ha[ha == full] ^= np.where(rng.random((ha == full).sum()) < 0.3, 1, 0).astype(np.int32)
    ax = rng.integers(0, d, B)
    for ops_bits, flags in ((JAX_STEP, 0), (FUSED_STEP, TORCH_FLAGS), (O.OP_NEWTON, 0), (O.OP_SHIFT, 0),
                            (FUSED_STEP | O.OP_RESCALE, TORCH_FLAGS)):
        got = assert_step_matches_oracles(x, ha, ax, ops_bits, flags, (ops_bits, flags))
        if N * N * d * B <= 2_000_000:
            assert np.array_equal(got[0], O.step(x, ha, ax, ops_bits, flags)[0]), (ops_bits, flags, "numpy")


@gpu
@pytest.mark.parametrize("N", [5, 10, 20])
def test_feature_key_borders(hb, family, N):
    """Sorted features of integer and fractional values at the packed-key borders of the thread-per-game family
    (d = 3): 2^9 - 1 and 2^9 for the sorting network's 9-bit fields, 2^19 - 1, 2^19 and 2^19 + 1 for the rolled sort;
    whole warps on one side and warps that mix them."""
    from hironaka_b200 import ops
    rng = np.random.default_rng(N)
    d = 3
    games = []
    for top in (511, 512, 2 ** 19 - 1, 2 ** 19, 2 ** 19 + 1, 511.5, 2 ** 19 - 0.5):
        for _ in range(32):
            x = rng.integers(0, 4, size=(N, d)).astype(f32)
            x[rng.random(N) < 0.3] = -1.0
            x[rng.integers(0, N), rng.integers(0, d)] = top
            x[rng.integers(0, N)] = [top, top - 1, 0]
            games.append(x)
    x = np.stack(games)
    mixed = x[rng.permutation(len(x))]
    for state in (x, mixed):
        for sort in OBS_FLAGS:
            for resc in (0, O.F_OBS_RESCALE):
                got = host(ops.features(dev(state), flags=sort | resc))
                assert np.array_equal(bits(got), bits(cport.features(state, sort | resc))), (sort, resc)
