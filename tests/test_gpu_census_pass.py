"""The census pass of hk_step_census (four games per lane, vector stores for the games at rest, one counting sort)
against the C port after every step of a short rollout: state, census, done, reward, num_points, done_bits and
done_count, with outputs at offsets that rule out the vector stores, census buffers that are not word aligned,
and guard words past every output that must stay untouched.

Small batches give every warp a single tile (one group, lanes 8-31 without games, the one-chunk compaction);
batches of a few hundred thousand games give every warp several tiles — groups of four with a partial last group,
a warp with a shorter run at the end, and rounds sorted by class with more than 32 games in play."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import cport  # noqa: E402
from oracle import hk_oracle as O  # noqa: E402
from tests.test_gpu_parity import TORCH_FLAGS, dev, random_state  # noqa: E402

pytestmark = pytest.mark.gpu

GUARD = 16  # guard elements past each output
JAX = (O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, O.F_ACT_DISCRETE)
# torch flavour: ended games are frozen and nothing moves their lone point, so an ended game rests wherever it is
TORCH = (O.OP_SHIFT | O.OP_NEWTON, TORCH_FLAGS | O.F_ACT_DISCRETE | O.F_ROLE_AGENT)
OFFSETS = {"aligned": (0, 0, 0), "odd": (1, 1, 1), "word_census": (3, 1, 4)}
N, D = 20, 3


def guarded(n, dtype, off, fill):
    """A buffer of n elements starting `off` elements into a fresh allocation, followed by GUARD sentinel elements."""
    buf = torch.full((off + n + GUARD,), fill, dtype=dtype, device="cuda")
    return buf, buf[off:off + n]


def mixed_state(rng, B, dtype):
    """Groups of four games that mix every kind of census byte: empty games, lone points away from the origin and
    at it (ended; at rest or not, by flavour), and games with many rows."""
    x0 = random_state(rng, B, N, D, max_value=6, dead_frac=0.5, dup_frac=0.1)
    x0[::3] = -1
    x0[1::5, 1:] = -1
    x0[1::5, 0] = np.abs(x0[1::5, 0])
    x0[2::7, 1:] = -1
    x0[2::7, 0] = 0
    return x0.astype(dtype)


def sorted_rounds(c, B, frozen_rest, nw):
    """Rounds that take the class sort with more than 32 games in play (census c before the step), for a launch of
    nw warps, each owning a contiguous run of tiles scheduled in rounds of 32 (hk_sched.cuh)."""
    ntiles = (B + 31) // 32
    tpw = (ntiles + nw - 1) // nw
    rest = ((c & 0x80) != 0) & (((c & 2) != 0) | frozen_rest)
    play = np.concatenate([~rest, np.zeros(ntiles * 32 - B, bool)]).reshape(ntiles, 32).sum(1)
    games = np.minimum(B - np.arange(ntiles) * 32, 32)
    n = 0
    for t0 in range(0, ntiles, tpw):
        for r0 in range(t0, min(t0 + tpw, ntiles), 32):
            r1 = min(r0 + 32, t0 + tpw, ntiles)
            ip, ng = play[r0:r1].sum(), games[r0:r1].sum()
            n += int(32 < ip and ip * 2 < ng)
    return n


def rollout(B, offsets, flavour, dtype, T, seed, nw=None):
    """T census steps of B mixed games against the C port; returns the number of steps that had sorted rounds of
    more than 32 games in play (counted when nw, the warps of the launch, is given)."""
    from hironaka_b200 import constants as C
    from hironaka_b200._lib import check, lib
    done_off, out_off, census_off = offsets  # done in bytes, reward / num_points in 4-byte words, census in bytes
    ops_bits, flags = flavour
    frozen_rest = bool(flags & O.F_FREEZE_ENDED) and not (ops_bits & O.OP_REPOSITION)
    rng = np.random.default_rng(seed)
    x0 = mixed_state(rng, B, dtype)
    g = dev(x0)
    nbytes = lib().hk_census_bytes(B, N, D)
    assert nbytes == B
    cbuf, census = guarded(nbytes, torch.uint8, census_off, 0)
    dbuf, done = guarded(B, torch.uint8, done_off, 0xA5)
    rbuf, reward = guarded(B, torch.float32, out_off, 7.5)
    nbuf, npts = guarded(B, torch.int32, out_off, -99)
    nw_bits = (B + 31) // 32
    bbuf, bits = guarded(nw_bits, torch.int32, 0, 0x5A5A5A5A)
    bufs = (cbuf, dbuf, rbuf, nbuf, bbuf)
    outer = [b.clone() for b in bufs]  # the elements in front of each output and the guards after it
    lead = (census_off, done_off, out_off, out_off, 0)
    ncls = 2 ** D - D - 1
    o = x0
    sorted_steps = 0
    for t in range(T):
        if nw is not None:
            sorted_steps += sorted_rounds(census.cpu().numpy(), B, frozen_rest, nw) > 0
        ha = rng.integers(0, ncls, B).astype(np.int32)
        ax = rng.integers(0, D, B).astype(np.int32)
        o, od, orw, onp = cport.step(o, ha, ax, ops_bits, flags)
        dc = torch.zeros(1, dtype=torch.int32, device="cuda")
        ha_d, ax_d = dev(ha), dev(ax)
        # every output the step writes is reset to a sentinel first, so a store that is missing shows
        done.fill_(0xA5)
        reward.fill_(7.5)
        npts.fill_(-99)
        bits.fill_(-1 if t % 2 else 0)
        check(lib().hk_step_census(g.data_ptr(), ha_d.data_ptr(), ax_d.data_ptr(), done.data_ptr(), bits.data_ptr(),
                                   reward.data_ptr(), npts.data_ptr(), census.data_ptr(), dc.data_ptr(), None, B, N, D,
                                   C.HK_DTYPE_F32 if dtype == np.float32 else C.HK_DTYPE_I32, ops_bits, flags, -1.0, 1e8,
                                   torch.cuda.current_stream().cuda_stream))
        assert np.array_equal(g.cpu().numpy(), o), t
        assert np.array_equal(done.cpu().numpy(), od.astype(np.uint8)), t
        assert np.array_equal(reward.cpu().numpy().view(np.int32), orw.view(np.int32)), t
        assert np.array_equal(npts.cpu().numpy(), onp), t
        assert int(dc.item()) == int(od.sum()), t
        want_bits = np.packbits(np.concatenate([od.astype(np.uint8), np.zeros(nw_bits * 32 - B, np.uint8)]),
                                bitorder="little").view(np.uint32)
        assert np.array_equal(bits.cpu().numpy().view(np.uint32), want_bits), t
        c = census.cpu().numpy()
        live = (o[:, :, 0] >= 0).sum(1)
        assert (c != 0).all(), t  # (20, 3): every stepped game gets its byte
        assert np.array_equal(np.where(c & 0x80, c & 1, c), live), t
        assert np.array_equal((c & 0x80) != 0, live <= 1), t
        for b, want, k in zip(bufs, outer, lead):
            assert torch.equal(b[-GUARD:], want[-GUARD:]), t
            assert torch.equal(b[:k], want[:k]), t
        if t == 3:  # the caller rewrites some games and zeroes their census bytes (unknown: read and counted)
            idx = rng.permutation(B)[:max(1, B // 9)]
            fresh = random_state(rng, len(idx), N, D, max_value=6, dead_frac=0.3).astype(dtype)
            o = o.copy()
            o[idx] = fresh
            ti = torch.from_numpy(idx).cuda()
            g[ti] = dev(fresh)
            census[ti] = 0
    return sorted_steps


@pytest.mark.parametrize("B", [1, 31, 33, 127, 128, 129, 4099])
@pytest.mark.parametrize("offsets", list(OFFSETS.values()), ids=list(OFFSETS))
@pytest.mark.parametrize("flavour", [JAX, TORCH], ids=["jax", "torch"])
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
def test_census_pass_outputs(B, offsets, flavour, dtype):
    rollout(B, offsets, flavour, dtype, T=9, seed=B * 7 + offsets[2])


@pytest.mark.parametrize("offsets", [OFFSETS["aligned"], OFFSETS["odd"]], ids=["aligned", "odd"])
@pytest.mark.parametrize("flavour", [JAX, TORCH], ids=["jax", "torch"])
@pytest.mark.parametrize("dtype", [np.int32, np.float32])
def test_census_pass_several_tiles_per_warp(offsets, flavour, dtype):
    """A batch sized so that a warp of the int32 launch (4 CTAs of 4 warps per SM, hk_sched_launch.inl) owns six
    tiles — a whole group and half of a second — and the last warp three, the last tile partial; the float32 launch
    (fewer warps) gives each warp a longer run.  The int32 rollouts must reach rounds sorted by class."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    nw = sms * 16
    B = (nw * 6 - 3) * 32 - 5
    steps = rollout(B, offsets, flavour, dtype, T=8, seed=11 + offsets[0], nw=nw if dtype == np.int32 else None)
    if dtype == np.int32:
        assert steps >= 2, steps
