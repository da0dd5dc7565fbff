"""Game-tree search of a fixed host (hk_search_depth, hironaka_b200.search_depth) against a level-synchronous search
built from the oracle's C port.

The reference expands every root of a batch level by level: a state with at most one live row has ended; any other
state gets the host's coordinate set S (zeillinger_fn decoded to a bitmask, or every coordinate) and one child per axis
of S in increasing order, the C port's step of the state with bitmask S and that axis (JAX flags).  Before a level is
added it applies the cuts in the library's order: int32 bound (a state to expand with a live entry >= 2^30 / d), node
budget (the root would pass max_nodes), frontier capacity (roots dropped from the highest index down until the level
fits); at level max_depth a state that has not ended stops its root.  depth, nodes and status must be equal.

The tests without the gpu mark hold the reference to hand cases.
"""
import numpy as np
import pytest

from hironaka_b200 import constants as C
from oracle import cport
from tests.test_gpu_record import zeillinger_masks

gpu = pytest.mark.gpu

RESOLVED, MAX_DEPTH, MAX_NODES, CAPACITY, INT32_BOUND = (C.HK_SEARCH_RESOLVED, C.HK_SEARCH_MAX_DEPTH,
                                                         C.HK_SEARCH_MAX_NODES, C.HK_SEARCH_CAPACITY,
                                                         C.HK_SEARCH_INT32_BOUND)


# ---------------------------------------------------------------- reference side (no GPU)


def host_masks(x, host):
    """The host's coordinate set of every state as a bitmask (zeillinger_masks is zeillinger_fn decoded, checked in
    tests/test_gpu_record.py)."""
    B, N, d = x.shape
    if host == "all_coord":
        return np.full(B, (1 << d) - 1, np.int32)
    out = np.empty(B, np.int32)
    for s in range(0, B, 4096):
        out[s:s + 4096] = zeillinger_masks(x[s:s + 4096])
    return out


def popcount(m):
    m = np.asarray(m, np.int64)
    return sum(((m >> k) & 1) for k in range(31)).astype(np.int64)


def reference_search(roots, host="zeillinger", reposition=True, max_depth=64, max_nodes=1 << 16, capacity=1 << 40):
    """(depth int32 [B], nodes int64 [B], status int8 [B]) of the level-synchronous search, from oracle.cport.step."""
    front = np.ascontiguousarray(roots, np.int32)
    B, N, d = front.shape
    ops = C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)
    bound = (1 << 30) // d
    depth = np.zeros(B, np.int32)
    nodes = np.ones(B, np.int64)
    status = np.zeros(B, np.int8)
    froot = np.arange(B)
    for level in range(max_depth + 1):
        live = front[:, :, 0] >= 0
        is_open = live.sum(1) > 1
        if level == max_depth:
            status[np.unique(froot[is_open])] = MAX_DEPTH
            break
        S = host_masks(front, host)
        c = np.where(is_open, popcount(S), 0)
        big = is_open & ((front >= bound) & live[:, :, None]).any((1, 2))
        children = np.bincount(froot, weights=c, minlength=B).astype(np.int64)
        flagged = np.bincount(froot, weights=big, minlength=B) > 0
        keep = np.zeros(B, bool)
        used, full = 0, False
        for r in np.unique(froot):  # increasing root order
            ch = children[r]
            if ch == 0:
                continue
            if flagged[r]:
                status[r] = INT32_BOUND
            elif nodes[r] + ch > max_nodes:
                status[r] = MAX_NODES
            elif full or used + ch > capacity:
                full = True  # dropping from the highest index down: every later root is dropped too
                status[r] = CAPACITY
            else:
                keep[r] = True
                used += ch
                nodes[r] += ch
                depth[r] = level + 1
        parents = np.nonzero(keep[froot] & (c > 0))[0]
        if len(parents) == 0:
            break
        idx = np.repeat(parents, c[parents])
        axes = np.concatenate([[a for a in range(d) if S[i] >> a & 1] for i in parents]).astype(np.int32)
        front = cport.step(np.ascontiguousarray(front[idx]), S[idx], axes, ops, 0)[0]
        froot = froot[idx]
    return depth, nodes, status


def filtered_roots(rng, B, N, d, max_value):
    """randint(0, max_value] roots after the Newton filter and reposition (generate_pts)."""
    x = rng.integers(0, max_value + 1, size=(B, N, d)).astype(np.int32)
    return cport.step(x, None, None, C.HK_OP_NEWTON | C.HK_OP_REPOSITION, 0)[0]


def test_reference_hand_cases():
    two = np.array([[[1, 0], [0, 1]]], np.int32)  # either reply leaves one point: both children end
    for host in ("zeillinger", "all_coord"):
        assert [a.tolist() for a in reference_search(two, host)] == [[1], [3], [RESOLVED]]
    ended = np.array([[[2, 3], [-1, -1]], [[-1, -1], [-1, -1]]], np.int32)
    assert [a.tolist() for a in reference_search(ended)] == [[0, 0], [1, 1], [RESOLVED, RESOLVED]]
    roots = filtered_roots(np.random.default_rng(3), 64, 5, 3, 10)
    full = reference_search(roots, max_depth=32)
    deep = np.nonzero(full[0] >= 2)[0]
    assert len(deep) > 0
    d1, n1, s1 = reference_search(roots, max_depth=1)
    assert (s1[deep] == MAX_DEPTH).all() and (d1[deep] == 1).all()
    assert ((s1 == MAX_DEPTH) == (full[0] >= 2)).all()
    assert (n1 == np.where(full[0] == 0, 1, 1 + popcount(host_masks(roots, "zeillinger")))).all()


def test_reference_budget_capacity_and_bound():
    roots = filtered_roots(np.random.default_rng(4), 16, 5, 3, 10)
    full = reference_search(roots, max_depth=32)
    d2, n2, s2 = reference_search(roots, max_depth=32, max_nodes=3)
    assert (n2 <= 3).all() and ((s2 == MAX_NODES) == (full[1] > 3)).all()
    first = popcount(host_masks(roots, "zeillinger")) * ((roots[:, :, 0] >= 0).sum(1) > 1)
    cap = int(first.sum() // 2)
    d3, n3, s3 = reference_search(roots, max_depth=32, capacity=cap)
    at_root = np.nonzero((s3 == CAPACITY) & (d3 == 0))[0]  # dropped before their first level
    assert len(at_root) > 0 and (n3[at_root] == 1).all()
    assert set(at_root) == {r for r in np.nonzero(first > 0)[0] if first[:r + 1].sum() > cap}
    bound = (1 << 30) // 3
    at = np.array([[[bound, 0, 0], [0, 1, 0], [-1, -1, -1], [-1, -1, -1], [-1, -1, -1]]], np.int32)
    assert [a.tolist() for a in reference_search(at)] == [[0], [1], [INT32_BOUND]]


# ---------------------------------------------------------------- the GPU


@pytest.fixture(scope="module")
def lib():
    import torch
    from hironaka_b200 import ops
    from hironaka_b200._lib import lib as _lib
    assert torch.cuda.is_available()
    ops.force_generic(False)
    yield _lib()
    ops.force_generic(False)


def gpu_search(roots, host="zeillinger", reposition=True, max_depth=64, max_nodes=1 << 16, capacity=None):
    import torch
    import hironaka_b200 as hb
    r = hb.search_depth(torch.as_tensor(np.ascontiguousarray(roots)).cuda(), host, reposition=reposition,
                        max_depth=max_depth, max_nodes=max_nodes, capacity=capacity)
    assert r.depth.dtype == torch.int32 and r.nodes.dtype == torch.int64 and r.status.dtype == torch.int8
    return r.depth.cpu().numpy(), r.nodes.cpu().numpy(), r.status.cpu().numpy()


def assert_same(got, exp, what):
    for name, g, e in zip(("depth", "nodes", "status"), got, exp):
        assert np.array_equal(g, e), (what, name, np.nonzero(g != e)[0][:8], g[g != e][:8], e[g != e][:8])


# (N, d), max value of the roots: trees of a few hundred to a few thousand states per root
SHAPES = [((5, 3), 10), ((10, 3), 8), ((20, 3), 5), ((7, 2), 12), ((6, 4), 5), ((16, 4), 3)]


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[0])))
@pytest.mark.parametrize("host", ["zeillinger", "all_coord"])
@pytest.mark.parametrize("reposition", [True, False], ids=["repos", "norepos"])
@pytest.mark.parametrize("B", [1, 33])
def test_search_matches_reference(lib, shape, host, reposition, B):
    (N, d), max_value = shape
    rng = np.random.default_rng(N * 100 + d * 10 + B)
    roots = filtered_roots(rng, B, N, d, max_value)
    args = dict(host=host, reposition=reposition, max_depth=24, max_nodes=3000)
    got = gpu_search(roots, **args)
    assert_same(got, reference_search(roots, **args), (shape, host, reposition, B))


@gpu
def test_search_warp_per_game_family(lib):
    """(10, 3) runs thread-per-game by default: the same search with the warp-per-game step everywhere."""
    from hironaka_b200 import ops
    roots = filtered_roots(np.random.default_rng(11), 97, 10, 3, 8)
    exp = reference_search(roots, max_depth=24, max_nodes=3000)
    ops.force_generic(True)
    try:
        got = gpu_search(roots, max_depth=24, max_nodes=3000)
    finally:
        ops.force_generic(False)
    assert_same(got, exp, "force_generic")
    assert_same(gpu_search(roots, max_depth=24, max_nodes=3000), exp, "default family")


@gpu
def test_search_large_shape(lib):
    roots = filtered_roots(np.random.default_rng(12), 8, 64, 5, 3)
    for host in ("zeillinger", "all_coord"):
        args = dict(host=host, max_depth=12, max_nodes=600)
        assert_same(gpu_search(roots, **args), reference_search(roots, **args), host)


@gpu
def test_search_statuses(lib):
    """Each cut provoked on purpose, and the results equal to the reference's."""
    rng = np.random.default_rng(13)
    roots = filtered_roots(rng, 65, 10, 3, 10)
    for max_depth in (1, 2, 3):
        got = gpu_search(roots, max_depth=max_depth)
        assert (got[2] == MAX_DEPTH).any()
        assert_same(got, reference_search(roots, max_depth=max_depth), ("max_depth", max_depth))
    for max_nodes in (1, 3, 20):
        got = gpu_search(roots, max_nodes=max_nodes, max_depth=40)
        assert (got[2] == MAX_NODES).any() and (got[1] <= max_nodes).all()
        assert_same(got, reference_search(roots, max_nodes=max_nodes, max_depth=40), ("max_nodes", max_nodes))
    first = popcount(host_masks(roots, "zeillinger")) * ((roots[:, :, 0] >= 0).sum(1) > 1)
    for capacity in (1, int(first.sum()) // 2, int(first.sum()), 500):
        got = gpu_search(roots, capacity=capacity, max_depth=30, max_nodes=2000)
        assert_same(got, reference_search(roots, capacity=capacity, max_depth=30, max_nodes=2000), ("capacity", capacity))
        # dropped before their first level: the roots whose first level no longer fits, from the highest index down
        at_root = set(np.nonzero((got[2] == CAPACITY) & (got[0] == 0))[0])
        assert at_root == {r for r in np.nonzero(first > 0)[0] if first[:r + 1].sum() > capacity}
        assert (capacity >= first.sum()) != bool(at_root)


@gpu
@pytest.mark.parametrize("d", [2, 3, 4])
def test_search_int32_bound(lib, d):
    """Roots whose live entries sit just below and at floor(2^30 / d): below, the root is expanded (its children may
    cross and be cut at the next level); at, the root is cut before its first level."""
    N = 6
    bound = (1 << 30) // d
    rng = np.random.default_rng(14 + d)
    roots = filtered_roots(rng, 40, N, d, 6)
    for b, v in enumerate([bound - 1, bound, bound - 1, bound, bound - 2, bound]):
        x = np.full((N, d), -1, np.int32)
        x[0] = 0
        x[0, 0] = v
        x[1] = 0
        x[1, 1] = 1 + b % 2
        x[2] = 0
        x[2, d - 1] += 3
        roots[5 * b] = cport.step(x[None], None, None, C.HK_OP_NEWTON | C.HK_OP_REPOSITION, 0)[0][0]
    for host in ("zeillinger", "all_coord"):
        args = dict(host=host, max_depth=20, max_nodes=2000)
        got = gpu_search(roots, **args)
        assert_same(got, reference_search(roots, **args), (d, host))
        assert (got[2] == INT32_BOUND).any()
        assert (got[2][[5, 15, 25]] == INT32_BOUND).all() and (got[0][[5, 15, 25]] == 0).all()


@gpu
def test_search_deterministic_and_permutation(lib):
    rng = np.random.default_rng(15)
    roots = filtered_roots(rng, 200, 10, 3, 10)
    args = dict(max_depth=30, max_nodes=5000, capacity=1 << 20)
    a = gpu_search(roots, **args)
    b = gpu_search(roots, **args)
    assert_same(a, b, "repeat")
    perm = rng.permutation(len(roots))
    c = gpu_search(roots[perm], **args)
    assert_same(c, tuple(x[perm] for x in a), "permuted")
    assert (a[2] != CAPACITY).all()


@gpu
def test_search_rejects_arguments(lib):
    import torch
    from hironaka_b200 import ops
    roots = torch.as_tensor(filtered_roots(np.random.default_rng(16), 4, 5, 3, 10)).cuda()
    B, N, d = roots.shape
    ws = torch.empty(ops.search_workspace_bytes(B, N, d, 64), dtype=torch.uint8, device="cuda")
    depth = torch.empty(B, dtype=torch.int32, device="cuda")
    nodes = torch.empty(B, dtype=torch.int64, device="cuda")
    status = torch.empty(B, dtype=torch.int8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    base = dict(x=roots, dtype=C.HK_DTYPE_I32, ops=C.HK_OP_SHIFT | C.HK_OP_NEWTON | C.HK_OP_REPOSITION,
                flags=C.HK_F_HOST_ZEILLINGER, max_depth=8, max_nodes=100, capacity=64)

    def call(**kw):
        a = dict(base, **kw)
        return lib.hk_search_depth(a["x"].data_ptr(), depth.data_ptr(), nodes.data_ptr(), status.data_ptr(), B, N, d,
                                   a["dtype"], a["ops"], a["flags"], a["max_depth"], a["max_nodes"], a["capacity"],
                                   ws.data_ptr(), stream)
    assert call() == C.HK_OK
    assert call(x=roots.float(), dtype=C.HK_DTYPE_F32) == C.HK_ERR_UNSUPPORTED
    for flags in (0, C.HK_F_HOST_ZEILLINGER | C.HK_F_HOST_ALL_COORD, C.HK_F_HOST_RANDOM,
                  C.HK_F_HOST_ZEILLINGER | C.HK_F_AGENT_FIRST, C.HK_F_HOST_ALL_COORD | C.HK_F_AGENT_RANDOM,
                  C.HK_F_HOST_ZEILLINGER | C.HK_F_NOOP_INVALID, C.HK_F_AGENT_LAST):
        assert call(flags=flags) == C.HK_ERR_BAD_ARG, flags
    for op in (C.HK_OP_SHIFT, C.HK_OP_NEWTON, C.HK_OP_SHIFT | C.HK_OP_REPOSITION,
               C.HK_OP_SHIFT | C.HK_OP_NEWTON | C.HK_OP_RESCALE, C.HK_OP_SHIFT | C.HK_OP_NEWTON | C.HK_OP_DEDUPE):
        assert call(ops=op) == C.HK_ERR_BAD_ARG, op
    assert call(max_depth=0) == C.HK_ERR_BAD_ARG
    assert call(max_nodes=0) == C.HK_ERR_BAD_ARG
    assert call(capacity=0) == C.HK_ERR_BAD_ARG
    assert call() == C.HK_OK
    with pytest.raises(ValueError):
        import hironaka_b200 as hb
        hb.search_depth(roots, "random")


@gpu
@pytest.mark.parametrize("host", ["zeillinger", "all_coord"])
def test_rollouts_never_outlast_the_search(lib, host):
    """Independent parts of the library agree: a GameBatch rollout against the same fixed host, with the choose_first,
    choose_last or random agent, never lasts longer than the searched depth of a resolved root.  (The random agent
    draws from every axis, so it stays inside the searched tree only against the all-coordinates host.)"""
    import torch
    from hironaka_b200 import GameBatch
    import hironaka_b200 as hb
    N, d, max_depth = 10, 3, 40
    pts = torch.as_tensor(np.random.default_rng(17).integers(0, 11, size=(257, N, d)).astype(np.int32)).cuda()
    roots = GameBatch(pts, semantics="jax", reposition=True, initial_filter=True).points
    res = hb.search_depth(roots, host, max_depth=max_depth)
    resolved = res.status == hb.STATUS_RESOLVED
    assert int(resolved.sum()) > 0
    agents = ["choose_first", "choose_last"] + (["random"] if host == "all_coord" else [])
    for agent in agents:
        gb = GameBatch(roots.clone(), semantics="jax", reposition=True, host_policy=host, agent_policy=agent, seed=5)
        _, _, _, length = gb.rollout(None, None, want_length=True, steps=max_depth)
        assert bool((length[resolved] <= res.depth[resolved]).all()), agent
        assert bool((length[resolved] > 0).eq(res.depth[resolved] > 0).all()), agent
