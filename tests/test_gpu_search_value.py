"""Game value by minimax search (hk_search_value, hironaka_b200.search_value) against a level-synchronous search built
from the oracle's C port.

The reference keeps the whole tree: for every state its parent, the set S of its group, its rank in the group, the
unsolved children of each group and the round in which it was solved.  Level by level it (1) solves the ended states
of the new level and walks up one level at a time: a group whose children are all solved is won, the parent of a won
group is solved in this round, a root's best set is the smallest S won; (2) expands every open state with no solved
ancestor into one child per (S, axis), S over the sets with |S| >= 2 in increasing order, the axes of S in increasing
order, the C port's step with JAX flags; (3) before the level is added, applies the cuts in the library's order:
int32 bound, node budget, frontier capacity, history, the last two from the highest root index down.  value,
best_mask, nodes and status must be equal.

The tests without the gpu mark hold the reference to hand cases.
"""
import numpy as np
import pytest

from hironaka_b200 import constants as C
from oracle import cport
from tests.test_gpu_search import filtered_roots, popcount, reference_search

gpu = pytest.mark.gpu

RESOLVED, MAX_DEPTH, MAX_NODES, CAPACITY, INT32_BOUND, HISTORY = (
    C.HK_SEARCH_RESOLVED, C.HK_SEARCH_MAX_DEPTH, C.HK_SEARCH_MAX_NODES, C.HK_SEARCH_CAPACITY, C.HK_SEARCH_INT32_BOUND,
    C.HK_SEARCH_HISTORY)
BIG = 1 << 40


# ---------------------------------------------------------------- reference side (no GPU)


def child_pairs(d):
    """(S, axis, rank of the axis in S) of every child of an expanded state, in order."""
    out = []
    for S in range(1 << d):
        axes = [a for a in range(d) if S >> a & 1]
        if len(axes) >= 2:
            out += [(S, a, k) for k, a in enumerate(axes)]
    return np.array(out, np.int64)


def reference_value(roots, reposition=True, max_depth=16, max_nodes=1 << 22, capacity=BIG, history=BIG):
    """(value int32 [B], best_mask int32 [B], nodes int64 [B], status int8 [B]), from oracle.cport.step."""
    front = np.ascontiguousarray(roots, np.int32)
    B, N, d = front.shape
    ops = C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)
    bound = (1 << 30) // d
    pairs = child_pairs(d)
    nc = len(pairs)
    # the history: one entry per state of every level, the roots first
    parent = np.full(B, -1, np.int64)
    gset = np.zeros(B, np.int64)
    rank = np.zeros(B, np.int64)
    rem = np.zeros(B, np.int64)
    solved = np.full(B, -1, np.int64)
    value = np.zeros(B, np.int32)
    best = np.full(B, BIG, np.int64)
    nodes = np.ones(B, np.int64)
    status = np.zeros(B, np.int8)
    fh = np.arange(B)     # history entry of each frontier state
    froot = np.arange(B)  # root of each frontier state
    for level in range(max_depth + 1):
        live = front[:, :, 0] >= 0
        ended = live.sum(1) <= 1
        # round `level`: the ended states, then one level up at a time
        new = fh[ended]
        solved[new] = level
        while len(new):
            new = new[parent[new] >= 0]
            heads, k = np.unique(new - rank[new], return_counts=True)
            rem[heads] -= k
            won = heads[rem[heads] == 0]
            par = parent[won]
            at_root = par < B
            np.minimum.at(best, par[at_root], gset[won][at_root])
            par = np.unique(par)
            new = par[solved[par] < 0]
            solved[new] = level
        # open states with no solved ancestor
        pruned = ended.copy()
        a = parent[fh]
        while (a >= 0).any():
            ok = a >= 0
            pruned[ok] |= solved[a[ok]] >= 0
            a = np.where(ok, parent[np.maximum(a, 0)], -1)
        grow = ~pruned
        big = grow & ((front >= bound) & live[:, :, None]).any((1, 2))
        expand = level < max_depth
        children = np.bincount(froot, weights=grow * nc, minlength=B).astype(np.int64) if expand else np.zeros(B, np.int64)
        opened = np.bincount(froot, weights=grow, minlength=B) > 0
        flagged = np.bincount(froot, weights=big, minlength=B) > 0
        keep = np.zeros(B, bool)
        used = 0
        for r in np.unique(froot):  # the roots in play, in increasing order
            value[r] = level
            ch = children[r]
            if solved[r] >= 0:
                continue
            if not expand and opened[r]:
                status[r] = MAX_DEPTH
            elif ch > 0:
                if flagged[r]:
                    status[r] = INT32_BOUND
                elif nodes[r] + ch > max_nodes:
                    status[r] = MAX_NODES
                else:
                    used += ch  # every candidate counts: dropping from the highest index down
                    if used > capacity:
                        status[r] = CAPACITY
                    elif len(parent) + used > history:
                        status[r] = HISTORY
                    else:
                        keep[r] = True
                        nodes[r] += ch
        parents = np.nonzero(keep[froot] & grow)[0] if expand else np.zeros(0, np.int64)
        if len(parents) == 0:
            break
        idx = np.repeat(parents, nc)
        S, A, R = (np.tile(pairs[:, k], len(parents)) for k in range(3))
        h0 = len(parent)
        parent = np.concatenate([parent, fh[idx]])
        gset = np.concatenate([gset, S])
        rank = np.concatenate([rank, R])
        rem = np.concatenate([rem, np.where(R == 0, popcount(S), 0)])
        solved = np.concatenate([solved, np.full(len(idx), -1, np.int64)])
        front = cport.step(np.ascontiguousarray(front[idx]), S.astype(np.int32), A.astype(np.int32), ops, 0)[0]
        froot = froot[idx]
        fh = h0 + np.arange(len(idx))
    best_mask = np.where(solved[:B] >= 0, np.where(best == BIG, 0, best), -1).astype(np.int32)
    return value, best_mask, nodes, status


def test_child_pairs():
    for d, n in ((2, 2), (3, 9), (4, 28), (5, 75), (6, 186)):
        p = child_pairs(d)
        assert len(p) == n == d * 2 ** (d - 1) - d
        assert (np.diff(p[:, 0]) >= 0).all() and (p[:, 1] < d).all()


def test_reference_hand_cases():
    ended = np.array([[[2, 3], [-1, -1]], [[-1, -1], [-1, -1]]], np.int32)
    assert [a.tolist() for a in reference_value(ended)] == [[0, 0], [0, 0], [1, 1], [RESOLVED, RESOLVED]]
    two = np.array([[[1, 0], [0, 1]]], np.int32)  # the one set {0, 1}: either reply leaves one point
    assert [a.tolist() for a in reference_value(two)] == [[1], [3], [3], [RESOLVED]]
    # a root whose value is below the depth Zeillinger's host lets the agent reach
    roots = filtered_roots(np.random.default_rng(3), 48, 5, 3, 4)
    v, m, n, s = reference_value(roots, max_depth=4, max_nodes=20000)
    zd, _, zs = reference_search(roots, max_depth=32)
    both = (s == RESOLVED) & (zs == RESOLVED)
    assert both.sum() >= 8
    assert (v[both] <= zd[both]).all() and (v[both] < zd[both]).any()
    assert ((m >= 3) == (s == RESOLVED) & (v > 0)).all() and ((m == -1) == (s != RESOLVED)).all()


def test_reference_statuses():
    roots = filtered_roots(np.random.default_rng(4), 24, 5, 3, 6)
    full = reference_value(roots, max_depth=3, max_nodes=1 << 20)
    deep = full[3] == MAX_DEPTH
    assert deep.any() and (full[0][deep] == 3).all() and (full[1][deep] == -1).all()
    v1 = reference_value(roots, max_depth=1)
    assert ((v1[3] == RESOLVED) == (full[0] <= 1) & (full[3] == RESOLVED)).all()
    small = reference_value(roots, max_depth=3, max_nodes=20)
    assert (small[3] == MAX_NODES).any() and (small[2] <= 20).all()
    first = 9 * ((roots[:, :, 0] >= 0).sum(1) > 1)
    cap = int(first.sum() // 2)
    c = reference_value(roots, max_depth=3, capacity=cap)
    at_root = set(np.nonzero((c[3] == CAPACITY) & (c[0] == 0))[0])
    assert at_root and at_root == {r for r in np.nonzero(first > 0)[0] if first[:r + 1].sum() > cap}
    h = reference_value(roots, max_depth=3, history=len(roots) + int(first.sum()) + 40)
    assert (h[3] == HISTORY).any() and (h[2].sum() <= len(roots) + first.sum() + 40)
    assert ((h[3] == RESOLVED) <= (full[3] == RESOLVED)).all()
    assert (h[0][h[3] == RESOLVED] == full[0][h[3] == RESOLVED]).all()
    bound = (1 << 30) // 3
    at = np.array([[[bound, 0, 0], [0, 1, 0], [-1, -1, -1], [-1, -1, -1], [-1, -1, -1]]], np.int32)
    assert [a.tolist() for a in reference_value(at)] == [[0], [-1], [1], [INT32_BOUND]]


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


def gpu_value(roots, **kw):
    import torch
    import hironaka_b200 as hb
    r = hb.search_value(torch.as_tensor(np.ascontiguousarray(roots)).cuda(), **kw)
    assert r.value.dtype == torch.int32 and r.best_mask.dtype == torch.int32
    assert r.nodes.dtype == torch.int64 and r.status.dtype == torch.int8
    return tuple(x.cpu().numpy() for x in r)


def assert_same(got, exp, what):
    for name, g, e in zip(("value", "best_mask", "nodes", "status"), got, exp):
        assert np.array_equal(g, e), (what, name, np.nonzero(g != e)[0][:8], g[g != e][:8], e[g != e][:8])


# (N, d), max value of the roots, depth limit, node budget: trees of up to a few tens of thousands of states per root
SHAPES = [((5, 3), 6, 5, 4000), ((10, 3), 4, 5, 4000), ((5, 4), 3, 3, 25000), ((6, 5), 3, 2, 6000),
          ((4, 6), 2, 2, 40000)]


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[0])))
@pytest.mark.parametrize("reposition", [True, False], ids=["repos", "norepos"])
def test_value_matches_reference(lib, shape, reposition):
    (N, d), max_value, max_depth, max_nodes = shape
    roots = filtered_roots(np.random.default_rng(N * 100 + d), 12 if d == 6 else 33, N, d, max_value)
    args = dict(reposition=reposition, max_depth=max_depth, max_nodes=max_nodes)
    exp = reference_value(roots, **args)
    assert (exp[3] == RESOLVED).any() and (exp[0][exp[3] == RESOLVED] > 0).any()
    assert_same(gpu_value(roots, **args), exp, (shape, reposition))


@gpu
def test_value_warp_per_game_family(lib):
    """(10, 3) runs thread-per-game by default: the same search with the warp-per-game step everywhere."""
    from hironaka_b200 import ops
    roots = filtered_roots(np.random.default_rng(11), 65, 10, 3, 5)
    args = dict(max_depth=5, max_nodes=4000)
    exp = reference_value(roots, **args)
    ops.force_generic(True)
    try:
        got = gpu_value(roots, **args)
    finally:
        ops.force_generic(False)
    assert_same(got, exp, "force_generic")
    assert_same(gpu_value(roots, **args), exp, "default family")


@gpu
@pytest.mark.parametrize("reposition", [True, False], ids=["repos", "norepos"])
def test_value_statuses(lib, reposition):
    """Each cut provoked on purpose, and the results equal to the reference's."""
    roots = filtered_roots(np.random.default_rng(13), 40, 5, 3, 6)
    base = dict(reposition=reposition, max_depth=5, max_nodes=3000)
    for kw, st in ((dict(max_depth=1), MAX_DEPTH), (dict(max_depth=2), MAX_DEPTH), (dict(max_nodes=1), MAX_NODES),
                   (dict(max_nodes=40), MAX_NODES)):
        args = dict(base, **kw)
        got = gpu_value(roots, **args)
        assert (got[3] == st).any(), kw
        assert_same(got, reference_value(roots, **args), kw)
    first = 9 * ((roots[:, :, 0] >= 0).sum(1) > 1)
    for kw, st in ((dict(capacity=1), CAPACITY), (dict(capacity=int(first.sum()) // 2), CAPACITY),
                   (dict(capacity=400), CAPACITY), (dict(history=len(roots)), HISTORY),
                   (dict(history=len(roots) + int(first.sum()) // 2), HISTORY),
                   (dict(history=len(roots) + int(first.sum()) + 500), HISTORY),
                   (dict(capacity=300, history=2000), CAPACITY)):
        args = dict(base, **kw)
        got = gpu_value(roots, **args)
        assert (got[3] == st).any(), kw
        assert_same(got, reference_value(roots, **args), kw)


@gpu
@pytest.mark.parametrize("d", [2, 3, 5])
def test_value_int32_bound(lib, d):
    """Roots whose live entries sit just below and at floor(2^30 / d): below, the root is expanded; at, the root is cut
    before its first level."""
    N = 5
    bound = (1 << 30) // d
    roots = filtered_roots(np.random.default_rng(14 + d), 30, N, d, 4)
    for b, v in enumerate([bound - 1, bound, bound - 1, bound, bound - 2, bound]):
        x = np.full((N, d), -1, np.int32)
        x[0] = 0
        x[0, 0] = v
        x[1] = 0
        x[1, 1] = 1 + b % 2
        x[2] = 0
        x[2, d - 1] += 3
        roots[5 * b] = cport.step(x[None], None, None, C.HK_OP_NEWTON | C.HK_OP_REPOSITION, 0)[0][0]
    args = dict(max_depth=4 if d < 5 else 2, max_nodes=8000)
    got = gpu_value(roots, **args)
    assert_same(got, reference_value(roots, **args), d)
    assert (got[3][[5, 15, 25]] == INT32_BOUND).all() and (got[0][[5, 15, 25]] == 0).all()


@gpu
def test_value_deterministic_and_permutation(lib):
    rng = np.random.default_rng(15)
    roots = filtered_roots(rng, 200, 10, 3, 5)
    args = dict(max_depth=5, max_nodes=5000)
    a = gpu_value(roots, **args)
    assert_same(gpu_value(roots, **args), a, "repeat")
    perm = rng.permutation(len(roots))
    assert_same(gpu_value(roots[perm], **args), tuple(x[perm] for x in a), "permuted")
    assert (a[3] != CAPACITY).all() and (a[3] != HISTORY).all()


@gpu
def test_value_not_above_fixed_hosts(lib):
    """No fixed host ends the game sooner than the best host: value <= search_depth of Zeillinger's host and of the
    all-coordinates host wherever both are resolved."""
    import torch
    import hironaka_b200 as hb
    roots = filtered_roots(np.random.default_rng(16), 64, 5, 3, 5)
    v, m, n, s = gpu_value(roots, max_depth=6, max_nodes=1 << 16)
    ok = s == RESOLVED
    assert ok.sum() >= 16
    t = torch.as_tensor(roots).cuda()
    for host in ("zeillinger", "all_coord"):
        r = hb.search_depth(t, host, max_depth=40)
        both = ok & (r.status.cpu().numpy() == RESOLVED)
        assert both.sum() >= 8, host
        assert (v[both] <= r.depth.cpu().numpy()[both]).all(), host


@gpu
def test_value_best_mask_children(lib):
    """Playing best_mask at a resolved root and searching each agent reply gives value - 1 as the largest child value."""
    roots = filtered_roots(np.random.default_rng(17), 64, 5, 3, 5)
    v, m, n, s = gpu_value(roots, max_depth=6, max_nodes=1 << 16)
    idx = np.nonzero((s == RESOLVED) & (v > 0))[0]
    assert len(idx) >= 8
    ops = C.HK_OP_SHIFT | C.HK_OP_NEWTON | C.HK_OP_REPOSITION
    for r in idx:
        axes = [a for a in range(3) if m[r] >> a & 1]
        kids = cport.step(np.repeat(roots[r:r + 1], len(axes), 0), np.full(len(axes), m[r], np.int32),
                          np.array(axes, np.int32), ops, 0)[0]
        cv, _, _, cs = gpu_value(kids, max_depth=6, max_nodes=1 << 16)
        assert (cs == RESOLVED).all() and cv.max() == v[r] - 1, (r, cv, v[r])


@gpu
def test_value_rejects_arguments(lib):
    import torch
    import hironaka_b200 as hb
    from hironaka_b200 import ops
    roots = torch.as_tensor(filtered_roots(np.random.default_rng(18), 4, 5, 3, 6)).cuda()
    B, N, d = roots.shape
    ws = torch.empty(ops.search_value_workspace_bytes(B, N, d, 64, 1000), dtype=torch.uint8, device="cuda")
    outs = [torch.empty(B, dtype=t, device="cuda") for t in (torch.int32, torch.int32, torch.int64, torch.int8)]
    stream = torch.cuda.current_stream().cuda_stream
    base = dict(x=roots, N=N, d=d, dtype=C.HK_DTYPE_I32, ops=C.HK_OP_SHIFT | C.HK_OP_NEWTON | C.HK_OP_REPOSITION,
                max_depth=4, max_nodes=100, capacity=64, history=1000)

    def call(**kw):
        a = dict(base, **kw)
        return lib.hk_search_value(a["x"].data_ptr(), *(o.data_ptr() for o in outs), B, a["N"], a["d"], a["dtype"],
                                   a["ops"], a["max_depth"], a["max_nodes"], a["capacity"], a["history"], ws.data_ptr(),
                                   stream)
    assert call() == C.HK_OK
    assert call(x=roots.float(), dtype=C.HK_DTYPE_F32) == C.HK_ERR_UNSUPPORTED
    for dd in (1, 7):  # the same bytes read as another dimension
        assert call(N=N * d // dd if N * d % dd == 0 else 1, d=dd) == C.HK_ERR_UNSUPPORTED, dd
    for op in (C.HK_OP_SHIFT, C.HK_OP_NEWTON, C.HK_OP_SHIFT | C.HK_OP_REPOSITION,
               C.HK_OP_SHIFT | C.HK_OP_NEWTON | C.HK_OP_RESCALE, C.HK_OP_SHIFT | C.HK_OP_NEWTON | C.HK_OP_DEDUPE):
        assert call(ops=op) == C.HK_ERR_BAD_ARG, op
    for kw in (dict(max_depth=0), dict(max_nodes=0), dict(capacity=0), dict(history=B - 1), dict(history=1 << 31)):
        assert call(**kw) == C.HK_ERR_BAD_ARG, kw
    assert ops.search_value_workspace_bytes(B, N, 7, 64, 1000) == 0
    assert call() == C.HK_OK
    got = hb.search_value(roots, max_depth=4, max_nodes=100, capacity=64, history=1000)
    assert all(torch.equal(o, g) for o, g in zip(outs, got))
