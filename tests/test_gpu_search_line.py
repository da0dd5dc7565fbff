"""Lines of play from the game-tree searches (hk_search_depth_line, hk_search_value_line, hironaka_b200.search_*_line,
play_line) against level-synchronous references built from the oracle's C port.

The references are copies of tests/test_gpu_search.py's reference_search and tests/test_gpu_search_value.py's
reference_value that also keep each state's parent and return the lines:
- the worst line against a fixed host is the path to the first state of the root's deepest level (frontiers are in
  lexicographic order of the axes that lead to them), depth[r] moves;
- the optimal line of a resolved root of value v takes, from each state, the first group whose children are all solved
  by the root's round, and in it the lowest-rank child solved in that round, v moves.
The depth-line reference also keeps the history cut of the library: the states of all levels of the batch, cut after
the capacity, roots dropped from the highest index down.

The tests without the gpu mark hold the references to an independent recursive definition (a depth-first search on
the C port's step that plays the greedy rules) on hand cases, and replay the reference lines with the C port.  On the
GPU the lines and every other output must equal the references bit for bit, with every output prefilled with a
sentinel; the replayed lines must have their claimed properties under the library's own searches.
"""
import functools
import os

import numpy as np
import pytest

from hironaka_b200 import constants as C
from oracle import cport
from tests.test_gpu_search import filtered_roots, host_masks, popcount
from tests.test_gpu_search import SHAPES as DEPTH_SHAPES
from tests.test_gpu_search import reference_search
from tests.test_gpu_search_value import SHAPES as VALUE_SHAPES
from tests.test_gpu_search_value import child_pairs, reference_value

gpu = pytest.mark.gpu

RESOLVED, MAX_DEPTH, MAX_NODES, CAPACITY, INT32_BOUND, HISTORY = (
    C.HK_SEARCH_RESOLVED, C.HK_SEARCH_MAX_DEPTH, C.HK_SEARCH_MAX_NODES, C.HK_SEARCH_CAPACITY, C.HK_SEARCH_INT32_BOUND,
    C.HK_SEARCH_HISTORY)
BIG = 1 << 40


def step_ops(reposition):
    return C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)


def ended(x):
    return (np.asarray(x)[..., 0] >= 0).sum(-1) <= 1


# ---------------------------------------------------------------- reference side (no GPU)


def reference_depth_line(roots, host="zeillinger", reposition=True, max_depth=64, max_nodes=1 << 16, capacity=BIG,
                         history=BIG):
    """(depth, nodes, status, line_mask [B, max_depth], line_axis [B, max_depth]): reference_search with parents kept
    and the history as one more cut."""
    front = np.ascontiguousarray(roots, np.int32)
    B, N, d = front.shape
    ops = step_ops(reposition)
    bound = (1 << 30) // d
    depth = np.zeros(B, np.int32)
    nodes = np.ones(B, np.int64)
    status = np.zeros(B, np.int8)
    froot = np.arange(B)
    parent = np.full(B, -1, np.int64)  # the history: one entry per state of every level, the roots first
    hset = np.zeros(B, np.int64)
    haxis = np.zeros(B, np.int64)
    fh = np.arange(B)
    deep = np.arange(B)  # entry of the first state of the root's deepest level
    for level in range(max_depth + 1):
        first = np.r_[True, froot[1:] != froot[:-1]]
        deep[froot[first]] = fh[first]
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
        used = 0
        for r in np.unique(froot):  # increasing root order
            ch = children[r]
            if ch == 0:
                continue
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
                    depth[r] = level + 1
        parents = np.nonzero(keep[froot] & (c > 0))[0]
        if len(parents) == 0:
            break
        idx = np.repeat(parents, c[parents])
        axes = np.concatenate([[a for a in range(d) if S[i] >> a & 1] for i in parents]).astype(np.int32)
        h0 = len(parent)
        parent = np.concatenate([parent, fh[idx]])
        hset = np.concatenate([hset, S[idx]])
        haxis = np.concatenate([haxis, axes])
        front = cport.step(np.ascontiguousarray(front[idx]), S[idx], axes, ops, 0)[0]
        froot = froot[idx]
        fh = h0 + np.arange(len(idx))
    line_mask = np.zeros((B, max_depth), np.int32)
    line_axis = np.full((B, max_depth), -1, np.int32)
    for r in range(B):
        h = deep[r]
        for t in range(depth[r] - 1, -1, -1):
            line_mask[r, t], line_axis[r, t] = hset[h], haxis[h]
            h = parent[h]
        assert h == r
    return depth, nodes, status, line_mask, line_axis


def reference_value_line(roots, reposition=True, max_depth=16, max_nodes=1 << 22, capacity=BIG, history=BIG):
    """(value, best_mask, nodes, status, line_mask [B, max_depth], line_axis [B, max_depth]): reference_value with the
    whole history returned and walked down."""
    front = np.ascontiguousarray(roots, np.int32)
    B, N, d = front.shape
    ops = step_ops(reposition)
    bound = (1 << 30) // d
    pairs = child_pairs(d)
    nc = len(pairs)
    parent = np.full(B, -1, np.int64)
    gset = np.zeros(B, np.int64)
    rank = np.zeros(B, np.int64)
    rem = np.zeros(B, np.int64)
    solved = np.full(B, -1, np.int64)
    value = np.zeros(B, np.int32)
    best = np.full(B, BIG, np.int64)
    nodes = np.ones(B, np.int64)
    status = np.zeros(B, np.int8)
    fh = np.arange(B)
    froot = np.arange(B)
    for level in range(max_depth + 1):
        live = front[:, :, 0] >= 0
        is_ended = live.sum(1) <= 1
        new = fh[is_ended]
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
        pruned = is_ended.copy()
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
        for r in np.unique(froot):
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
                    used += ch
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
    line_mask = np.zeros((B, max_depth), np.int32)
    line_axis = np.full((B, max_depth), -1, np.int32)
    first_child = np.searchsorted(parent, np.arange(len(parent)))  # parent is non-decreasing
    for r in np.nonzero(status == RESOLVED)[0]:
        R = solved[r]
        h = r
        for t in range(R):
            kids = first_child[h] + np.arange(nc)
            assert (parent[kids] == h).all()
            s = solved[kids]
            for S_ in np.unique(pairs[:, 0]):  # increasing S
                g = pairs[:, 0] == S_
                if ((s[g] >= 0) & (s[g] <= R)).all():
                    j = np.nonzero(g & (s == R))[0][0]
                    break
            line_mask[r, t], line_axis[r, t] = pairs[j, 0], pairs[j, 1]
            h = kids[j]
    return value, best_mask, nodes, status, line_mask, line_axis


def one_step(x, S, a, reposition):
    return cport.step(np.ascontiguousarray(x[None]), np.array([S], np.int32), np.array([a], np.int32),
                      step_ops(reposition), 0)[0][0]


def dfs_depth_line(x, host, reposition):
    """The greedy rule by recursion: at each state the host's set, the smallest axis whose subtree is the deepest."""
    if ended(x):
        return []
    S = int(host_masks(x[None], host)[0])
    best = None
    for a in range(x.shape[1]):
        if S >> a & 1:
            line = [(S, a)] + dfs_depth_line(one_step(x, S, a, reposition), host, reposition)
            if best is None or len(line) > len(best):
                best = line
    return best


def dfs_value_line(x, reposition, max_value):
    """The optimal line by recursion: win(x, k) <=> the host can end the game in k moves; the host plays the smallest
    S that wins in v - 1 more moves whatever the reply, the agent the smallest axis whose child has value v - 1."""
    d = x.shape[1]
    sets = [S for S in range(1 << d) if bin(S).count("1") >= 2]

    @functools.lru_cache(maxsize=None)
    def kid(key, S, a):
        return one_step(np.frombuffer(key, np.int32).reshape(x.shape), S, a, reposition).tobytes()

    @functools.lru_cache(maxsize=None)
    def win(key, k):
        if ended(np.frombuffer(key, np.int32).reshape(x.shape)):
            return k >= 0
        if k <= 0:
            return False
        return any(all(win(kid(key, S, a), k - 1) for a in range(d) if S >> a & 1) for S in sets)

    key = x.tobytes()
    v = next((k for k in range(max_value + 1) if win(key, k)), None)
    if v is None:
        return None, []
    line = []
    for u in range(v, 0, -1):
        S = next(S for S in sets if all(win(kid(key, S, a), u - 1) for a in range(d) if S >> a & 1))
        a = next(a for a in range(d) if S >> a & 1 and not win(kid(key, S, a), u - 2))
        line.append((S, a))
        key = kid(key, S, a)
    return v, line


def as_moves(mask, axis, n):
    return [(int(mask[t]), int(axis[t])) for t in range(n)]


def test_reference_depth_line_hand_cases():
    two = np.array([[[1, 0], [0, 1]]], np.int32)  # either reply ends the game: the line is the smaller axis
    for host in ("zeillinger", "all_coord"):
        d, n, s, m, a = reference_depth_line(two, host, max_depth=3)
        assert d.tolist() == [1] and m.tolist() == [[3, 0, 0]] and a.tolist() == [[0, -1, -1]]
    # the all-coordinates host lets the agent cycle at d = 3: its trees resolve at d = 2
    for host, (N, dim), max_value in (("zeillinger", (5, 3), 5), ("all_coord", (5, 2), 10)):
        roots = filtered_roots(np.random.default_rng(21), 24, N, dim, max_value)
        for reposition in (True, False):
            d, n, s, m, a = reference_depth_line(roots, host, reposition, max_depth=32)
            full = reference_search(roots, host, reposition, max_depth=32)
            assert all(np.array_equal(x, y) for x, y in zip((d, n, s), full))
            assert (s == RESOLVED).all() and (d >= 3).sum() >= 4
            for r in range(len(roots)):
                assert as_moves(m[r], a[r], d[r]) == dfs_depth_line(roots[r], host, reposition), (host, r)
                assert (m[r, d[r]:] == 0).all() and (a[r, d[r]:] == -1).all()


def test_reference_value_line_hand_cases():
    two = np.array([[[1, 0], [0, 1]]], np.int32)
    v, b, n, s, m, a = reference_value_line(two, max_depth=2)
    assert v.tolist() == [1] and m.tolist() == [[3, 0]] and a.tolist() == [[0, -1]]
    roots = filtered_roots(np.random.default_rng(22), 24, 5, 3, 4)
    for reposition in (True, False):
        out = reference_value_line(roots, reposition, max_depth=3)
        assert all(np.array_equal(x, y) for x, y in zip(out[:4], reference_value(roots, reposition, max_depth=3)))
        v, b, n, s, m, a = out
        assert (s == RESOLVED).sum() >= 8 and (v[s == RESOLVED] >= 2).sum() >= 4 and (s == MAX_DEPTH).any()
        for r in range(len(roots)):
            dv, dline = dfs_value_line(roots[r], reposition, 3)
            if s[r] == RESOLVED:
                assert dv == v[r] and as_moves(m[r], a[r], v[r]) == dline, (reposition, r)
            else:
                assert s[r] == MAX_DEPTH and dv is None and (m[r] == 0).all() and (a[r] == -1).all()


def test_reference_lines_replay():
    """The reference lines replayed with the C port: the depth line plays the host's set and lasts depth moves; along
    the value line the value drops by one per move."""
    roots = filtered_roots(np.random.default_rng(23), 12, 5, 3, 5)
    d, n, s, m, a = reference_depth_line(roots, max_depth=32)
    for r in range(len(roots)):
        x = roots[r]
        for t in range(d[r]):
            assert not ended(x) and m[r, t] == host_masks(x[None], "zeillinger")[0] and m[r, t] >> a[r, t] & 1
            x = one_step(x, m[r, t], a[r, t], True)
            assert reference_search(x[None], max_depth=32)[0][0] == d[r] - t - 1
        assert ended(x)
    roots = filtered_roots(np.random.default_rng(22), 24, 5, 3, 4)
    v, b, n, s, m, a = reference_value_line(roots, max_depth=3)
    ok = np.nonzero((s == RESOLVED) & (v > 0))[0]
    assert len(ok) >= 4
    for r in ok:
        assert m[r, 0] == b[r]
        x = roots[r]
        for t in range(v[r]):
            x = one_step(x, m[r, t], a[r, t], True)
            assert reference_value(x[None], max_depth=3)[0][0] == v[r] - t - 1
        assert ended(x)


def test_reference_depth_line_history_cut():
    roots = filtered_roots(np.random.default_rng(24), 16, 5, 3, 8)
    first = popcount(host_masks(roots, "zeillinger")) * ~ended(roots)
    B = len(roots)
    for history, cap in ((B, BIG), (B + int(first.sum()) // 2, BIG), (B + int(first.sum()) // 2, int(first.sum()) // 4)):
        d, n, s, m, a = reference_depth_line(roots, max_depth=32, history=history, capacity=cap)
        at_root = {r for r in np.nonzero(first > 0)[0] if first[:r + 1].sum() > min(cap, history - B)}
        assert set(np.nonzero(d == 0)[0]) - set(np.nonzero(first == 0)[0]) == at_root
        expect = {r: CAPACITY if first[:r + 1].sum() > cap else HISTORY for r in at_root}
        assert {r: s[r] for r in at_root} == expect
    d, n, s, m, a = reference_depth_line(roots, max_depth=32, history=B + int(first.sum()) + 30)
    assert (s == HISTORY).any() and (n.sum() <= B + first.sum() + 30)


def test_workspace_sizes():
    """The old entries' workspaces are what they were; the depth line adds 7 bytes per history state and 12 per root."""
    import hironaka_b200
    if not os.path.exists(hironaka_b200.LIB_PATH):
        pytest.skip("library not built in this checkout (run python -m hironaka_b200.build)")
    from hironaka_b200 import ops

    def al(v):
        return (v + 255) // 256 * 256

    for B, N, d, cap, hist in ((1, 5, 3, 64, 1000), (33, 10, 3, 5000, 1 << 20), (1000, 64, 5, 1 << 16, 1 << 24)):
        P = max(B, cap)
        search = (2 * al(cap * N * d * 4) + 4 * al(cap * 4) + al(P * 4) + al(P) + al((P + 255) // 256 * 8) +
                  al(B * 8) + al(B * 4) + al(B * 8) + 2 * al(B * 4) + al(16))
        assert ops.search_workspace_bytes(B, N, d, cap) == search + 256
        value = search - al(P * 4) + al(P) + 2 * al(hist * 4) + al(hist * 4) + 2 * al(hist)
        assert ops.search_value_workspace_bytes(B, N, d, cap, hist) == value + 256
        line = search + al(hist * 4) + al(hist * 2) + al(hist) + al(B * 4) + al(B * 8)
        assert ops.search_depth_line_workspace_bytes(B, N, d, cap, hist) == line + 256
    assert ops.search_depth_line_workspace_bytes(4, 5, 3, 64, 3) == 0
    assert ops.search_depth_line_workspace_bytes(4, 5, 3, 64, 1 << 31) == 0
    assert ops.search_depth_line_workspace_bytes(4, 5, 3, 0, 100) == 0


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


SENTINEL = 0x5A5A5A5A


def sentinel_outputs(B, L, dtypes):
    import torch
    outs = [torch.full((B,), -7, dtype=t, device="cuda") for t in dtypes]
    outs += [torch.full((B, L), SENTINEL, dtype=torch.int32, device="cuda") for _ in range(2)]
    return outs


def gpu_depth_line(roots, host="zeillinger", reposition=True, max_depth=64, max_nodes=1 << 16, capacity=1 << 22,
                   history=1 << 24):
    """hk_search_depth_line through the C-ABI, every output prefilled with a sentinel."""
    import torch
    from hironaka_b200 import ops
    from hironaka_b200._lib import lib as _lib
    x = torch.as_tensor(np.ascontiguousarray(roots)).cuda()
    B, N, d = x.shape
    outs = sentinel_outputs(B, max_depth, (torch.int32, torch.int64, torch.int8))
    ws = torch.empty(ops.search_depth_line_workspace_bytes(B, N, d, capacity, history), dtype=torch.uint8, device="cuda")
    flags = C.HK_F_HOST_ZEILLINGER if host == "zeillinger" else C.HK_F_HOST_ALL_COORD
    rc = _lib().hk_search_depth_line(x.data_ptr(), *(o.data_ptr() for o in outs), B, N, d, C.HK_DTYPE_I32,
                                     step_ops(reposition), flags, max_depth, max_nodes, capacity, history,
                                     ws.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc == C.HK_OK
    return tuple(o.cpu().numpy() for o in outs)


def gpu_value_line(roots, reposition=True, max_depth=16, max_nodes=1 << 22, capacity=1 << 22, history=1 << 24):
    """hk_search_value_line through the C-ABI, every output prefilled with a sentinel."""
    import torch
    from hironaka_b200 import ops
    from hironaka_b200._lib import lib as _lib
    x = torch.as_tensor(np.ascontiguousarray(roots)).cuda()
    B, N, d = x.shape
    outs = sentinel_outputs(B, max_depth, (torch.int32, torch.int32, torch.int64, torch.int8))
    ws = torch.empty(ops.search_value_workspace_bytes(B, N, d, capacity, history), dtype=torch.uint8, device="cuda")
    rc = _lib().hk_search_value_line(x.data_ptr(), *(o.data_ptr() for o in outs), B, N, d, C.HK_DTYPE_I32,
                                     step_ops(reposition), max_depth, max_nodes, capacity, history, ws.data_ptr(),
                                     torch.cuda.current_stream().cuda_stream)
    assert rc == C.HK_OK
    return tuple(o.cpu().numpy() for o in outs)


def assert_same(got, exp, names, what):
    for name, g, e in zip(names, got, exp):
        assert g.shape == e.shape and np.array_equal(g, e), (what, name, np.argwhere(g != e)[:8].tolist())


DEPTH_NAMES = ("depth", "nodes", "status", "line_mask", "line_axis")
VALUE_NAMES = ("value", "best_mask", "nodes", "status", "line_mask", "line_axis")


def old_depth(roots, host, reposition, max_depth, max_nodes, capacity=1 << 22):
    import torch
    import hironaka_b200 as hb
    r = hb.search_depth(torch.as_tensor(np.ascontiguousarray(roots)).cuda(), host, reposition=reposition,
                        max_depth=max_depth, max_nodes=max_nodes, capacity=capacity)
    return tuple(x.cpu().numpy() for x in r)


def old_value(roots, **kw):
    import torch
    import hironaka_b200 as hb
    return tuple(x.cpu().numpy() for x in hb.search_value(torch.as_tensor(np.ascontiguousarray(roots)).cuda(), **kw))


# the shapes of tests/test_gpu_search.py, and d = 9 and 10, whose host sets use bits 8 and 9
WIDE_SHAPES = [((4, 9), 2), ((6, 9), 3), ((5, 10), 2)]


@gpu
@pytest.mark.parametrize("shape", DEPTH_SHAPES + WIDE_SHAPES, ids=lambda s: "x".join(map(str, s[0])))
@pytest.mark.parametrize("host", ["zeillinger", "all_coord"])
@pytest.mark.parametrize("reposition", [True, False], ids=["repos", "norepos"])
def test_depth_line_matches_reference(lib, shape, host, reposition):
    (N, d), max_value = shape
    roots = filtered_roots(np.random.default_rng(N * 100 + d * 10 + 7), 33, N, d, max_value)
    args = dict(host=host, reposition=reposition, max_depth=24, max_nodes=3000)
    got = gpu_depth_line(roots, **args)
    exp = reference_depth_line(roots, **args)
    if d > 8:
        assert (exp[3] >= 256).any(), "the lines should play sets with bit 8 or 9"
    assert_same(got, exp, DEPTH_NAMES, (shape, host, reposition))
    assert_same(got[:3], old_depth(roots, **args), DEPTH_NAMES, "search_depth")


@gpu
def test_depth_line_wide_sets_replay(lib):
    """At d = 9 the all-coordinates host plays 0x1FF: the lines replayed with play_line play host_policy's set."""
    import torch
    import hironaka_b200 as hb
    from hironaka_b200 import ops
    roots = torch.as_tensor(filtered_roots(np.random.default_rng(33), 33, 4, 9, 2)).cuda()
    for host in ("zeillinger", "all_coord"):
        res = hb.search_depth_line(roots, host, max_depth=12, max_nodes=3000)
        states = hb.play_line(roots, res.mask, res.axis)
        depth, mask = res.depth.cpu().numpy(), res.mask.cpu().numpy()
        assert (mask >= 256).any(), host
        for t in range(12):
            on = depth > t
            policy = ops.host_policy(states[:, t].contiguous(), host).cpu().numpy()
            assert (mask[on, t] == policy[on]).all(), (host, t)


@gpu
@pytest.mark.parametrize("shape", VALUE_SHAPES, ids=lambda s: "x".join(map(str, s[0])))
@pytest.mark.parametrize("reposition", [True, False], ids=["repos", "norepos"])
def test_value_line_matches_reference(lib, shape, reposition):
    (N, d), max_value, max_depth, max_nodes = shape
    roots = filtered_roots(np.random.default_rng(N * 100 + d), 12 if d == 6 else 33, N, d, max_value)
    args = dict(reposition=reposition, max_depth=max_depth, max_nodes=max_nodes)
    exp = reference_value_line(roots, **args)
    assert ((exp[3] == RESOLVED) & (exp[0] > 0)).any()
    got = gpu_value_line(roots, **args)
    assert_same(got, exp, VALUE_NAMES, (shape, reposition))
    assert_same(got[:4], old_value(roots, **args), VALUE_NAMES, "search_value")


@gpu
def test_lines_warp_per_game_family(lib):
    """(10, 3) runs thread-per-game by default: the same lines with the warp-per-game step everywhere."""
    from hironaka_b200 import ops
    roots = filtered_roots(np.random.default_rng(25), 65, 10, 3, 5)
    dargs = dict(max_depth=24, max_nodes=3000)
    vargs = dict(max_depth=5, max_nodes=4000)
    dexp = reference_depth_line(roots, **dargs)
    vexp = reference_value_line(roots, **vargs)
    ops.force_generic(True)
    try:
        dgot = gpu_depth_line(roots, **dargs)
        vgot = gpu_value_line(roots, **vargs)
    finally:
        ops.force_generic(False)
    assert_same(dgot, dexp, DEPTH_NAMES, "force_generic depth")
    assert_same(vgot, vexp, VALUE_NAMES, "force_generic value")
    assert_same(gpu_depth_line(roots, **dargs), dexp, DEPTH_NAMES, "default family depth")
    assert_same(gpu_value_line(roots, **vargs), vexp, VALUE_NAMES, "default family value")


@gpu
@pytest.mark.parametrize("host", ["zeillinger", "all_coord"])
@pytest.mark.parametrize("reposition", [True, False], ids=["repos", "norepos"])
def test_depth_line_properties(lib, host, reposition):
    """Replayed with play_line: every mask is the host's choice on its state; a resolved root's line ends after exactly
    depth moves at an ended state; the search from the state after t moves has depth - t.  (The all-coordinates host
    lets the agent cycle at d = 3, so its roots are d = 2.)"""
    import torch
    import hironaka_b200 as hb
    from hironaka_b200 import ops
    d = 3 if host == "zeillinger" else 2
    roots = torch.as_tensor(filtered_roots(np.random.default_rng(26), 200, 10, d, 8 if d == 3 else 30)).cuda()
    B = len(roots)
    res = hb.search_depth_line(roots, host, reposition=reposition, max_depth=40, max_nodes=5000)
    assert isinstance(res, hb.DepthLine) and res.mask.shape == (B, 40)
    states = hb.play_line(roots, res.mask, res.axis, reposition=reposition)
    assert states.shape == (B, 41) + tuple(roots.shape[1:]) and states.dtype == torch.int32
    depth = res.depth.cpu().numpy()
    resolved = res.status.cpu().numpy() == RESOLVED
    assert resolved.sum() >= 100 and (depth[resolved] >= 3).sum() >= 20
    mask, axis = res.mask.cpu().numpy(), res.axis.cpu().numpy()
    st = states.cpu().numpy()
    for t in range(40):
        on = depth > t
        if not on.any():
            break
        policy = ops.host_policy(states[:, t].contiguous(), host).cpu().numpy()
        assert (mask[on, t] == policy[on]).all() and (mask[on, t] >> axis[on, t] & 1).all(), t
        assert not ended(st[on, t]).any(), t
        sub = np.nonzero(on & resolved)[0]
        r = hb.search_depth(states[sub, t].contiguous(), host, reposition=reposition, max_depth=40, max_nodes=5000)
        assert (r.depth.cpu().numpy() == depth[sub] - t).all(), t
    rows = np.arange(B)
    assert ended(st[rows[resolved], depth[resolved]]).all()
    assert all((st[r, depth[r]:] == st[r, depth[r]]).all() for r in range(B))


@gpu
@pytest.mark.parametrize("reposition", [True, False], ids=["repos", "norepos"])
def test_value_line_properties(lib, reposition):
    """Replayed with play_line: the state after t moves of a resolved root's line has value - t, the first mask is
    best_mask, and the line ends at an ended state."""
    import hironaka_b200 as hb
    import torch
    roots = torch.as_tensor(filtered_roots(np.random.default_rng(27), 128, 5, 3, 5)).cuda()
    res = hb.search_value_line(roots, reposition=reposition, max_depth=6, max_nodes=1 << 16)
    assert isinstance(res, hb.ValueLine)
    value, best = res.value.cpu().numpy(), res.best_mask.cpu().numpy()
    resolved = res.status.cpu().numpy() == RESOLVED
    assert (resolved & (value >= 3)).sum() >= 8
    states = hb.play_line(roots, res.mask, res.axis, reposition=reposition)
    st = states.cpu().numpy()
    mask = res.mask.cpu().numpy()
    on = resolved & (value > 0)
    assert (mask[on, 0] == best[on]).all()
    for t in range(1, 7):
        sub = np.nonzero(resolved & (value >= t))[0]
        if not len(sub):
            break
        r = hb.search_value(states[sub, t].contiguous(), reposition=reposition, max_depth=6, max_nodes=1 << 16)
        assert (r.status.cpu().numpy() == RESOLVED).all() and (r.value.cpu().numpy() == value[sub] - t).all(), t
    rows = np.nonzero(resolved)[0]
    assert ended(st[rows, value[rows]]).all()
    assert (res.axis.cpu().numpy()[~resolved] == -1).all()


@gpu
def test_depth_line_statuses(lib):
    """Each cut provoked, the history from the highest root index down; a cut root's line is still a path of depth
    moves that plays the host's choice."""
    roots = filtered_roots(np.random.default_rng(28), 65, 10, 3, 10)
    B = len(roots)
    first = popcount(host_masks(roots, "zeillinger")) * ~ended(roots)
    base = dict(max_depth=30, max_nodes=2000)
    cases = [(dict(max_depth=2), MAX_DEPTH), (dict(max_nodes=20), MAX_NODES), (dict(capacity=int(first.sum()) // 2),
             CAPACITY), (dict(capacity=500), CAPACITY), (dict(history=B), HISTORY),
             (dict(history=B + int(first.sum()) // 2), HISTORY), (dict(history=B + int(first.sum()) + 700), HISTORY),
             (dict(history=B + int(first.sum()) // 2, capacity=int(first.sum()) * 3 // 4), HISTORY),
             (dict(history=3000, capacity=300), CAPACITY)]
    for kw, st in cases:
        args = dict(base, **kw)
        got = gpu_depth_line(roots, **args)
        assert (got[2] == st).any(), kw
        assert_same(got, reference_depth_line(roots, **args), DEPTH_NAMES, kw)
        # dropped before their first level, from the highest index down: CAPACITY past the capacity, else HISTORY
        cap, room = kw.get("capacity", 1 << 22), kw.get("history", 1 << 24) - B
        at_root = {r for r in np.nonzero(first > 0)[0] if first[:r + 1].sum() > min(cap, room)}
        assert at_root == set(np.nonzero((first > 0) & (got[0] == 0))[0]), kw
        assert {r: got[2][r] for r in at_root} == {r: CAPACITY if first[:r + 1].sum() > cap else HISTORY
                                                   for r in at_root}, kw
        depth, status, mask, axis = got[0], got[2], got[3], got[4]
        for r in np.nonzero(status != RESOLVED)[0][:12]:
            x = roots[r]
            for t in range(depth[r]):
                assert not ended(x) and mask[r, t] == host_masks(x[None], "zeillinger")[0], (kw, r, t)
                x = one_step(x, mask[r, t], axis[r, t], True)
            assert (axis[r, depth[r]:] == -1).all()


@gpu
def test_value_line_statuses(lib):
    """Each cut provoked: the outputs equal the reference's, and cut roots have empty lines."""
    roots = filtered_roots(np.random.default_rng(29), 40, 5, 3, 6)
    first = 9 * ~ended(roots)
    base = dict(max_depth=5, max_nodes=3000)
    for kw, st in ((dict(max_depth=2), MAX_DEPTH), (dict(max_nodes=40), MAX_NODES),
                   (dict(capacity=int(first.sum()) // 2), CAPACITY),
                   (dict(history=len(roots) + int(first.sum()) + 500), HISTORY)):
        args = dict(base, **kw)
        got = gpu_value_line(roots, **args)
        assert (got[3] == st).any(), kw
        assert_same(got, reference_value_line(roots, **args), VALUE_NAMES, kw)
        cut = got[3] != RESOLVED
        assert (got[4][cut] == 0).all() and (got[5][cut] == -1).all()


@gpu
def test_lines_deterministic_and_permutation(lib):
    rng = np.random.default_rng(30)
    roots = filtered_roots(rng, 200, 10, 3, 8)
    perm = rng.permutation(len(roots))
    dargs = dict(max_depth=30, max_nodes=5000)
    a = gpu_depth_line(roots, **dargs)
    assert_same(gpu_depth_line(roots, **dargs), a, DEPTH_NAMES, "repeat")
    assert_same(gpu_depth_line(roots[perm], **dargs), tuple(x[perm] for x in a), DEPTH_NAMES, "permuted")
    vargs = dict(max_depth=5, max_nodes=5000)
    roots = filtered_roots(rng, 200, 10, 3, 5)
    b = gpu_value_line(roots, **vargs)
    assert_same(gpu_value_line(roots, **vargs), b, VALUE_NAMES, "repeat")
    assert_same(gpu_value_line(roots[perm], **vargs), tuple(x[perm] for x in b), VALUE_NAMES, "permuted")
    assert (a[2] == RESOLVED).sum() > 100 and ((b[3] == RESOLVED) & (b[0] > 1)).sum() > 5


@gpu
def test_lines_python_entries(lib):
    """hironaka_b200.search_*_line with their defaults give what the C-ABI gives, and the old entries' results."""
    import torch
    import hironaka_b200 as hb
    roots = filtered_roots(np.random.default_rng(31), 40, 5, 3, 5)
    t = torch.as_tensor(roots).cuda()
    dl = hb.search_depth_line(t, "all_coord", max_depth=20)
    assert_same(tuple(x.cpu().numpy() for x in dl), gpu_depth_line(roots, "all_coord", max_depth=20,
                                                                   max_nodes=1 << 16), DEPTH_NAMES, "depth")
    assert_same(tuple(x.cpu().numpy() for x in dl[:3]), old_depth(roots, "all_coord", True, 20, 1 << 16), DEPTH_NAMES,
                "old depth")
    vl = hb.search_value_line(t, max_depth=4, max_nodes=1 << 14)
    assert_same(tuple(x.cpu().numpy() for x in vl), gpu_value_line(roots, max_depth=4, max_nodes=1 << 14), VALUE_NAMES,
                "value")
    assert_same(tuple(x.cpu().numpy() for x in vl[:4]), old_value(roots, max_depth=4, max_nodes=1 << 14), VALUE_NAMES,
                "old value")
    ended_root = np.full((1, 5, 3), -1, np.int32)
    ended_root[0, 0] = [1, 2, 3]
    for out in (hb.search_depth_line(torch.as_tensor(ended_root).cuda(), max_depth=3),
                hb.search_value_line(torch.as_tensor(ended_root).cuda(), max_depth=3)):
        assert out.mask.tolist() == [[0, 0, 0]] and out.axis.tolist() == [[-1, -1, -1]]
        assert torch.equal(hb.play_line(torch.as_tensor(ended_root).cuda(), out.mask, out.axis)[0, 3].cpu(),
                           torch.as_tensor(ended_root[0]))


@gpu
def test_lines_reject_arguments(lib):
    import torch
    from hironaka_b200 import ops
    roots = torch.as_tensor(filtered_roots(np.random.default_rng(32), 4, 5, 3, 6)).cuda()
    B, N, d = roots.shape
    L = 4
    ws = torch.empty(max(ops.search_depth_line_workspace_bytes(B, N, d, 64, 1000),
                         ops.search_value_workspace_bytes(B, N, d, 64, 1000)), dtype=torch.uint8, device="cuda")
    dout = sentinel_outputs(B, L, (torch.int32, torch.int64, torch.int8))
    vout = sentinel_outputs(B, L, (torch.int32, torch.int32, torch.int64, torch.int8))
    stream = torch.cuda.current_stream().cuda_stream
    ops_ = C.HK_OP_SHIFT | C.HK_OP_NEWTON | C.HK_OP_REPOSITION

    def depth_call(x=roots, n=N, dd=d, dtype=C.HK_DTYPE_I32, history=1000, line_mask=True, line_axis=True):
        p = [o.data_ptr() for o in dout]
        p[3] = p[3] if line_mask else None
        p[4] = p[4] if line_axis else None
        return lib.hk_search_depth_line(x.data_ptr(), *p, B, n, dd, dtype, ops_, C.HK_F_HOST_ZEILLINGER, L, 100, 64,
                                        history, ws.data_ptr(), stream)

    def value_call(x=roots, n=N, dd=d, dtype=C.HK_DTYPE_I32, history=1000, line_mask=True, line_axis=True):
        p = [o.data_ptr() for o in vout]
        p[4] = p[4] if line_mask else None
        p[5] = p[5] if line_axis else None
        return lib.hk_search_value_line(x.data_ptr(), *p, B, n, dd, dtype, ops_, L, 100, 64, history, ws.data_ptr(),
                                        stream)

    for call in (depth_call, value_call):
        assert call() == C.HK_OK
        assert call(line_mask=False) == C.HK_ERR_BAD_ARG
        assert call(line_axis=False) == C.HK_ERR_BAD_ARG
        for h in (B - 1, 0, 1 << 31):
            assert call(history=h) == C.HK_ERR_BAD_ARG, h
        assert call(x=roots.float(), dtype=C.HK_DTYPE_F32) == C.HK_ERR_UNSUPPORTED
        assert call() == C.HK_OK
    for dd in (1, 7):  # the same bytes read as another dimension
        assert value_call(n=N * d // dd if N * d % dd == 0 else 1, dd=dd) == C.HK_ERR_UNSUPPORTED, dd
    with pytest.raises(ValueError):
        import hironaka_b200 as hb
        hb.search_depth_line(roots, "random")
