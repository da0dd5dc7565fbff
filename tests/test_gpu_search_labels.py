"""Value labels from the game-value search (hk_search_value_labels, hironaka_b200.search_value_labels) against a
level-synchronous reference built from the oracle's C port.

The reference is a copy of tests/test_gpu_search_line.py's reference_value_line that also keeps, for every entry of
the history, its level, its root and its rows.  Its labels are the entries solved in a round R above their level l, in
history order: the value R - l, host move g optimal when every child of group g is solved, the path from the parents
and the rows from the frontier.

The tests without the gpu mark hold the reference labels to an independent recursive definition (win(x, k): the host
can end the game from x within k moves, on the C port's step): win(x, v) holds and win(x, v - 1) does not, and the
optimal set is exactly the sets S whose every child wins within v - 1.  On the GPU every output must equal the
reference bit for bit, with every output prefilled with a sentinel; the labels must have their claimed properties
under the library's own searches.
"""
import functools
import os

import numpy as np
import pytest

from hironaka_b200 import constants as C
from oracle import cport
from tests.test_gpu_search import filtered_roots, popcount
from tests.test_gpu_search_value import SHAPES as VALUE_SHAPES
from tests.test_gpu_search_value import child_pairs, reference_value

gpu = pytest.mark.gpu

RESOLVED, MAX_DEPTH, MAX_NODES, CAPACITY, INT32_BOUND, HISTORY = (
    C.HK_SEARCH_RESOLVED, C.HK_SEARCH_MAX_DEPTH, C.HK_SEARCH_MAX_NODES, C.HK_SEARCH_CAPACITY, C.HK_SEARCH_INT32_BOUND,
    C.HK_SEARCH_HISTORY)
BIG = 1 << 40
LABEL_NAMES = ("root", "level", "value", "optimal", "mask", "axis")


def step_ops(reposition):
    return C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)


def ended(x):
    return (np.asarray(x)[..., 0] >= 0).sum(-1) <= 1


# ---------------------------------------------------------------- reference side (no GPU)


def reference_history(roots, reposition=True, max_depth=16, max_nodes=1 << 22, capacity=BIG, history=BIG):
    """(value, best_mask, nodes, status, hist): reference_value_line's search, with the whole history returned as a
    dict of per-entry arrays: parent, gset, rank, rem, solved, level, root and rows."""
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
    hlevel = np.zeros(B, np.int64)
    hroot = np.arange(B)
    rows = [front]
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
        hlevel = np.concatenate([hlevel, np.full(len(idx), level + 1, np.int64)])
        front = cport.step(np.ascontiguousarray(front[idx]), S.astype(np.int32), A.astype(np.int32), ops, 0)[0]
        froot = froot[idx]
        hroot = np.concatenate([hroot, froot])
        rows.append(front)
        fh = h0 + np.arange(len(idx))
    best_mask = np.where(solved[:B] >= 0, np.where(best == BIG, 0, best), -1).astype(np.int32)
    hist = dict(parent=parent, gset=gset, rank=rank, rem=rem, solved=solved, level=hlevel, root=hroot,
                rows=np.concatenate(rows))
    return value, best_mask, nodes, status, hist


def labels_of(hist, d, max_depth):
    """The labels of a reference history: (count, dict of root, level, value, optimal (int64 bit sets), mask, axis,
    state), in history order."""
    parent, solved, level = hist["parent"], hist["solved"], hist["level"]
    pairs = child_pairs(d)
    starts = np.nonzero(np.r_[True, pairs[1:, 0] != pairs[:-1, 0]])[0]  # first child of each group, group g = id g
    first_child = np.searchsorted(parent, np.arange(len(parent)))  # parent is non-decreasing
    lab = np.nonzero((solved >= 0) & (solved > level))[0]
    K = len(lab)
    out = dict(root=hist["root"][lab].astype(np.int32), level=level[lab].astype(np.int32),
               value=(solved[lab] - level[lab]).astype(np.int32), optimal=np.zeros(K, np.int64),
               mask=np.zeros((K, max_depth), np.int32), axis=np.full((K, max_depth), -1, np.int32),
               state=hist["rows"][lab])
    for k, h in enumerate(lab):
        kids = first_child[h] + starts
        assert (parent[kids] == h).all()
        out["optimal"][k] = sum(1 << g for g in np.nonzero(hist["rem"][kids] == 0)[0].tolist())
        e = h
        for t in range(level[h] - 1, -1, -1):
            S = hist["gset"][e]
            out["mask"][k, t] = S
            out["axis"][k, t] = [a for a in range(d) if S >> a & 1][hist["rank"][e]]
            e = parent[e]
        assert e == hist["root"][h]
    return K, out


def reference_labels(roots, reposition=True, max_depth=16, max_nodes=1 << 22, capacity=BIG, history=BIG):
    """(value, best_mask, nodes, status, count, labels)"""
    v, b, n, s, hist = reference_history(roots, reposition, max_depth, max_nodes, capacity, history)
    count, labels = labels_of(hist, np.asarray(roots).shape[2], max_depth)
    return v, b, n, s, count, labels


def one_step(x, S, a, reposition):
    return cport.step(np.ascontiguousarray(x[None]), np.array([S], np.int32), np.array([a], np.int32),
                      step_ops(reposition), 0)[0][0]


def win_oracle(shape, reposition):
    """win(key, k): the host can end the game from the state with bytes `key` within k moves, whatever the agent
    replies; and the sets S that end it within k moves."""
    N, d = shape
    sets = [S for S in range(1 << d) if bin(S).count("1") >= 2]

    @functools.lru_cache(maxsize=None)
    def kid(key, S, a):
        return one_step(np.frombuffer(key, np.int32).reshape(N, d), S, a, reposition).tobytes()

    @functools.lru_cache(maxsize=None)
    def win(key, k):
        if ended(np.frombuffer(key, np.int32).reshape(N, d)):
            return k >= 0
        if k <= 0:
            return False
        return any(winning(key, S, k) for S in sets)

    def winning(key, S, k):
        return all(win(kid(key, S, a), k - 1) for a in range(d) if S >> a & 1)

    def optimal(key, k):
        return sum(1 << g for g, S in enumerate(sets) if winning(key, S, k))
    return win, optimal


def check_against_win(roots, reposition, labels, limit=None):
    """Every label (the first `limit`): value exact, optimal set exact."""
    win, optimal = win_oracle(roots.shape[1:], reposition)
    K = len(labels["value"]) if limit is None else min(limit, len(labels["value"]))
    for k in range(K):
        key = np.ascontiguousarray(labels["state"][k]).tobytes()
        v = int(labels["value"][k])
        assert win(key, v) and not win(key, v - 1), k
        assert int(labels["optimal"][k]) == optimal(key, v), k
    return K


# d = 6: two live rows that differ only in coordinates 4 and 5 are ended by the set {4, 5} (mask 48, HostActionEncoder
# id 41) and by no other set; a third row makes a root whose labels lie one level down
D6_ROOTS = np.array([
    [[0, 0, 0, 0, 1, 0], [0, 0, 0, 0, 0, 1], [-1] * 6, [-1] * 6],
    [[1, 0, 0, 0, 2, 0], [1, 0, 0, 0, 0, 2], [-1] * 6, [-1] * 6],
    [[0, 0, 0, 0, 1, 0], [0, 0, 0, 0, 0, 1], [1, 1, 0, 0, 0, 0], [-1] * 6],
    [[0, 0, 0, 1, 1, 0], [0, 0, 0, 0, 1, 1], [0, 0, 0, 1, 0, 1], [-1] * 6],
], np.int32)
D6_ARGS = dict(max_depth=2, max_nodes=1 << 16)


def test_reference_labels_hand_cases():
    two = np.array([[[1, 0], [0, 1]]], np.int32)  # the one set {0, 1} (id 0) ends the game: value 1
    v, b, n, s, count, lab = reference_labels(two, max_depth=2)
    assert count == 1 and lab["root"].tolist() == [0] and lab["level"].tolist() == [0]
    assert lab["value"].tolist() == [1] and lab["optimal"].tolist() == [1]
    assert lab["mask"].tolist() == [[0, 0]] and lab["axis"].tolist() == [[-1, -1]]
    gone = np.array([[[2, 3], [-1, -1]], [[-1, -1], [-1, -1]]], np.int32)  # ended roots: no label
    assert reference_labels(gone)[4] == 0


def test_reference_labels_against_win():
    """Random (5, 3) and (5, 4) batches, with and without reposition: every label's value and optimal set are those of
    the win recursion, and a group is fully solved exactly when rem at its first child is 0."""
    for (N, d), mv, depth, budget, B, seed in (((5, 3), 6, 5, 4000, 24, 1), ((5, 4), 3, 3, 25000, 8, 3)):
        roots = filtered_roots(np.random.default_rng(seed), B, N, d, mv)
        for reposition in (True, False):
            v, b, n, s, hist = reference_history(roots, reposition, depth, budget)
            count, lab = labels_of(hist, d, depth)
            assert count >= 10 and (lab["value"] >= 2).any(), ((N, d), reposition)
            assert check_against_win(roots, reposition, lab) == count
            assert all(np.array_equal(x, y) for x, y in zip((v, b, n, s), reference_value(roots, reposition, depth,
                                                                                          budget)))
            # rem at a group's first child counts its unsolved children
            parent, solved, rem = hist["parent"], hist["solved"], hist["rem"]
            heads = np.nonzero((hist["rank"] == 0) & (parent >= 0))[0]
            size = popcount(hist["gset"][heads])
            unsolved = np.array([(solved[h:h + k] < 0).sum() for h, k in zip(heads, size)])
            assert np.array_equal(rem[heads], unsolved)


def test_reference_labels_under_cut_roots():
    """Roots cut by the node budget and by the depth limit still contribute exact labels."""
    roots = filtered_roots(np.random.default_rng(41), 40, 5, 3, 6)
    for kw, st in ((dict(max_depth=3, max_nodes=1 << 20), MAX_DEPTH), (dict(max_depth=5, max_nodes=3000), MAX_NODES)):
        v, b, n, s, count, lab = reference_labels(roots, **kw)
        under = s[lab["root"]] == st
        assert under.sum() >= 3, kw
        sub = {k: x[under] for k, x in lab.items()}
        assert check_against_win(roots, True, sub, limit=40) > 0


def test_reference_labels_d6_upper_word():
    v, b, n, s, count, lab = reference_labels(D6_ROOTS, **D6_ARGS)
    assert (lab["optimal"] >> 41 & 1).any() and (lab["optimal"] >= 1 << 32).sum() >= 2
    assert lab["optimal"][:1].tolist() == [1 << 41]
    assert (lab["level"] == 1).any()
    check_against_win(D6_ROOTS, True, lab, limit=12)


def test_reference_labels_replay():
    """The reference labels' paths replayed with the C port give their rows."""
    roots = filtered_roots(np.random.default_rng(6), 16, 5, 3, 6)
    for reposition in (True, False):
        v, b, n, s, count, lab = reference_labels(roots, reposition, max_depth=5, max_nodes=4000)
        assert count > 20 and (lab["level"] >= 2).any()
        for k in range(count):
            x = roots[lab["root"][k]]
            for t in range(lab["level"][k]):
                x = one_step(x, lab["mask"][k, t], lab["axis"][k, t], reposition)
            assert np.array_equal(x, lab["state"][k]), k
            L = lab["level"][k]
            assert (lab["mask"][k, L:] == 0).all() and (lab["axis"][k, L:] == -1).all()


def test_workspace_sizes():
    """hk_search_value's workspace, then 8 bytes per 256-state tile of the history, 8 per 1024 tiles, 8 for the total
    and 4 per tile for its level."""
    import hironaka_b200
    if not os.path.exists(hironaka_b200.LIB_PATH):
        pytest.skip("library not built in this checkout (run python -m hironaka_b200.build)")
    from hironaka_b200 import ops

    def al(v):
        return (v + 255) // 256 * 256

    for B, N, d, cap, hist in ((1, 5, 3, 64, 1000), (33, 10, 3, 5000, 1 << 20), (1000, 64, 5, 1 << 16, (1 << 31) - 1)):
        tiles = (hist + 255) // 256
        extra = al(tiles * 8) + al((tiles + 1023) // 1024 * 8) + al(8) + al(tiles * 4)
        assert (ops.search_value_labels_workspace_bytes(B, N, d, cap, hist) ==
                ops.search_value_workspace_bytes(B, N, d, cap, hist) + extra)
    for args in ((4, 5, 3, 64, 3), (4, 5, 3, 64, 1 << 31), (4, 5, 3, 0, 100), (4, 5, 7, 64, 100)):
        assert ops.search_value_labels_workspace_bytes(*args) == 0, args


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
SENTINEL64 = 0x5A5A5A5A5A5A5A5A


def gpu_labels(roots, max_labels=None, reposition=True, max_depth=16, max_nodes=1 << 22, capacity=1 << 22,
               history=1 << 24, null_labels=False):
    """hk_search_value_labels through the C-ABI, every output prefilled with a sentinel: (value, best_mask, nodes,
    status, count, labels) with the label buffers whole ([max_labels] ...; the default max_labels is 4096)."""
    import ctypes
    import torch
    from hironaka_b200 import ops
    from hironaka_b200._lib import lib as _lib
    x = torch.as_tensor(np.ascontiguousarray(roots)).cuda()
    B, N, d = x.shape
    M = 4096 if max_labels is None else max_labels
    outs = [torch.full((B,), -7, dtype=t, device="cuda") for t in (torch.int32, torch.int32, torch.int64, torch.int8)]
    lab = dict(root=torch.full((M,), SENTINEL, dtype=torch.int32, device="cuda"),
               level=torch.full((M,), SENTINEL, dtype=torch.int32, device="cuda"),
               value=torch.full((M,), SENTINEL, dtype=torch.int32, device="cuda"),
               optimal=torch.full((M,), SENTINEL64, dtype=torch.int64, device="cuda"),
               mask=torch.full((M, max_depth), SENTINEL, dtype=torch.int32, device="cuda"),
               axis=torch.full((M, max_depth), SENTINEL, dtype=torch.int32, device="cuda"))
    ws = torch.empty(max(ops.search_value_labels_workspace_bytes(B, N, d, capacity, history), 1), dtype=torch.uint8,
                     device="cuda")
    count = ctypes.c_int64(-3)
    ptrs = [None] * 6 if null_labels else [lab[k].data_ptr() for k in LABEL_NAMES]
    rc = _lib().hk_search_value_labels(x.data_ptr(), *(o.data_ptr() for o in outs), M, ctypes.addressof(count), *ptrs,
                                       B, N, d, C.HK_DTYPE_I32, step_ops(reposition), max_depth, max_nodes, capacity,
                                       history, ws.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc == C.HK_OK
    return tuple(o.cpu().numpy() for o in outs) + (count.value, {k: t.cpu().numpy() for k, t in lab.items()})


def assert_labels(got, exp, what):
    """got: gpu_labels' output; exp: reference_labels' output.  The shared outputs, the count, the first
    min(count, max_labels) labels, and the sentinel in the rest of every buffer."""
    for name, g, e in zip(("value", "best_mask", "nodes", "status"), got[:4], exp[:4]):
        assert np.array_equal(g, e), (what, name, np.nonzero(g != e)[0][:8])
    assert got[4] == exp[4], (what, "count", got[4], exp[4])
    M = len(got[5]["root"])
    K = min(got[4], M)
    for name in LABEL_NAMES:
        g, e = got[5][name], exp[5][name]
        assert g[:K].shape == e[:K].shape and np.array_equal(g[:K], e[:K]), (what, name,
                                                                               np.argwhere(g[:K] != e[:K])[:8].tolist())
        assert (g[K:] == (SENTINEL64 if name == "optimal" else SENTINEL)).all(), (what, name, "written past the labels")


def old_value(roots, **kw):
    import torch
    import hironaka_b200 as hb
    return tuple(x.cpu().numpy() for x in hb.search_value(torch.as_tensor(np.ascontiguousarray(roots)).cuda(), **kw))


@gpu
@pytest.mark.parametrize("shape", VALUE_SHAPES, ids=lambda s: "x".join(map(str, s[0])))
@pytest.mark.parametrize("reposition", [True, False], ids=["repos", "norepos"])
def test_labels_match_reference(lib, shape, reposition):
    (N, d), max_value, max_depth, max_nodes = shape
    roots = filtered_roots(np.random.default_rng(N * 100 + d + 1), 12 if d == 6 else 33, N, d, max_value)
    args = dict(reposition=reposition, max_depth=max_depth, max_nodes=max_nodes)
    exp = reference_labels(roots, **args)
    got = gpu_labels(roots, max_labels=exp[4] + 5, **args)
    assert_labels(got, exp, (shape, reposition))
    assert all(np.array_equal(g, e) for g, e in zip(got[:4], old_value(roots, **args)))


@gpu
def test_labels_d6_upper_word(lib):
    exp = reference_labels(D6_ROOTS, **D6_ARGS)
    assert (exp[5]["optimal"] >= 1 << 32).sum() >= 2
    assert_labels(gpu_labels(D6_ROOTS, **D6_ARGS), exp, "d = 6")


@gpu
def test_labels_warp_per_game_family(lib):
    """(10, 3) runs thread-per-game by default: the same labels with the warp-per-game step everywhere."""
    from hironaka_b200 import ops
    roots = filtered_roots(np.random.default_rng(40), 65, 10, 3, 5)
    args = dict(max_depth=5, max_nodes=4000)
    exp = reference_labels(roots, **args)
    assert exp[4] > 100
    ops.force_generic(True)
    try:
        got = gpu_labels(roots, **args)
        got6 = gpu_labels(D6_ROOTS, **D6_ARGS)
    finally:
        ops.force_generic(False)
    assert_labels(got, exp, "force_generic")
    assert_labels(got6, reference_labels(D6_ROOTS, **D6_ARGS), "force_generic d = 6")
    assert_labels(gpu_labels(roots, **args), exp, "default family")


@gpu
def test_labels_statuses(lib):
    """Each cut provoked, CAPACITY and HISTORY included: the outputs are still the reference's, and the cut roots have
    labels."""
    roots = filtered_roots(np.random.default_rng(41), 40, 5, 3, 6)
    first = 9 * ~ended(roots)
    base = dict(max_depth=5, max_nodes=3000)
    for kw, st in ((dict(max_depth=2), MAX_DEPTH), (dict(), MAX_NODES), (dict(capacity=int(first.sum()) * 3), CAPACITY),
                   (dict(history=len(roots) + int(first.sum()) * 4), HISTORY)):
        args = dict(base, **kw)
        exp = reference_labels(roots, **args)
        got = gpu_labels(roots, **args)
        assert_labels(got, exp, kw)
        assert (got[3][exp[5]["root"]] == st).any(), kw


@gpu
def test_labels_truncation(lib):
    """max_labels below the count: the reference prefix, the full count, the sentinel after; max_labels = 0 with null
    label pointers: the count alone."""
    roots = filtered_roots(np.random.default_rng(42), 40, 5, 3, 6)
    args = dict(max_depth=5, max_nodes=3000)
    exp = reference_labels(roots, **args)
    assert exp[4] > 100
    for M in (1, 7, 64, exp[4] - 1, exp[4], exp[4] + 1):
        assert_labels(gpu_labels(roots, max_labels=M, **args), exp, M)
    got = gpu_labels(roots, max_labels=0, null_labels=True, **args)
    assert got[4] == exp[4] and all(np.array_equal(g, e) for g, e in zip(got[:4], exp[:4]))


@gpu
def test_labels_small_batches(lib):
    """Ended-only roots give no label; B = 1; B = 0 gives count 0."""
    import torch
    import hironaka_b200 as hb
    gone = np.full((3, 5, 3), -1, np.int32)
    gone[0, 0] = [1, 2, 3]
    gone[2, 1] = [0, 4, 1]
    got = gpu_labels(gone, max_depth=3)
    assert got[4] == 0 and (got[5]["root"] == SENTINEL).all()
    assert_labels(got, reference_labels(gone, max_depth=3), "ended")
    roots = filtered_roots(np.random.default_rng(43), 40, 5, 3, 6)
    r = reference_labels(roots, max_depth=5, max_nodes=3000)[5]["root"][0]
    one = roots[r:r + 1]
    exp = reference_labels(one, max_depth=5, max_nodes=3000)
    assert exp[4] >= 1
    assert_labels(gpu_labels(one, max_depth=5, max_nodes=3000), exp, "B = 1")
    assert gpu_labels(np.zeros((0, 5, 3), np.int32))[4] == 0
    res = hb.search_value_labels(torch.zeros((0, 5, 3), dtype=torch.int32, device="cuda"), max_depth=3)
    assert res.count == 0 and res.state.shape == (0, 5, 3) and res.optimal.shape == (0, 4)


@gpu
def test_labels_python_entry(lib):
    """hironaka_b200.search_value_labels: the C-ABI's labels, the optimal sets decoded into HostActionEncoder columns,
    and the rows of the reference."""
    import torch
    import hironaka_b200 as hb
    from hironaka_b200 import host_action
    roots = filtered_roots(np.random.default_rng(44), 33, 5, 3, 6)
    for reposition in (True, False):
        exp = reference_labels(roots, reposition, max_depth=5, max_nodes=4000)
        res = hb.search_value_labels(torch.as_tensor(roots).cuda(), reposition=reposition, max_depth=5,
                                     max_nodes=4000)
        assert isinstance(res, hb.ValueLabels) and res.count == exp[4] and res.state.dtype == torch.int32
        assert all(np.array_equal(g.cpu().numpy(), e) for g, e in zip(res[:4], exp[:4]))
        lab = exp[5]
        for name, got in (("root", res.root), ("level", res.level), ("value", res.label_value), ("mask", res.mask),
                          ("axis", res.axis), ("state", res.state)):
            assert np.array_equal(got.cpu().numpy(), lab[name]), (reposition, name)
        G = len(host_action.action_masks(3))
        bits = (lab["optimal"][:, None] >> np.arange(G)) & 1
        assert res.optimal.shape == (exp[4], G) and np.array_equal(res.optimal.cpu().numpy(), bits.astype(bool))
    few = hb.search_value_labels(torch.as_tensor(roots).cuda(), max_depth=5, max_nodes=4000, max_labels=10)
    assert few.count == exp[4] and len(few.root) == 10 and few.state.shape == (10, 5, 3)


@gpu
@pytest.mark.parametrize("reposition", [True, False], ids=["repos", "norepos"])
def test_labels_properties(lib, reposition):
    """Through the library's own searches: search_value of each label's state gives its value; best_mask of a
    label's state is its lowest optimal move; every child of an optimal move has a smaller value; every state of a
    resolved root's optimal line is a label with the line's prefix as its path."""
    import torch
    import hironaka_b200 as hb
    from hironaka_b200 import host_action
    roots = torch.as_tensor(filtered_roots(np.random.default_rng(45), 96, 5, 3, 6)).cuda()
    kw = dict(reposition=reposition, max_depth=6, max_nodes=1 << 14)
    res = hb.search_value_labels(roots, **kw)
    K = res.count
    assert K >= 200 and (res.status.cpu().numpy() != RESOLVED).any()
    lv = res.label_value.cpu().numpy()
    sv = hb.search_value(res.state, **kw)
    assert (sv.status.cpu().numpy() == RESOLVED).all() and np.array_equal(sv.value.cpu().numpy(), lv)
    masks = np.array(host_action.action_masks(3))
    opt = res.optimal.cpu().numpy()
    assert np.array_equal(sv.best_mask.cpu().numpy(), masks[opt.argmax(1)])
    # the children of every optimal move: value below the label's
    k_idx, g_idx = np.nonzero(opt)
    S = masks[g_idx]
    rows, sets, axes = [], [], []
    for a in range(3):
        on = (S >> a & 1).astype(bool)
        rows.append(k_idx[on])
        sets.append(S[on])
        axes.append(np.full(on.sum(), a))
    rows, sets, axes = np.concatenate(rows), np.concatenate(sets), np.concatenate(axes)
    kids = res.state[torch.as_tensor(rows, device="cuda")].contiguous()
    hb.ops.step(kids, torch.as_tensor(sets, dtype=torch.int32, device="cuda"),
                torch.as_tensor(axes, dtype=torch.int32, device="cuda"), ops=step_ops(reposition))
    kv = hb.search_value(kids, **kw)
    assert (kv.status.cpu().numpy() == RESOLVED).all() and (kv.value.cpu().numpy() < lv[rows]).all()
    # optimal lines are made of labels
    line = hb.search_value_line(roots, **kw)
    root, level = res.root.cpu().numpy(), res.level.cpu().numpy()
    mask, axis = res.mask.cpu().numpy(), res.axis.cpu().numpy()
    found = {}
    for k in range(K):
        found.setdefault((int(root[k]), int(level[k])), set()).add(tuple(mask[k, :level[k]]) + tuple(axis[k, :level[k]]))
    value, status = line.value.cpu().numpy(), line.status.cpu().numpy()
    lm, la = line.mask.cpu().numpy(), line.axis.cpu().numpy()
    checked = 0
    for r in np.nonzero((status == RESOLVED) & (value > 0))[0]:
        for t in range(value[r]):
            assert tuple(lm[r, :t]) + tuple(la[r, :t]) in found.get((int(r), t), set()), (r, t)
            checked += 1
    assert checked >= 20


@gpu
def test_labels_deterministic_and_permutation(lib):
    """The same call twice gives the same labels; a permuted batch gives, root by root, the same labels as sets."""
    rng = np.random.default_rng(46)
    roots = filtered_roots(rng, 120, 10, 3, 5)
    perm = rng.permutation(len(roots))
    args = dict(max_depth=5, max_nodes=5000, max_labels=1 << 15)
    a = gpu_labels(roots, **args)
    assert a[4] > 500
    b = gpu_labels(roots, **args)
    assert a[4] == b[4] and all(np.array_equal(a[5][k], b[5][k]) for k in LABEL_NAMES)
    p = gpu_labels(roots[perm], **args)
    assert p[4] == a[4]

    def per_root(out, relabel):
        lab = out[5]
        K = out[4]
        return sorted((int(relabel[lab["root"][k]]), int(lab["level"][k]), int(lab["value"][k]), int(lab["optimal"][k]),
                       tuple(lab["mask"][k]), tuple(lab["axis"][k])) for k in range(K))
    assert per_root(a, np.arange(len(roots))) == per_root(p, perm)


@gpu
def test_labels_reject_arguments(lib):
    import ctypes
    import torch
    from hironaka_b200 import ops
    roots = torch.as_tensor(filtered_roots(np.random.default_rng(47), 4, 5, 3, 6)).cuda()
    B, N, d = roots.shape
    L, M = 4, 16
    ws = torch.empty(ops.search_value_labels_workspace_bytes(B, N, d, 64, 1000), dtype=torch.uint8, device="cuda")
    outs = [torch.empty(B, dtype=t, device="cuda") for t in (torch.int32, torch.int32, torch.int64, torch.int8)]
    lab = [torch.empty(M, dtype=torch.int32, device="cuda") for _ in range(3)]
    lab += [torch.empty(M, dtype=torch.int64, device="cuda")]
    lab += [torch.empty((M, L), dtype=torch.int32, device="cuda") for _ in range(2)]
    stream = torch.cuda.current_stream().cuda_stream
    count = ctypes.c_int64(0)

    def call(x=roots, n=N, dd=d, dtype=C.HK_DTYPE_I32, history=1000, max_labels=M, null=None, count_ptr=True,
             max_depth=L):
        p = [t.data_ptr() for t in lab]
        if null is not None:
            p[null] = None
        return lib.hk_search_value_labels(x.data_ptr(), *(o.data_ptr() for o in outs), max_labels,
                                          ctypes.addressof(count) if count_ptr else None, *p, B, n, dd, dtype,
                                          step_ops(True), max_depth, 100, 64, history, ws.data_ptr(), stream)
    assert call() == C.HK_OK
    for k in range(6):
        assert call(null=k) == C.HK_ERR_BAD_ARG, k
        assert call(null=k, max_labels=0) == C.HK_OK, k
    assert call(max_labels=-1) == C.HK_ERR_BAD_ARG
    assert call(count_ptr=False) == C.HK_ERR_BAD_ARG
    for h in (B - 1, 0, 1 << 31):
        assert call(history=h) == C.HK_ERR_BAD_ARG, h
    assert call(max_depth=0) == C.HK_ERR_BAD_ARG
    assert call(x=roots.float(), dtype=C.HK_DTYPE_F32) == C.HK_ERR_UNSUPPORTED
    for dd in (1, 7):  # the same bytes read as another dimension
        assert call(n=N * d // dd if N * d % dd == 0 else 1, dd=dd) == C.HK_ERR_UNSUPPORTED, dd
    count.value = -1
    assert call() == C.HK_OK and count.value >= 0
