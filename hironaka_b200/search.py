"""Game-tree search of a fixed host: how long can an adversarial agent make each game last?

The batched form of search_depth (hironaka/util/search.py), which explores every agent reply to one host strategy
recursively on one ListPoints game.  Here every root of a batch is searched at once, level by level on the GPU
(hk_search_depth, include/hironaka_b200.h), with explicit limits: a depth limit, a node budget per root and a
frontier capacity.  A root that hits a limit is a normal result, reported in `status`.

search_value (hk_search_value) answers the minimax question over the same tree with every host move: the fewest moves
the best host needs to end the game, whatever the agent replies.

search_depth_line and search_value_line return, with the same numbers, a line of play for each root: the agent's
longest line against the fixed host, and an optimal line of the best host with the agent's best replies.  play_line
replays lines into the states along them.  Along an optimal line the value drops by one per move, so its states with
value - t at move t are exact value labels.

search_value_labels returns far more such labels: every state the value search solved with a value of at least one,
under resolved roots and cut ones alike, with its exact value, every optimal host move (as HostActionEncoder ids) and
its rows.
"""
from __future__ import annotations

from typing import NamedTuple, Optional

import torch

from . import constants as C
from . import ops as _ops

STATUS_RESOLVED = C.HK_SEARCH_RESOLVED        # every line of play has ended
STATUS_MAX_DEPTH = C.HK_SEARCH_MAX_DEPTH      # states at level max_depth have not ended
STATUS_MAX_NODES = C.HK_SEARCH_MAX_NODES      # the next level would take the root past max_nodes
STATUS_CAPACITY = C.HK_SEARCH_CAPACITY        # the next level of the batch did not fit in the frontier capacity
STATUS_INT32_BOUND = C.HK_SEARCH_INT32_BOUND  # a state to expand has an entry >= 2^30 / d: its children would be inexact
STATUS_HISTORY = C.HK_SEARCH_HISTORY          # search_value: the next level did not fit in the batch's history

FRONTIER_BYTES = 1 << 28  # default capacity: one frontier fills 256 MiB
HISTORY_BYTES = 1 << 32   # search_value's default history: 4 GiB
HISTORY_NODE_BYTES = 14   # parent, solved round and group count (int32 each), group set and rank (one byte each)
DEPTH_LINE_NODE_BYTES = 7  # search_depth_line's history: parent (int32), set (16 bits, d <= 10), axis (one byte)
MAX_HISTORY = (1 << 31) - 1  # parents are int32 entries


class SearchResult(NamedTuple):
    depth: torch.Tensor   # [B] int32 height of the explored tree (a lower bound unless status == STATUS_RESOLVED)
    nodes: torch.Tensor   # [B] int64 states in the explored tree, root and ended leaves included
    status: torch.Tensor  # [B] int8 STATUS_*


def default_capacity(N: int, d: int) -> int:
    """Frontier capacity used when none is given: FRONTIER_BYTES / (N * d * 4) nodes."""
    return max(1, FRONTIER_BYTES // (N * d * 4))


def search_depth(points: torch.Tensor, host: str = "zeillinger", *, reposition: bool = True, max_depth: int = 64,
                 max_nodes: int = 1 << 16, capacity: Optional[int] = None) -> SearchResult:
    """For each root of `points` (int32 [B, N, d] on a CUDA device, taken as given: pass
    GameBatch(..., initial_filter=True).points for filtered roots), the longest game an agent can force against the
    fixed `host` ("zeillinger" or "all_coord"), found by trying every agent reply.

    A state with at most one live row has ended.  Any other state at level k is expanded: the host chooses its
    coordinate set S, and each axis in S (in increasing order) gives one child at level k + 1, the state after the JAX
    step (shift, reposition if `reposition`, Newton polytope).  Equal states are not merged.

    Limits: `max_depth` levels below the root; `max_nodes` states per root (the level that would pass it is not
    added); `capacity` states in one level of the whole batch (when the next level does not fit, roots are dropped from
    the highest index down until it does).  The default capacity is default_capacity(N, d) = 2^28 / (N * d * 4)
    states: the search keeps two frontiers of N * d * 4 bytes per state, so 512 MiB for both, plus a few words per state
    and per root.  Only STATUS_CAPACITY depends on the capacity and on the other roots of the batch.

    The call is synchronous (the number of states of each level is read back to size the next)."""
    if host not in ("zeillinger", "all_coord"):
        raise ValueError(f"host must be 'zeillinger' or 'all_coord'; got {host!r}")
    B, N, d = points.shape
    flags = C.HK_F_HOST_ZEILLINGER if host == "zeillinger" else C.HK_F_HOST_ALL_COORD
    step_ops = C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)
    cap = default_capacity(N, d) if capacity is None else int(capacity)
    depth, nodes, status = _ops.search_depth(points, flags=flags, ops=step_ops, max_depth=max_depth,
                                             max_nodes=max_nodes, capacity=cap)
    return SearchResult(depth, nodes, status)


class ValueResult(NamedTuple):
    value: torch.Tensor      # [B] int32 game value (a strict lower bound minus one unless status == STATUS_RESOLVED)
    best_mask: torch.Tensor  # [B] int32 the host's first move in an optimal line; 0 for an ended root, -1 unresolved
    nodes: torch.Tensor      # [B] int64 states in the explored tree, root and ended leaves included
    status: torch.Tensor     # [B] int8 STATUS_*


def default_history() -> int:
    """History used when none is given: HISTORY_BYTES / HISTORY_NODE_BYTES nodes."""
    return HISTORY_BYTES // HISTORY_NODE_BYTES


def search_value(points: torch.Tensor, *, reposition: bool = True, max_depth: int = 16, max_nodes: int = 1 << 22,
                 capacity: Optional[int] = None, history: Optional[int] = None) -> ValueResult:
    """For each root of `points` (int32 [B, N, d] on a CUDA device, 2 <= d <= 6, taken as given), the game value: the
    fewest moves the best host needs to end the game, whatever the agent replies.

    A state with at most one live row has ended (value 0).  Any other state is expanded into one child per host move
    and agent reply: every coordinate set S with |S| >= 2 in increasing bitmask order, and each axis of S in
    increasing order, the JAX step (shift, reposition if `reposition`, Newton polytope).  The children of one S form a
    group.  After each level L is built, its ended states are solved; a group is won when all its children are solved
    and a state is solved when its first group is won, up to the root.  A state at level l solved then has value L - l,
    and `best_mask` of a root is the smallest S won in that round.  Only open states with no solved ancestor are
    expanded.

    Limits, as search_depth's: `max_depth` levels, `max_nodes` states per root, `capacity` states in one level of the
    batch, the int32 bound; and `history`, the states of all levels of the batch, roots included, which the search keeps
    to walk up from solved states (STATUS_HISTORY when the next level would not fit; roots are dropped from the highest
    index down).  A root with another status has `value` = the last level checked, and its true value is larger.

    Memory: the defaults are capacity = default_capacity(N, d) = 2^28 / (N * d * 4) states, two frontiers of 256 MiB,
    and history = default_history() = 2^32 / 14 states at 14 bytes each, 4 GiB; plus a few words per frontier state
    and per root.  The call is synchronous."""
    B, N, d = points.shape
    step_ops = C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)
    cap = default_capacity(N, d) if capacity is None else int(capacity)
    hist = default_history() if history is None else int(history)
    value, best_mask, nodes, status = _ops.search_value(points, ops=step_ops, max_depth=max_depth, max_nodes=max_nodes,
                                                        capacity=cap, history=hist)
    return ValueResult(value, best_mask, nodes, status)


class DepthLine(NamedTuple):
    depth: torch.Tensor   # [B] int32 as SearchResult.depth: the length of the line
    nodes: torch.Tensor   # [B] int64 as SearchResult.nodes
    status: torch.Tensor  # [B] int8 STATUS_*
    mask: torch.Tensor    # [B, max_depth] int32 the host's set at each move; 0 past the line's end
    axis: torch.Tensor    # [B, max_depth] int32 the agent's axis at each move; -1 past the line's end


def default_depth_line_history() -> int:
    """search_depth_line's history when none is given: HISTORY_BYTES / DEPTH_LINE_NODE_BYTES states, at most
    MAX_HISTORY."""
    return min(HISTORY_BYTES // DEPTH_LINE_NODE_BYTES, MAX_HISTORY)


def search_depth_line(points: torch.Tensor, host: str = "zeillinger", *, reposition: bool = True, max_depth: int = 64,
                      max_nodes: int = 1 << 16, capacity: Optional[int] = None,
                      history: Optional[int] = None) -> DepthLine:
    """search_depth, and for each root the agent's worst line against the fixed `host`: depth[b] moves (mask, axis),
    each mask the host's choice on the state it is played on, the axes the lexicographically smallest sequence among
    the lines that reach level depth[b] of the explored tree.  For a resolved root this is the smallest of the longest
    games, and it ends at an ended state; for a cut root it is the smallest line to the deepest level explored, whose
    end need not have ended.

    The search keeps every state of every level in a history of DEPTH_LINE_NODE_BYTES = 7 bytes per state (parent
    entry int32, set 16 bits, axis one byte), so `history` is one more limit: the states of all levels of the batch,
    roots included, at most 2^31 - 1 because parents are int32 entries.  The default, default_depth_line_history(), is
    2^32 / 7 states, 4 GiB.  A root cut by it gets STATUS_HISTORY; the cuts apply in the order of search_value (int32
    bound, node budget, capacity, history, the last two from the highest root index down).  With a history large enough
    for the whole search, depth, nodes and status equal search_depth's.  Synchronous."""
    if host not in ("zeillinger", "all_coord"):
        raise ValueError(f"host must be 'zeillinger' or 'all_coord'; got {host!r}")
    B, N, d = points.shape
    flags = C.HK_F_HOST_ZEILLINGER if host == "zeillinger" else C.HK_F_HOST_ALL_COORD
    step_ops = C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)
    cap = default_capacity(N, d) if capacity is None else int(capacity)
    hist = default_depth_line_history() if history is None else int(history)
    return DepthLine(*_ops.search_depth_line(points, flags=flags, ops=step_ops, max_depth=max_depth,
                                             max_nodes=max_nodes, capacity=cap, history=hist))


class ValueLine(NamedTuple):
    value: torch.Tensor      # [B] int32 as ValueResult.value: the length of the line of a resolved root
    best_mask: torch.Tensor  # [B] int32 as ValueResult.best_mask: the line's first mask
    nodes: torch.Tensor      # [B] int64
    status: torch.Tensor     # [B] int8 STATUS_*
    mask: torch.Tensor       # [B, max_depth] int32 the host's set at each move; 0 past the line's end
    axis: torch.Tensor       # [B, max_depth] int32 the agent's axis at each move; -1 past the line's end


def search_value_line(points: torch.Tensor, *, reposition: bool = True, max_depth: int = 16, max_nodes: int = 1 << 22,
                      capacity: Optional[int] = None, history: Optional[int] = None) -> ValueLine:
    """search_value, and for each resolved root of value v > 0 an optimal line of v moves.  From a state of value
    u > 0 the host plays the smallest S whose children all have value <= u - 1 (best_mask at the root), and the agent
    the smallest axis of S whose child has value exactly u - 1; the line ends at an ended state.  Roots that had ended
    and roots with another status than STATUS_RESOLVED get an empty line.  The line is read from the search's own
    history: the memory and limits are search_value's.  Synchronous."""
    B, N, d = points.shape
    step_ops = C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)
    cap = default_capacity(N, d) if capacity is None else int(capacity)
    hist = default_history() if history is None else int(history)
    return ValueLine(*_ops.search_value_line(points, ops=step_ops, max_depth=max_depth, max_nodes=max_nodes,
                                             capacity=cap, history=hist))


def play_line(points: torch.Tensor, mask: torch.Tensor, axis: torch.Tensor, *, reposition: bool = True) -> torch.Tensor:
    """The states along lines: int32 [B, L + 1, N, d], state t after the first t moves of mask / axis ([B, L] each, as
    search_depth_line and search_value_line return them), each move the searches' step (shift, reposition if
    `reposition`, Newton polytope).  Past a line's end (axis -1) the state repeats: such a game is not stepped, since a
    step with axis -1 would, under reposition, move a lone point to the origin.  One ops.step launch per move."""
    B, N, d = points.shape
    L = mask.shape[1]
    if mask.shape != (B, L) or axis.shape != (B, L):
        raise ValueError(f"mask and axis must both be [{B}, L]; got {tuple(mask.shape)} and {tuple(axis.shape)}")
    step_ops = C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)
    mask = mask.to(points.device, torch.int32)
    axis = axis.to(points.device, torch.int32)
    out = torch.empty((B, L + 1, N, d), dtype=points.dtype, device=points.device)
    out[:, 0] = points
    for t in range(L):
        out[:, t + 1] = out[:, t]
        idx = torch.nonzero(axis[:, t] >= 0).flatten()
        if len(idx):
            out[idx, t + 1] = _ops.step(out[idx, t].contiguous(), mask[idx, t], axis[idx, t], ops=step_ops).state
    return out


class ValueLabels(NamedTuple):
    value: torch.Tensor        # [B] int32 as ValueResult
    best_mask: torch.Tensor    # [B] int32
    nodes: torch.Tensor        # [B] int64
    status: torch.Tensor       # [B] int8 STATUS_*
    count: int                 # labels found; the tensors below hold the first K = min(count, max_labels)
    root: torch.Tensor         # [K] int32 the root the state lies under
    level: torch.Tensor        # [K] int32 moves from the root (non-decreasing over the labels)
    label_value: torch.Tensor  # [K] int32 the state's exact value, >= 1
    optimal: torch.Tensor      # [K, 2^d - d - 1] bool column g: the host move of HostActionEncoder id g is optimal
    mask: torch.Tensor         # [K, max_depth] int32 the host's set at each move from the root; 0 past the level
    axis: torch.Tensor         # [K, max_depth] int32 the agent's axis at each move from the root; -1 past the level
    state: torch.Tensor        # [K, N, d] int32 the state


def search_value_labels(points: torch.Tensor, *, reposition: bool = True, max_depth: int = 16,
                        max_nodes: int = 1 << 22, capacity: Optional[int] = None, history: Optional[int] = None,
                        max_labels: int = 1 << 22) -> ValueLabels:
    """search_value, and every state it solved with a value of at least one, as training labels.

    A state of level l solved in round R has the exact value R - l: once a state is solved its subtree stops growing,
    so nothing below it is solved later.  This holds under every root, whatever its status, so roots cut by a limit
    contribute labels too.  The optimal host moves of such a state are exactly its groups whose children were all
    solved; column g of `optimal` is the set of HostActionEncoder id g (the sets with |S| >= 2 in increasing bitmask
    order, the order of host_action.action_masks).  Each label also has its root, its level, its path from the root
    (mask, axis) and its rows, replayed from the root with the searches' step.

    Labels are in the order of the search's history: level non-decreasing and, within a level, root non-decreasing.
    `count` is the number found; the first min(count, max_labels) are returned.  Equal states reached by different
    paths are separate labels.  Memory and limits are search_value's, plus 12 bytes per 256 history states for the
    label scan and the outputs (about 4 * (2 * max_depth + 4) bytes per label and N * d * 4 for its rows).
    Synchronous."""
    B, N, d = points.shape
    step_ops = C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)
    cap = default_capacity(N, d) if capacity is None else int(capacity)
    hist = default_history() if history is None else int(history)
    (value, best_mask, nodes, status, count, root, level, label_value, optimal, mask,
     axis) = _ops.search_value_labels(points, ops=step_ops, max_depth=max_depth, max_nodes=max_nodes, capacity=cap,
                                      history=hist, max_labels=max_labels)
    ids = torch.arange((1 << d) - d - 1, dtype=torch.int64, device=points.device)
    optimal = ((optimal[:, None] >> ids) & 1).bool()
    state = points[root.long()]
    # the labels with level > t are a suffix: one step per level advances exactly them
    starts = torch.searchsorted(level, torch.arange(1, max_depth + 1, dtype=torch.int32, device=points.device),
                                right=False).tolist()
    for t, start in enumerate(starts):
        if start == len(level):
            break
        _ops.step(state[start:], mask[start:, t], axis[start:, t], ops=step_ops)
    return ValueLabels(value, best_mask, nodes, status, count, root, level, label_value, optimal, mask, axis, state)
