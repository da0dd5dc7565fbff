"""Tensor-level entry to the C-ABI: torch CUDA tensors in, raw device pointers out.

PyTorch is plumbing here (device memory, streams); every game operation is a launch of the
hand-written kernels behind include/hironaka_b200.h.  Nothing in this module computes on the
CPU or through torch ops, and nothing falls back: a CPU tensor or a missing library raises.
"""
from __future__ import annotations

import ctypes
from typing import List, NamedTuple, Optional, Sequence, Union

import torch

from . import constants as C
from ._lib import HironakaB200Error, check, lib

_DT = {torch.int32: C.HK_DTYPE_I32, torch.float32: C.HK_DTYPE_F32}
_PACK_DT = {torch.int32: 0, torch.float32: 1, torch.int64: 2, torch.uint8: 3, torch.bool: 3}


class StepResult(NamedTuple):
    state: Optional[torch.Tensor]       # [B,N,d] new state (the input tensor itself when in place)
    done: Optional[torch.Tensor]        # [B] bool
    reward: Optional[torch.Tensor]      # [B] float32
    num_points: Optional[torch.Tensor]  # [B] int32
    obs: Optional[torch.Tensor]         # [B, N*d (+d)] float32


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require_state(state: torch.Tensor) -> int:
    if not isinstance(state, torch.Tensor):
        raise TypeError(f"state must be a torch.Tensor, got {type(state)}")
    if not state.is_cuda:
        raise HironakaB200Error("hironaka_b200 has no CPU path: the point tensor must live on a CUDA device")
    if state.dim() != 3:
        raise ValueError(f"state must be [B, N, d]; got shape {tuple(state.shape)}")
    if state.dtype not in _DT:
        raise TypeError(f"state dtype must be int32 or float32; got {state.dtype}")
    if not state.is_contiguous():
        raise ValueError("state must be contiguous")
    return _DT[state.dtype]


def _as_i32(x, B: int, device, name: str) -> torch.Tensor:
    if isinstance(x, torch.Tensor):
        t = x
        if t.device != device:
            t = t.to(device)
        if t.dtype != torch.int32:
            t = t.to(torch.int32)
    else:
        t = torch.as_tensor(x, dtype=torch.int32, device=device)
    if t.shape != (B,):
        raise ValueError(f"{name} must have shape ({B},); got {tuple(t.shape)}")
    return t.contiguous()


def coords_to_mask(coords: Union[torch.Tensor, Sequence[Sequence[int]]], dimension: int, device) -> torch.Tensor:
    """Coordinate sets -> int32 bitmasks (bit k <=> coordinate k).

    Accepts what the reference's shift accepts (hironaka/src/_torch_ops.py:54-72): a list of
    index lists, e.g. [[1, 2], [0, 2, 3]], or a [B, d] multi-binary tensor of any dtype.  The
    two are NOT the same encoding: [[1, 2]] == Tensor([[0, 1, 1]]) in dimension 3."""
    if isinstance(coords, (list, tuple)):
        masks = []
        for c in coords:
            m = 0
            for k in c:
                if not 0 <= int(k) < dimension:
                    raise ValueError(f"coordinate {k} out of range for dimension {dimension}")
                m |= 1 << int(k)
            masks.append(m)
        return torch.tensor(masks, dtype=torch.int32, device=device)
    if not isinstance(coords, torch.Tensor):
        raise Exception(f"unsupported input type for coord. Got {type(coords)}.")
    if coords.dim() != 2 or coords.shape[1] != dimension:
        raise ValueError(f"coords must be [B, {dimension}]; got {tuple(coords.shape)}")
    if coords.is_cuda:  # one launch of hk_pack_coords
        code = _PACK_DT.get(coords.dtype)
        if code is None:
            coords, code = coords.to(torch.float32), 1
        coords = coords.contiguous()
        mask = torch.empty(coords.shape[0], dtype=torch.int32, device=coords.device)
        with torch.cuda.device(coords.device):
            rc = lib().hk_pack_coords(coords.data_ptr(), code, mask.data_ptr(), coords.shape[0], dimension,
                                      torch.cuda.current_stream(coords.device).cuda_stream)
        check(rc, "hk_pack_coords")
        return mask if mask.device == torch.device(device) else mask.to(device)
    weights = (1 << torch.arange(dimension, device=coords.device, dtype=torch.int32))  # host-side lists / CPU tensors
    return ((coords > 0.5).to(torch.int32) * weights).sum(1, dtype=torch.int32).to(device)


def step(state: torch.Tensor, host_action=None, axis=None, *, ops: int, flags: int = 0,
         padding_value: float = -1.0, inplace: bool = True, out: Optional[torch.Tensor] = None,
         write_state: bool = True, want_done: bool = False, want_reward: bool = False,
         want_num_points: bool = False, want_obs: bool = False, obs_coord=None,
         exceed_flag: Optional[torch.Tensor] = None, value_threshold: float = 1e8,
         census: Optional[torch.Tensor] = None, done_count: Optional[torch.Tensor] = None,
         done_bits: Optional[torch.Tensor] = None) -> StepResult:
    """One fused game-step (hk_step).  `host_action` is an int32 [B] tensor of coordinate
    bitmasks, or discrete ids when HK_F_ACT_DISCRETE is set; `axis` an int [B] tensor.

    `census` (uint8 [B], in/out; see `new_census`) selects hk_step_census: the in-place step whose work
    follows the games still in play (games at rest are not read, the others are ordered by live count).
    Zero the bytes of any game you rewrite between calls.  `done_count` (int32 [1]) is incremented by the
    number of finished games; `done_bits` (int32 [ceil(B/32)]) receives the done flags as a bit mask."""
    dt = _require_state(state)
    B, N, d = state.shape
    dev = state.device
    if write_state:
        if inplace:
            dst = state
        else:
            dst = out if out is not None else torch.empty_like(state)
            if dst.shape != state.shape or dst.dtype != state.dtype or not dst.is_contiguous() or dst.device != dev:
                raise ValueError("out must match state in shape, dtype, device and be contiguous")
    else:
        dst = None
    ha = ax = None
    if ops & C.HK_OP_SHIFT:
        host_fixed = flags & (C.HK_F_HOST_ALL_COORD | C.HK_F_HOST_ZEILLINGER)
        agent_fixed = flags & (C.HK_F_AGENT_FIRST | C.HK_F_AGENT_LAST)
        if (host_action is None and not host_fixed) or (axis is None and not agent_fixed):
            raise ValueError("shift needs host_action and axis (or a fixed-player flag for the missing one)")
        ha = None if host_fixed else _as_i32(host_action, B, dev, "host_action")
        ax = None if agent_fixed else _as_i32(axis, B, dev, "axis")
    done = torch.empty(B, dtype=torch.uint8, device=dev) if want_done else None
    reward = torch.empty(B, dtype=torch.float32, device=dev) if want_reward else None
    npts = torch.empty(B, dtype=torch.int32, device=dev) if want_num_points else None
    oc = None
    obs = None
    if want_obs:
        if obs_coord is not None:
            oc = _as_i32(obs_coord, B, dev, "obs_coord")
        obs = torch.empty((B, N * d + (d if oc is not None else 0)), dtype=torch.float32, device=dev)
    if exceed_flag is not None and (exceed_flag.dtype != torch.int32 or exceed_flag.device != dev):
        raise ValueError("exceed_flag must be an int32 tensor on the state's device")
    if done_bits is not None and (census is None or done_bits.dtype != torch.int32 or done_bits.numel() != (B + 31) // 32
                                  or done_bits.device != dev):
        raise ValueError("done_bits needs a census and must be an int32 [ceil(B/32)] tensor on the state's device")
    if census is not None:
        need = lib().hk_census_bytes(B, N, d)
        if census.dtype != torch.uint8 or census.numel() < need or census.device != dev or not census.is_contiguous():
            raise ValueError(f"census must be a contiguous uint8 tensor of {need} bytes (new_census) on the state's device")
        if not (write_state and inplace):
            raise ValueError("the census step runs in place")
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            if want_obs:  # thread-per-game shapes, sorted observation modes
                rc = lib().hk_step_census_obs(_ptr(state), _ptr(ha), _ptr(ax), _ptr(done), _ptr(done_bits), _ptr(reward),
                                              _ptr(npts), _ptr(obs), _ptr(oc), _ptr(census), _ptr(done_count), _ptr(exceed_flag),
                                              B, N, d, dt, ops, flags, float(padding_value), float(value_threshold), stream)
            else:
                rc = lib().hk_step_census(_ptr(state), _ptr(ha), _ptr(ax), _ptr(done), _ptr(done_bits), _ptr(reward), _ptr(npts),
                                          _ptr(census), _ptr(done_count), _ptr(exceed_flag), B, N, d, dt, ops, flags,
                                          float(padding_value), float(value_threshold), stream)
        check(rc, "hk_step_census")
        return StepResult(dst, None if done is None else done.view(torch.bool), reward, npts, obs)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib().hk_step(_ptr(state), _ptr(dst), _ptr(ha), _ptr(ax), _ptr(done), _ptr(reward), _ptr(npts),
                           _ptr(obs), _ptr(oc), _ptr(exceed_flag), B, N, d, dt, ops, flags, float(padding_value),
                           float(value_threshold), stream)
    check(rc, "hk_step")
    return StepResult(dst, None if done is None else done.view(torch.bool), reward, npts, obs)


def new_census(state: torch.Tensor) -> torch.Tensor:
    """A zeroed census for `state` (every game unknown); pass it to `step(..., census=)`.  uint8
    [hk_census_bytes(B, N, d)]: byte g describes game g (zero it when you rewrite the game); large padded shapes
    append a 64-bit live mask per game."""
    B, N, d = state.shape
    return torch.zeros(lib().hk_census_bytes(B, N, d), dtype=torch.uint8, device=state.device)


def rollout(state: torch.Tensor, host_actions: Optional[torch.Tensor], axes: Optional[torch.Tensor], *, ops: int,
            flags: int = 0, padding_value: float = -1.0, inplace: bool = True, want_done: bool = False,
            want_reward: bool = False, want_done_count: bool = True, want_length: bool = False,
            steps: Optional[int] = None, value_threshold: Optional[float] = None, stop_at_threshold: bool = False,
            over_step: Optional[torch.Tensor] = None):
    """T fused steps in one launch (hk_rollout): host_actions / axes are int32 [T, B]; either may be
    None when the matching fixed-player flag (HK_F_HOST_* / HK_F_AGENT_*) is set, in which case
    `steps` gives T if both are None.  With `value_threshold` the rollout runs through hk_rollout_threshold:
    `over_step` (int32 [B], written when given) receives each game's crossing step, and `stop_at_threshold` stops
    the games that cross."""
    _require_state(state)
    B = state.shape[0]
    host_fixed = flags & (C.HK_F_HOST_ALL_COORD | C.HK_F_HOST_ZEILLINGER)
    agent_fixed = flags & (C.HK_F_AGENT_FIRST | C.HK_F_AGENT_LAST)
    if (host_actions is None and not host_fixed) or (axes is None and not agent_fixed):
        raise ValueError("rollout needs host_actions and axes (or a fixed-player flag for the missing one)")
    shapes = [t.shape for t in (None if host_fixed else host_actions, None if agent_fixed else axes) if t is not None]
    if shapes:
        if any(len(sh) != 2 or sh[1] != B for sh in shapes) or len(set(shapes)) != 1:
            raise ValueError("host_actions and axes must be [T, B]")
        T = shapes[0][0]
    else:
        if not steps:
            raise ValueError("steps is required when both players are fixed")
        T = int(steps)
    tr = _rollout(state, None if host_fixed else host_actions, None if agent_fixed else axes, T, "hk_rollout", ops=ops,
                  flags=flags, padding_value=padding_value, inplace=inplace, want_done=want_done, want_reward=want_reward,
                  want_done_count=want_done_count, want_length=want_length, value_threshold=value_threshold,
                  stop_at_threshold=stop_at_threshold, over_step=over_step)
    return tr.state, tr.done, tr.reward, tr.done_count, tr.length


def rollout_random(state: torch.Tensor, steps: int, seed: int, *, ops: int, flags: int = 0, host_actions=None, axes=None,
                   step_offset: int = 0, padding_value: float = -1.0, inplace: bool = True, want_done: bool = False,
                   want_reward: bool = False, want_length: bool = False, value_threshold: Optional[float] = None,
                   stop_at_threshold: bool = False, over_step: Optional[torch.Tensor] = None):
    """`steps` fused steps with random players drawn INSIDE the kernel (hk_rollout_seeded): no [T, B] action streams.
    `flags` carries HK_F_HOST_RANDOM and / or HK_F_AGENT_RANDOM; the other player comes from its [T, B] stream or a
    fixed-player flag.  Philox4x32-10 keyed by `seed`, counter (game, step_offset + t): see `random_actions`.
    `value_threshold`, `stop_at_threshold`, `over_step`: as in `rollout` (hk_rollout_threshold)."""
    _require_state(state)
    if value_threshold is not None and not flags & (C.HK_F_HOST_RANDOM | C.HK_F_AGENT_RANDOM):
        raise ValueError("rollout_random needs HK_F_HOST_RANDOM and / or HK_F_AGENT_RANDOM")
    tr = _rollout(state, host_actions, axes, int(steps), "hk_rollout_seeded", ops=ops, flags=flags,
                  padding_value=padding_value, inplace=inplace, want_done=want_done, want_reward=want_reward,
                  want_length=want_length, seed=seed, step_offset=step_offset, value_threshold=value_threshold,
                  stop_at_threshold=stop_at_threshold, over_step=over_step)
    return tr.state, tr.done, tr.reward, tr.done_count, tr.length


class Trajectory(NamedTuple):
    state: torch.Tensor                  # [B,N,d] state after the last step (the input tensor itself when in place)
    obs: Optional[torch.Tensor]          # [T, B, N*d (+d)] float32: features of the state BEFORE each step
    host_mask: Optional[torch.Tensor]    # [T, B] int32 coordinate bitmask each step's shift used
    axis: Optional[torch.Tensor]         # [T, B] int32 axis each step's shift used
    done: Optional[torch.Tensor]         # [T, B] bool
    reward: Optional[torch.Tensor]       # [T, B] float32
    done_count: Optional[torch.Tensor]   # [T] int32 finished games after each step
    length: Optional[torch.Tensor]       # [B] int32


def rollout_record(state: torch.Tensor, steps: Optional[int] = None, host_actions: Optional[torch.Tensor] = None,
                   axes: Optional[torch.Tensor] = None, *, ops: int, flags: int = 0, seed: int = 0, step_offset: int = 0,
                   want_obs: bool = True, agent_obs: bool = False, want_actions: bool = True, want_done: bool = True,
                   want_reward: bool = True, want_length: bool = True, inplace: bool = True,
                   padding_value: float = -1.0, value_threshold: Optional[float] = None, stop_at_threshold: bool = False,
                   over_step: Optional[torch.Tensor] = None) -> Trajectory:
    """T fused steps in one launch that also record the trajectory (hk_rollout_record): obs[t] are the features of the
    state the players see at step t (the observation flags of `features`), host_mask / axis what step t played, as
    bitmasks and axes (replayed through `rollout` without HK_F_ACT_DISCRETE and the player flags they give the same
    rollout).  `agent_obs` appends step t's host coordinates to obs[t] as d floats 0/1.  The players are [T, B] int32
    streams, fixed-player flags, or the in-kernel random players (HK_F_HOST_RANDOM / HK_F_AGENT_RANDOM, keyed by `seed`
    and `step_offset`); `steps` gives T when no stream does.  The features after the last step are
    features(trajectory.state).  `value_threshold`, `stop_at_threshold`, `over_step`: as in `rollout`
    (hk_rollout_threshold); a stopped game records the features of its frozen state, host_mask 0 and axis -1."""
    _require_state(state)
    B = state.shape[0]
    streams = [t for t in (host_actions, axes) if t is not None]
    if any(t.dim() != 2 or t.shape[1] != B for t in streams) or len({tuple(t.shape) for t in streams}) > 1:
        raise ValueError("host_actions and axes must be [T, B]")
    T = int(steps) if steps is not None else (streams[0].shape[0] if streams else 0)
    if T < 1 or (streams and streams[0].shape[0] != T):
        raise ValueError("steps must be >= 1 and match the action streams")
    if agent_obs and not want_obs:
        raise ValueError("agent_obs needs want_obs")
    return _rollout(state, host_actions, axes, T, "hk_rollout_record", ops=ops, flags=flags, padding_value=padding_value,
                    inplace=inplace, want_done=want_done, want_reward=want_reward, want_length=want_length, seed=seed,
                    step_offset=step_offset, want_obs=want_obs, agent_obs=agent_obs, want_actions=want_actions,
                    value_threshold=value_threshold, stop_at_threshold=stop_at_threshold, over_step=over_step)


def _rollout(state, host_actions, axes, T, entry, *, ops, flags, padding_value, inplace, want_done, want_reward,
             want_length, want_done_count=True, seed=0, step_offset=0, want_obs=False, agent_obs=False,
             want_actions=False, value_threshold=None, stop_at_threshold=False, over_step=None) -> Trajectory:
    """A one-launch rollout of T steps on the players' [T, B] streams (None: no stream): allocates the outputs the
    caller wants and launches `entry` (hk_rollout, hk_rollout_seeded or hk_rollout_record), or hk_rollout_threshold
    when `value_threshold` is given; `over_step` is the caller's int32 [B]."""
    dt = _DT[state.dtype]
    B, N, d = state.shape
    dev = state.device
    ha = None if host_actions is None else host_actions.to(device=dev, dtype=torch.int32).contiguous()
    ax = None if axes is None else axes.to(device=dev, dtype=torch.int32).contiguous()
    dst = state if inplace else torch.empty_like(state)
    obs = torch.empty((T, B, N * d + (d if agent_obs else 0)), dtype=torch.float32, device=dev) if want_obs else None
    hmask = torch.empty((T, B), dtype=torch.int32, device=dev) if want_actions else None
    axis = torch.empty((T, B), dtype=torch.int32, device=dev) if want_actions else None
    done = torch.empty((T, B), dtype=torch.uint8, device=dev) if want_done else None
    reward = torch.empty((T, B), dtype=torch.float32, device=dev) if want_reward else None
    dcount = torch.zeros(T, dtype=torch.int32, device=dev) if want_done_count else None
    length = torch.empty(B, dtype=torch.int32, device=dev) if want_length else None
    if value_threshold is not None:
        entry = "hk_rollout_threshold"
        if over_step is not None and (over_step.dtype != torch.int32 or tuple(over_step.shape) != (B,) or
                                      over_step.device != dev or not over_step.is_contiguous()):
            raise ValueError("over_step must be a contiguous int32 [B] tensor on the state's device")
    seed = int(seed) & (2 ** 64 - 1)
    pad = float(padding_value)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        if entry == "hk_rollout_threshold":
            rc = lib().hk_rollout_threshold(_ptr(state), _ptr(dst), _ptr(ha), _ptr(ax), _ptr(obs), 1 if agent_obs else 0,
                                            _ptr(hmask), _ptr(axis), _ptr(done), _ptr(reward), _ptr(dcount), _ptr(length), B,
                                            N, d, T, dt, ops, flags, pad, seed, int(step_offset), float(value_threshold),
                                            1 if stop_at_threshold else 0, _ptr(over_step), stream)
        elif entry == "hk_rollout_record":
            rc = lib().hk_rollout_record(_ptr(state), _ptr(dst), _ptr(ha), _ptr(ax), _ptr(obs), 1 if agent_obs else 0,
                                         _ptr(hmask), _ptr(axis), _ptr(done), _ptr(reward), _ptr(dcount), _ptr(length), B, N,
                                         d, T, dt, ops, flags, pad, seed, int(step_offset), stream)
        elif entry == "hk_rollout_seeded":
            rc = lib().hk_rollout_seeded(_ptr(state), _ptr(dst), _ptr(ha), _ptr(ax), _ptr(done), _ptr(reward), _ptr(dcount),
                                         _ptr(length), B, N, d, T, dt, ops, flags, pad, seed, int(step_offset), stream)
        else:
            rc = lib().hk_rollout(_ptr(state), _ptr(dst), _ptr(ha), _ptr(ax), _ptr(done), _ptr(reward), _ptr(dcount),
                                  _ptr(length), B, N, d, T, dt, ops, flags, pad, stream)
    check(rc, entry)
    return Trajectory(dst, obs, hmask, axis, None if done is None else done.view(torch.bool), reward, dcount, length)


def random_actions(B: int, d: int, steps: int, seed: int, step_offset: int = 0, device="cuda"):
    """The action streams the in-kernel random players draw, written out: (host ids [T, B], axes [T, B]) int32."""
    dev = torch.device(device)
    ha = torch.empty((steps, B), dtype=torch.int32, device=dev)
    ax = torch.empty((steps, B), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib().hk_random_actions(_ptr(ha), _ptr(ax), B, d, steps, int(seed) & (2 ** 64 - 1), int(step_offset),
                                     torch.cuda.current_stream(dev).cuda_stream)
    check(rc, "hk_random_actions")
    return ha, ax


def features(state: torch.Tensor, *, flags: int = 0, obs_coord=None, padding_value: float = -1.0) -> torch.Tensor:
    """Observation features [B, N*d (+d)] float32 of a state (hk_features)."""
    dt = _require_state(state)
    B, N, d = state.shape
    dev = state.device
    oc = None if obs_coord is None else _as_i32(obs_coord, B, dev, "obs_coord")
    obs = torch.empty((B, N * d + (d if oc is not None else 0)), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib().hk_features(_ptr(state), _ptr(obs), _ptr(oc), B, N, d, dt, flags, float(padding_value), stream)
    check(rc, "hk_features")
    return obs


def dones(state: torch.Tensor, want_num_points: bool = False):
    """(done [B] bool, num_points [B] int32 | None) of a state (hk_dones)."""
    dt = _require_state(state)
    B, N, d = state.shape
    dev = state.device
    done = torch.empty(B, dtype=torch.uint8, device=dev)
    npts = torch.empty(B, dtype=torch.int32, device=dev) if want_num_points else None
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib().hk_dones(_ptr(state), _ptr(done), _ptr(npts), B, N, d, dt, stream)
    check(rc, "hk_dones")
    return done.view(torch.bool), npts


def overflow(state: torch.Tensor, value_threshold: float, strict: bool = False) -> torch.Tensor:
    """Per-game overflow flags [B] bool: some entry >= value_threshold (> when strict) (hk_overflow)."""
    dt = _require_state(state)
    B, N, d = state.shape
    out = torch.empty(B, dtype=torch.uint8, device=state.device)
    with torch.cuda.device(state.device):
        stream = torch.cuda.current_stream(state.device).cuda_stream
        rc = lib().hk_overflow(_ptr(state), _ptr(out), B, N, d, dt, float(value_threshold), 1 if strict else 0, stream)
    check(rc, "hk_overflow")
    return out.view(torch.bool)


def host_policy(state: torch.Tensor, host: str, padding_value: float = -1.0) -> torch.Tensor:
    """Coordinate set a fixed host ("zeillinger" | "all_coord") would choose on each game, as an int32
    bitmask [B] (hk_host_policy); nothing is moved.  Pairs are scanned in slot order, so a state kept in
    ListPoints order reproduces hironaka/host.py:50-92."""
    dt = _require_state(state)
    flag = {"zeillinger": C.HK_F_HOST_ZEILLINGER, "all_coord": C.HK_F_HOST_ALL_COORD}[host]
    B, N, d = state.shape
    mask = torch.empty(B, dtype=torch.int32, device=state.device)
    with torch.cuda.device(state.device):
        stream = torch.cuda.current_stream(state.device).cuda_stream
        rc = lib().hk_host_policy(_ptr(state), _ptr(mask), B, N, d, dt, flag, float(padding_value), stream)
    check(rc, "hk_host_policy")
    return mask


def _workspace(workspace: Optional[torch.Tensor], need: int, dev) -> torch.Tensor:
    if workspace is None:
        return torch.empty(max(need, 1), dtype=torch.uint8, device=dev)
    if workspace.dtype != torch.uint8 or workspace.numel() < need or workspace.device != dev:
        raise ValueError(f"workspace must be a uint8 tensor of at least {need} bytes on the roots' device")
    return workspace


def search_workspace_bytes(B: int, N: int, d: int, capacity: int) -> int:
    """Bytes of device workspace `search_depth` needs (hk_search_workspace_bytes)."""
    return int(lib().hk_search_workspace_bytes(B, N, d, capacity))


def search_depth(roots: torch.Tensor, *, flags: int, ops: int, max_depth: int, max_nodes: int, capacity: int,
                 workspace: Optional[torch.Tensor] = None):
    """Game-tree search of a fixed host against every agent reply (hk_search_depth): (depth [B] int32, nodes [B]
    int64, status [B] int8).  `flags` is HK_F_HOST_ZEILLINGER or HK_F_HOST_ALL_COORD, `ops` HK_OP_SHIFT | HK_OP_NEWTON
    (| HK_OP_REPOSITION).  `workspace` is a uint8 tensor of at least search_workspace_bytes(B, N, d, capacity) bytes on
    the roots' device (allocated here when None).  Synchronous: the call returns when the search is over."""
    dt = _require_state(roots)
    B, N, d = roots.shape
    dev = roots.device
    workspace = _workspace(workspace, search_workspace_bytes(B, N, d, capacity), dev)
    depth = torch.empty(B, dtype=torch.int32, device=dev)
    nodes = torch.empty(B, dtype=torch.int64, device=dev)
    status = torch.empty(B, dtype=torch.int8, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib().hk_search_depth(_ptr(roots), _ptr(depth), _ptr(nodes), _ptr(status), B, N, d, dt, ops, flags,
                                   int(max_depth), int(max_nodes), int(capacity), _ptr(workspace), stream)
    check(rc, "hk_search_depth")
    return depth, nodes, status


def search_value_workspace_bytes(B: int, N: int, d: int, capacity: int, history: int) -> int:
    """Bytes of device workspace `search_value` needs (hk_search_value_workspace_bytes; 0 for refused arguments)."""
    return int(lib().hk_search_value_workspace_bytes(B, N, d, capacity, history))


def search_value(roots: torch.Tensor, *, ops: int, max_depth: int, max_nodes: int, capacity: int, history: int,
                 workspace: Optional[torch.Tensor] = None):
    """Game value by minimax search over the host's choices (hk_search_value): (value [B] int32, best_mask [B] int32,
    nodes [B] int64, status [B] int8).  `ops` is HK_OP_SHIFT | HK_OP_NEWTON (| HK_OP_REPOSITION).  `workspace` is a
    uint8 tensor of at least search_value_workspace_bytes(B, N, d, capacity, history) bytes on the roots' device
    (allocated here when None).  Synchronous: the call returns when the search is over."""
    dt = _require_state(roots)
    B, N, d = roots.shape
    dev = roots.device
    workspace = _workspace(workspace, search_value_workspace_bytes(B, N, d, capacity, history), dev)
    value = torch.empty(B, dtype=torch.int32, device=dev)
    best_mask = torch.empty(B, dtype=torch.int32, device=dev)
    nodes = torch.empty(B, dtype=torch.int64, device=dev)
    status = torch.empty(B, dtype=torch.int8, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib().hk_search_value(_ptr(roots), _ptr(value), _ptr(best_mask), _ptr(nodes), _ptr(status), B, N, d, dt,
                                   ops, int(max_depth), int(max_nodes), int(capacity), int(history), _ptr(workspace),
                                   stream)
    check(rc, "hk_search_value")
    return value, best_mask, nodes, status


def search_depth_line_workspace_bytes(B: int, N: int, d: int, capacity: int, history: int) -> int:
    """Bytes of device workspace `search_depth_line` needs (hk_search_depth_line_workspace_bytes; 0 for refused
    arguments)."""
    return int(lib().hk_search_depth_line_workspace_bytes(B, N, d, capacity, history))


def search_depth_line(roots: torch.Tensor, *, flags: int, ops: int, max_depth: int, max_nodes: int, capacity: int,
                      history: int, workspace: Optional[torch.Tensor] = None):
    """search_depth with the worst line against the fixed host (hk_search_depth_line): (depth [B] int32, nodes [B]
    int64, status [B] int8, line_mask [B, max_depth] int32, line_axis [B, max_depth] int32).  `workspace` is a uint8
    tensor of at least search_depth_line_workspace_bytes(B, N, d, capacity, history) bytes on the roots' device
    (allocated here when None).  Synchronous."""
    dt = _require_state(roots)
    B, N, d = roots.shape
    dev = roots.device
    workspace = _workspace(workspace, search_depth_line_workspace_bytes(B, N, d, capacity, history), dev)
    depth = torch.empty(B, dtype=torch.int32, device=dev)
    nodes = torch.empty(B, dtype=torch.int64, device=dev)
    status = torch.empty(B, dtype=torch.int8, device=dev)
    line_mask = torch.empty((B, max(int(max_depth), 0)), dtype=torch.int32, device=dev)
    line_axis = torch.empty_like(line_mask)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib().hk_search_depth_line(_ptr(roots), _ptr(depth), _ptr(nodes), _ptr(status), _ptr(line_mask),
                                        _ptr(line_axis), B, N, d, dt, ops, flags, int(max_depth), int(max_nodes),
                                        int(capacity), int(history), _ptr(workspace), stream)
    check(rc, "hk_search_depth_line")
    return depth, nodes, status, line_mask, line_axis


def search_value_line(roots: torch.Tensor, *, ops: int, max_depth: int, max_nodes: int, capacity: int, history: int,
                      workspace: Optional[torch.Tensor] = None):
    """search_value with an optimal line of every resolved root (hk_search_value_line): (value [B] int32, best_mask [B]
    int32, nodes [B] int64, status [B] int8, line_mask [B, max_depth] int32, line_axis [B, max_depth] int32).  The
    workspace is search_value's.  Synchronous."""
    dt = _require_state(roots)
    B, N, d = roots.shape
    dev = roots.device
    workspace = _workspace(workspace, search_value_workspace_bytes(B, N, d, capacity, history), dev)
    value = torch.empty(B, dtype=torch.int32, device=dev)
    best_mask = torch.empty(B, dtype=torch.int32, device=dev)
    nodes = torch.empty(B, dtype=torch.int64, device=dev)
    status = torch.empty(B, dtype=torch.int8, device=dev)
    line_mask = torch.empty((B, max(int(max_depth), 0)), dtype=torch.int32, device=dev)
    line_axis = torch.empty_like(line_mask)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib().hk_search_value_line(_ptr(roots), _ptr(value), _ptr(best_mask), _ptr(nodes), _ptr(status),
                                        _ptr(line_mask), _ptr(line_axis), B, N, d, dt, ops, int(max_depth),
                                        int(max_nodes), int(capacity), int(history), _ptr(workspace), stream)
    check(rc, "hk_search_value_line")
    return value, best_mask, nodes, status, line_mask, line_axis


def search_value_labels_workspace_bytes(B: int, N: int, d: int, capacity: int, history: int) -> int:
    """Bytes of device workspace `search_value_labels` needs (hk_search_value_labels_workspace_bytes; 0 for refused
    arguments)."""
    return int(lib().hk_search_value_labels_workspace_bytes(B, N, d, capacity, history))


def search_value_labels(roots: torch.Tensor, *, ops: int, max_depth: int, max_nodes: int, capacity: int, history: int,
                        max_labels: int, workspace: Optional[torch.Tensor] = None):
    """search_value with every solved state of value >= 1 as a label (hk_search_value_labels): (value [B] int32,
    best_mask [B] int32, nodes [B] int64, status [B] int8, count, root [K] int32, level [K] int32, label_value [K]
    int32, optimal [K] int64, mask [K, max_depth] int32, axis [K, max_depth] int32), `count` the number of labels (a
    Python int) and K = min(count, max_labels), the first labels in history order.  Bit g of `optimal` is set when the
    host move of action id g is optimal.  `workspace` is a uint8 tensor of at least
    search_value_labels_workspace_bytes(B, N, d, capacity, history) bytes on the roots' device (allocated here when
    None).  Synchronous."""
    dt = _require_state(roots)
    B, N, d = roots.shape
    dev = roots.device
    workspace = _workspace(workspace, search_value_labels_workspace_bytes(B, N, d, capacity, history), dev)
    value = torch.empty(B, dtype=torch.int32, device=dev)
    best_mask = torch.empty(B, dtype=torch.int32, device=dev)
    nodes = torch.empty(B, dtype=torch.int64, device=dev)
    status = torch.empty(B, dtype=torch.int8, device=dev)
    L = max(int(max_labels), 0)
    root, level, label_value = (torch.empty(L, dtype=torch.int32, device=dev) for _ in range(3))
    optimal = torch.empty(L, dtype=torch.int64, device=dev)
    mask = torch.empty((L, max(int(max_depth), 0)), dtype=torch.int32, device=dev)
    axis = torch.empty_like(mask)
    count = ctypes.c_int64(0)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib().hk_search_value_labels(_ptr(roots), _ptr(value), _ptr(best_mask), _ptr(nodes), _ptr(status),
                                          int(max_labels), ctypes.addressof(count), _ptr(root), _ptr(level),
                                          _ptr(label_value), _ptr(optimal), _ptr(mask), _ptr(axis), B, N, d, dt, ops,
                                          int(max_depth), int(max_nodes), int(capacity), int(history),
                                          _ptr(workspace), stream)
    check(rc, "hk_search_value_labels")
    K = min(count.value, L)
    return (value, best_mask, nodes, status, count.value, root[:K], level[:K], label_value[:K], optimal[:K], mask[:K],
            axis[:K])


def _single_op(fn_name: str, state: torch.Tensor, inplace: bool, padding_value: float) -> Optional[torch.Tensor]:
    dt = _require_state(state)
    B, N, d = state.shape
    dst = state if inplace else torch.empty_like(state)
    with torch.cuda.device(state.device):
        stream = torch.cuda.current_stream(state.device).cuda_stream
        rc = getattr(lib(), fn_name)(_ptr(state), _ptr(dst), B, N, d, dt, float(padding_value), stream)
    check(rc, fn_name)
    return None if inplace else dst


def kernel_class(N: int, d: int) -> int:
    return lib().hk_kernel_class(N, d)


def force_generic(on: bool) -> None:
    """Test hook: route thread-per-game shapes through the warp-per-game kernel."""
    lib().hk_debug_force_generic(1 if on else 0)
