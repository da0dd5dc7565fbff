"""Resident int32 game batches: the engine form of the env step.

``GameBatch`` keeps one shard of games on one GPU as an int32 [B, N, d] tensor (padding -1) and
advances it with one launch per step (``step``) or one launch per T steps (``rollout``); it is
what the random-play / validation loops of the reference (``JAXTrainer.compute_rho``,
hironaka/jax/jax_trainer.py:467-556; ``Trainer.get_rho_for_pair``,
hironaka/trainer/trainer.py:302-325) reduce to once the per-step host round-trips are gone.

Games are independent, so multi-GPU is a partition of the batch: ``shard_range`` gives rank r
its contiguous chunk and nothing on the step path communicates.  ``gather_rollout`` is the one
collective: an all-gather (NCCL on GPUs) that assembles per-rank rollout buffers for training —
the analogue of the leading device axis that ``pmap`` returns in ``JAXTrainer.simulate``
(hironaka/jax/jax_trainer.py:316-320).
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch

from . import constants as C
from . import ops as _ops


def shard_range(total: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Contiguous chunk [lo, hi) of `total` games owned by `rank`; sizes differ by at most one."""
    if world_size < 1 or not 0 <= rank < world_size:
        raise ValueError(f"bad rank/world_size: {rank}/{world_size}")
    base, rem = divmod(total, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gather_rollout(tensors: Sequence[torch.Tensor], group=None) -> Tuple[torch.Tensor, ...]:
    """All-gather per-rank rollout buffers (obs / policy / value ...) along a new leading rank
    axis: each [n, ...] -> [world, n, ...].  Requires equal shapes on all ranks.  Without an
    initialised process group it returns the single-rank form [1, n, ...]."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return tuple(t.unsqueeze(0) for t in tensors)
    world = dist.get_world_size(group)
    out = []
    for t in tensors:
        t = t.contiguous()
        buf = torch.empty((world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(buf.view(world * t.shape[0], *t.shape[1:]) if t.dim() > 0 else buf, t, group=group)
        out.append(buf)
    return tuple(out)


class GameBatch:
    """B independent games resident on one GPU as int32 [B, N, d].

    semantics="jax": shift always applied, order shift -> (reposition) -> newton
                     (get_take_actions, hironaka/jax/util.py:117-123)
    semantics="torch": invalid actions and ended games are no-ops, order shift -> newton
                     (FusedGame.agent_move, hironaka/trainer/fused_game.py:150-162)

    value_threshold: every step runs through hk_rollout_threshold, which follows each game against the threshold
    (TensorPoints.value_threshold, hironaka/core/tensor_points.py:57-63): `crossed` (bool [B]) turns true once a
    live entry of a game has reached it.  With stop_at_threshold a game that crosses is not stepped again (the gym
    environments' stop_at_threshold); it enters every later call over the threshold, so it stays stopped.  For the
    int32 state the threshold must be <= 2^30 / d.  `step` is then a one-step rollout without the census.
    """

    HOST_POLICIES = {None: 0, "stream": 0, "all_coord": C.HK_F_HOST_ALL_COORD, "zeillinger": C.HK_F_HOST_ZEILLINGER,
                     "random": C.HK_F_HOST_RANDOM}
    AGENT_POLICIES = {None: 0, "stream": 0, "choose_first": C.HK_F_AGENT_FIRST, "choose_last": C.HK_F_AGENT_LAST,
                      "random": C.HK_F_AGENT_RANDOM}

    def __init__(self, points: torch.Tensor, *, semantics: str = "jax", reposition: bool = True,
                 discrete_host_action: bool = True, role: str = "host", initial_filter: bool = False,
                 host_policy: Optional[str] = None, agent_policy: Optional[str] = None, census: bool = True,
                 seed: int = 0, value_threshold: Optional[float] = None, stop_at_threshold: bool = False):
        if semantics not in ("jax", "torch"):
            raise ValueError("semantics must be 'jax' or 'torch'")
        if not points.is_cuda:
            raise _ops.HironakaB200Error("GameBatch has no CPU path: points must be a CUDA tensor")
        if points.dtype != torch.int32:
            points = points.to(torch.int32)
        self.points = points.contiguous()
        self.B, self.N, self.d = self.points.shape
        self.ops = C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0)
        # fixed players evaluated in the kernel (hironaka/jax/players.py): their action array is not needed
        self.flags = (C.TORCH_SEMANTICS if semantics == "torch" else C.JAX_SEMANTICS) | \
            (C.HK_F_ACT_DISCRETE if discrete_host_action else 0) | (C.HK_F_ROLE_AGENT if role == "agent" else 0) | \
            self.HOST_POLICIES[host_policy] | self.AGENT_POLICIES[agent_policy]
        self.reposition = reposition
        self.seed, self.steps_played = int(seed), 0  # key and step counter of the in-kernel random players
        # The census (one byte per game, hk_step_census) lets a step skip the games at rest and order the others
        # by live count.  It describes `self.points`: call reset_census() after writing into the tensor yourself.
        fixed = (self.HOST_POLICIES[host_policy] | self.AGENT_POLICIES[agent_policy]) & ~(C.HK_F_HOST_RANDOM | C.HK_F_AGENT_RANDOM)
        self.value_threshold = None if value_threshold is None else float(value_threshold)
        self.stop_at_threshold = bool(stop_at_threshold)
        threshold = self.value_threshold is not None
        self.census = _ops.new_census(self.points) if (census and not fixed and not threshold) else None
        self.crossed = torch.zeros(self.B, dtype=torch.bool, device=self.device) if threshold else None
        self._over_step = torch.empty(self.B, dtype=torch.int32, device=self.device) if threshold else None
        if initial_filter:  # generate_pts: newton -> (reposition) on the root states (util.py:385-392)
            _ops.step(self.points, ops=C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if reposition else 0), inplace=True,
                      census=self.census)

    @property
    def device(self):
        return self.points.device

    def step(self, host_action: Optional[torch.Tensor] = None, axis: Optional[torch.Tensor] = None,
             want_reward: bool = True):
        """One game-step in place; returns (done [B] bool, reward [B] f32 | None)."""
        if self.value_threshold is not None:  # a one-step rollout that follows the threshold
            ha = None if host_action is None else host_action.reshape(1, self.B)
            ax = None if axis is None else axis.reshape(1, self.B)
            done, reward, _, _ = self.rollout(ha, ax, want_done=True, want_reward=want_reward, want_length=False, steps=1)
            return done[0], (None if reward is None else reward[0])
        r = _ops.step(self.points, host_action, axis, ops=self.ops, flags=self.flags, inplace=True, want_done=True,
                      want_reward=want_reward, census=self.census)
        return r.done, r.reward

    def _threshold_args(self) -> dict:
        if self.value_threshold is None:
            return {}
        return dict(value_threshold=self.value_threshold, stop_at_threshold=self.stop_at_threshold,
                    over_step=self._over_step)

    def _note_crossings(self, steps: int) -> None:
        if self.value_threshold is not None:
            self.crossed |= self._over_step <= steps

    def reset_census(self) -> None:
        """Forget what is known about the games (after `points` was written from outside)."""
        if self.census is not None:
            self.census.zero_()

    def rollout(self, host_actions: Optional[torch.Tensor] = None, axes: Optional[torch.Tensor] = None,
                want_done: bool = False, want_reward: bool = False, want_length: bool = True,
                steps: Optional[int] = None):
        """T game-steps in ONE launch, state on chip in between.  Returns
        (done [T,B] | None, reward [T,B] | None, done_count [T] int32, length [B] int32 | None)."""
        if self.flags & (C.HK_F_HOST_RANDOM | C.HK_F_AGENT_RANDOM):  # random players drawn in the kernel: no streams
            T = steps if steps else (host_actions if host_actions is not None else axes).shape[0]
            _, done, reward, dcount, length = _ops.rollout_random(
                self.points, T, self.seed, ops=self.ops, flags=self.flags, host_actions=host_actions, axes=axes,
                step_offset=self.steps_played, inplace=True, want_done=want_done, want_reward=want_reward,
                want_length=want_length, **self._threshold_args())
            self.steps_played += T
        else:
            _, done, reward, dcount, length = _ops.rollout(self.points, host_actions, axes, ops=self.ops, flags=self.flags,
                                                           inplace=True, want_done=want_done, want_reward=want_reward,
                                                           want_done_count=True, want_length=want_length, steps=steps,
                                                           **self._threshold_args())
        self._note_crossings(dcount.shape[0])
        self.reset_census()  # the one-launch rollout does not keep it
        return done, reward, dcount, length

    def record(self, steps: Optional[int] = None, host_actions: Optional[torch.Tensor] = None,
               axes: Optional[torch.Tensor] = None, *, scale_observation: bool = True, sort: str = "lex",
               agent_obs: bool = False) -> _ops.Trajectory:
        """T game-steps in ONE launch that also record the trajectory (ops.rollout_record): obs [T, B, N*d (+d)] of the
        state before each step, with the observation options of `features` (agent_obs appends the host's coordinates
        of the step), the played host bitmasks and axes [T, B], done / reward [T, B], done_count [T] and length [B].
        The observation after the last step is features() of the batch afterwards."""
        obs_flags = (C.HK_F_OBS_RESCALE if scale_observation else 0) | \
            {"lex": C.HK_F_OBS_SORT_LEX, "coord0": C.HK_F_OBS_SORT_COORD0, "none": 0}[sort]
        traj = _ops.rollout_record(self.points, steps, host_actions, axes, ops=self.ops, flags=self.flags | obs_flags,
                                   seed=self.seed, step_offset=self.steps_played, agent_obs=agent_obs, inplace=True,
                                   **self._threshold_args())
        if self.flags & (C.HK_F_HOST_RANDOM | C.HK_F_AGENT_RANDOM):
            self.steps_played += traj.done_count.shape[0]
        self._note_crossings(traj.done_count.shape[0])
        self.reset_census()  # the one-launch rollout does not keep it
        return traj

    def step_host(self, host_action_host: torch.Tensor, axis_host: torch.Tensor) -> int:
        """One game-step driven from HOST buffers: copies this step's actions (int32 [B], ideally
        pinned) to the device, runs the step in place and returns the number of finished games
        after it, read back from the device (the per-step sync of compute_rho,
        hironaka/jax/jax_trainer.py:533-534).  Blocking."""
        if not hasattr(self, "_ha_dev"):
            self._ha_dev = torch.empty((1, self.B), dtype=torch.int32, device=self.device)
            self._ax_dev = torch.empty((1, self.B), dtype=torch.int32, device=self.device)
        self._ha_dev[0].copy_(host_action_host, non_blocking=True)
        self._ax_dev[0].copy_(axis_host, non_blocking=True)
        _, _, _, dcount, _ = _ops.rollout(self.points, self._ha_dev, self._ax_dev, ops=self.ops, flags=self.flags,
                                          inplace=True, want_done_count=True, **self._threshold_args())
        self._note_crossings(1)
        self.reset_census()
        return int(dcount.item())

    def dones(self):
        return _ops.dones(self.points)[0]

    def num_points(self):
        return _ops.dones(self.points, want_num_points=True)[1]

    def features(self, role: str = "host", scale_observation: bool = True, coords: Optional[torch.Tensor] = None,
                 sort: str = "lex"):
        """Network input of the current state: float32 [B, N*d (+d)] (get_feature_fn, util.py:172-214)."""
        flags = (C.HK_F_OBS_RESCALE if scale_observation else 0) | \
            {"lex": C.HK_F_OBS_SORT_LEX, "coord0": C.HK_F_OBS_SORT_COORD0, "none": 0}[sort] | \
            (self.flags & C.HK_F_ACT_DISCRETE)
        return _ops.features(self.points, flags=flags, obs_coord=coords if role == "agent" else None)

    @staticmethod
    def details(done_count_initial: int, done_count: torch.Tensor, batch: int):
        """Histogram of game lengths the way compute_rho accumulates it (jax_trainer.py:519-536):
        details[t] = games found finished after t steps (recorded before step t is taken),
        details[T] = games still running after T steps (last-step finishers are dropped, as there)."""
        c = [done_count_initial] + [int(v) for v in done_count.tolist()]
        T = len(c) - 1
        d = [0] * (T + 1)
        for t in range(T):
            d[t] += c[t] - (c[t - 1] if t >= 1 else 0)
        d[T] += batch - c[T]
        return d

    @staticmethod
    def rho(done_count_initial: int, done_count: torch.Tensor, batch: int) -> float:
        """rho = games finished / total steps played, from per-step finished counts
        (compute_rho, hironaka/jax/jax_trainer.py:519-555)."""
        c = [done_count_initial] + [int(v) for v in done_count.tolist()]  # c[t] = finished after t steps
        T = len(c) - 1
        details = [0] * (T + 1)
        for t in range(T):  # the reference records c[t] - c[t-1] BEFORE taking step t (jax_trainer.py:519-534)
            details[t] += c[t] - (c[t - 1] if t >= 1 else 0)
        details[T] += batch - c[T]  # games still running (:536); last-step finishers are dropped, as there
        denom = sum(i * n for i, n in enumerate(details))
        return float(sum(details[1:])) / denom if denom else float("nan")


def compute_rho(host: str, agent: str, batch_size: int, spec: Tuple[int, int], max_value: int, max_length: int,
                num_of_loops: int = 10, reposition: bool = True, generator: Optional[torch.Generator] = None,
                device="cuda", seed: int = 0):
    """rho between a fixed host and a fixed agent, the validation loop of the reference
    (JAXTrainer.compute_rho, hironaka/jax/jax_trainer.py:467-556) with every game-step on the device
    and ONE launch per batch of games: root states randint[0, max_value) -> newton -> (reposition),
    then max_length - 1 steps of `host` vs `agent`.

    host: "random" | "all_coord" | "zeillinger";  agent: "random" | "choose_first" | "choose_last"
    (hironaka/jax/players.py).  Every player is evaluated inside the kernel; the random ones draw from a
    counter-based generator keyed by `seed` (Philox, one key per loop), so no action stream is ever materialised.  Returns (rho, details) like the reference:
    rho = sum(details[1:]) / sum(i * details[i])."""
    n, d = spec
    if host not in ("random", "all_coord", "zeillinger") or agent not in ("random", "choose_first", "choose_last"):
        raise ValueError(f"unknown fixed player: {host!r} / {agent!r}")
    steps = max_length - 1
    ncls = 2 ** d - d - 1
    details = [0] * max_length
    for loop in range(num_of_loops):
        pts = torch.randint(0, max_value, (batch_size, n, d), generator=generator, device=device, dtype=torch.int32)
        gb = GameBatch(pts, semantics="jax", reposition=reposition, initial_filter=True, host_policy=host,
                       agent_policy=agent, seed=(int(seed) << 20) + loop)
        done0 = int(gb.dones().sum())
        _, _, dcount, _ = gb.rollout(None, None, want_length=False, steps=steps)
        for t, v in enumerate(GameBatch.details(done0, dcount, batch_size)):
            details[t] += v
    denom = sum(i * v for i, v in enumerate(details))
    return (float(sum(details[1:])) / denom if denom else float("nan")), details
