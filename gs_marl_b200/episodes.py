"""Episode return, cost and length on the device across rollouts, per agent and per team (SPEC.md §13).

The runner's episode logging (runner/mpe_runner.py, GSMARL.egg-info/SOURCES.txt:28) over the slots of the
rollout buffer (utils/graph_separated_buffer.py, SOURCES.txt:33): rollout windows and episodes are
decoupled — T need not equal episode_length, and masked resets or restored checkpoints stagger the episode
ends — so a per-row fp64 carry holds each agent's partial episode from one `update` to the next.

    tracker = EpisodeTracker(env, agent_cost_limit=..., team_cost_limit=...)
    buf.reset_env(); tracker.reset()
    for it in range(n_iters):
        collect_fused(env, actor, buf, ...)
        window += tracker.update(buf["reward"], buf["cost"], buf["done"])   # device fp64 [16], no sync
    stats = EpisodeTracker.summary(window)                                  # one sync

`totals` are additive: sum them over a logging window, and `torch.distributed.all_reduce` them (SUM)
across ranks before `summary` for the statistics of every rank's episodes.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import torch

from . import abi

# order of the totals (include/gsmarl_b200.h, GSM_EPISODE_STAT_FIELDS)
FIELDS = ("count", "return_sum", "return_sq_sum", "cost_sum", "cost_sq_sum", "length_sum", "safe", "over_limit")


def _check_update_inputs(reward, cost, done, n_envs, N, dtype, device):
    """The input checks of `EpisodeTracker.update`: they raise before anything is enqueued."""
    ts = (reward, cost, done)
    if not all(isinstance(t, torch.Tensor) for t in ts):
        raise TypeError("reward, cost and done must be torch tensors")
    if reward.dtype != dtype or cost.dtype != dtype or done.dtype != torch.uint8:
        raise TypeError(f"reward and cost must be {dtype} (the env's dtype), done uint8")
    shape = tuple(reward.shape)
    if len(shape) != 3 or shape[0] < 1 or shape[1:] != (n_envs, N) \
            or tuple(cost.shape) != shape or tuple(done.shape) != shape:
        raise ValueError(f"reward, cost and done must have the same shape (T, {n_envs}, {N}) with T >= 1, "
                         f"got {shape}, {tuple(cost.shape)}, {tuple(done.shape)}")
    if not all(t.is_cuda for t in ts):
        raise abi.GsmError("CUDA tensors required: gs_marl_b200 has no CPU fallback")
    if any(t.device != device for t in ts):
        raise abi.GsmError(f"reward, cost and done must be on {device}")
    if not all(t.is_contiguous() for t in ts):
        raise ValueError("reward, cost and done must be contiguous")


class EpisodeTracker:
    """Per-agent and per-team episode statistics of one env (a `MultiAgentGraphConstrainEnv` or a
    `StreamShardedEnv`), updated on the device from the buffer's reward / cost / done slots.

    Device state, [n_envs, N] per agent row and [n_envs] per env:
      carry_return, carry_cost (fp64), carry_length (int32) — the partial episode of each row;
      last_return, last_cost (fp64), last_length (int32) — the last agent episode a row completed
        (NaN / 0 until it completes one);
      team_last_return, team_last_cost (fp64) — the same per env (team return = mean over the agents,
        team cost = sum over the agents);
      episodes (int32) — the team episodes each env completed in the last `update`.
    An agent episode is safe if its cost is 0 and over the limit if its cost > agent_cost_limit; a team
    episode likewise with team_cost_limit."""

    def __init__(self, env, agent_cost_limit: float = 0.0, team_cost_limit: float = 0.0):
        self.lib = abi.load_library()
        w = env.world
        self.n_envs, self.N, self.device = int(env.n_envs), int(w.n_agents), torch.device(env.device)
        self.dtype = torch.float32 if w.dtype == "f32" else torch.float64
        self._gsm_dtype = abi.GSM_F32 if w.dtype == "f32" else abi.GSM_F64
        self.agent_cost_limit, self.team_cost_limit = float(agent_cost_limit), float(team_cost_limit)
        rows, envs = (self.n_envs, self.N), (self.n_envs,)
        f64, i32, dev = torch.float64, torch.int32, self.device
        self.carry_return = torch.zeros(rows, dtype=f64, device=dev)
        self.carry_cost = torch.zeros(rows, dtype=f64, device=dev)
        self.carry_length = torch.zeros(rows, dtype=i32, device=dev)
        self.last_return = torch.full(rows, math.nan, dtype=f64, device=dev)
        self.last_cost = torch.full(rows, math.nan, dtype=f64, device=dev)
        self.last_length = torch.zeros(rows, dtype=i32, device=dev)
        self.team_last_return = torch.full(envs, math.nan, dtype=f64, device=dev)
        self.team_last_cost = torch.full(envs, math.nan, dtype=f64, device=dev)
        self.episodes = torch.zeros(envs, dtype=i32, device=dev)
        n_ws = int(self.lib.gsm_episode_stats_workspace(self.n_envs * self.N, self.N))
        if n_ws < 0:
            raise abi.GsmError(f"{self.lib.gsm_status_string(n_ws).decode()}: gsm_episode_stats_workspace"
                               f"(n_rows={self.n_envs * self.N}, agents_per_env={self.N})")
        self._ws = torch.empty((max(n_ws, 1),), dtype=torch.uint8, device=dev)
        io = abi.GsmEpisodeIO()
        io.struct_size, io.dtype = C.sizeof(abi.GsmEpisodeIO), self._gsm_dtype
        for k in ("carry_return", "carry_cost", "carry_length", "episodes", "last_return", "last_cost",
                  "last_length", "team_last_return", "team_last_cost"):
            setattr(io, k, getattr(self, k).data_ptr())
        io.n_rows = io.slot_rows = self.n_envs * self.N
        io.agents_per_env = self.N
        io.agent_cost_limit, io.team_cost_limit = self.agent_cost_limit, self.team_cost_limit
        self._io = io

    def reset(self, mask: Optional[torch.Tensor] = None):
        """Drop the partial episodes of every env, or of the envs where mask [n_envs] (bool / uint8) is set.
        Call it after env.reset() / buf.reset_env() with the same mask."""
        if mask is None:
            for t in (self.carry_return, self.carry_cost, self.carry_length):
                t.zero_()
            return
        m = torch.as_tensor(mask, device=self.device)
        if tuple(m.shape) != (self.n_envs,):
            raise ValueError(f"mask must have shape ({self.n_envs},), got {tuple(m.shape)}")
        drop = (m != 0).unsqueeze(1)
        for t in (self.carry_return, self.carry_cost, self.carry_length):
            t.masked_fill_(drop, 0)

    def update(self, reward: torch.Tensor, cost: torch.Tensor, done: torch.Tensor) -> torch.Tensor:
        """Advance every row over the T slots of reward, cost [T, n_envs, N] (the env's real dtype) and done
        [T, n_envs, N] (uint8) — e.g. buf["reward"], buf["cost"], buf["done"] after a collect — on the current
        stream, without a host sync.  Returns this call's totals: a new device fp64 tensor
        [GSM_EPISODE_STAT_FIELDS] in the order agent (FIELDS), then team (FIELDS)."""
        _check_update_inputs(reward, cost, done, self.n_envs, self.N, self.dtype, self.device)
        totals = torch.empty((abi.GSM_EPISODE_STAT_FIELDS,), dtype=torch.float64, device=self.device)
        io = self._io
        io.reward, io.cost, io.done = reward.data_ptr(), cost.data_ptr(), done.data_ptr()
        io.totals, io.n_steps = totals.data_ptr(), int(reward.shape[0])
        st = self.lib.gsm_episode_stats(C.byref(io), C.c_void_p(self._ws.data_ptr()), self._ws.numel(),
                                        self.device.index or 0,
                                        C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
        if st != 0:
            raise abi.GsmError(f"{self.lib.gsm_status_string(st).decode()}: gsm_episode_stats")
        return totals

    @staticmethod
    def summary(totals: torch.Tensor) -> dict:
        """Statistics of the episodes counted in `totals` (one update's, or a sum of them).  Syncs.
        Keys: episodes, return_mean, return_std, cost_mean, cost_std, length_mean, safe_rate,
        over_limit_rate, then the same with a "team_" prefix.  Means are NaN when no episode completed;
        stds are the population standard deviation."""
        t = [float(x) for x in totals.detach().to("cpu", torch.float64)]
        if len(t) != abi.GSM_EPISODE_STAT_FIELDS:
            raise ValueError(f"totals must have {abi.GSM_EPISODE_STAT_FIELDS} entries, got {len(t)}")
        out = {}
        for prefix, (n, r, r2, c, c2, ln, safe, over) in (("", t[:8]), ("team_", t[8:])):
            def mean(x):
                return x / n if n > 0 else math.nan

            def std(s, s2):
                return math.sqrt(max(mean(s2) - mean(s) ** 2, 0.0)) if n > 0 else math.nan
            out.update({f"{prefix}episodes": int(n), f"{prefix}return_mean": mean(r),
                        f"{prefix}return_std": std(r, r2), f"{prefix}cost_mean": mean(c),
                        f"{prefix}cost_std": std(c, c2), f"{prefix}length_mean": mean(ln),
                        f"{prefix}safe_rate": mean(safe), f"{prefix}over_limit_rate": mean(over)})
        return out
