"""Batched counterparts of the reference's three env classes
(gsmarl/envs/mpe_env/multiagent/environment.py, GSMARL.egg-info/SOURCES.txt:15;
described in reference readme.md:27-41):

    MultiAgentEnv               fixed-size obs, no cost           (readme.md:29-33)
    MultiAgentConstrainEnv      fixed-size obs + cost             (readme.md:34-37)
    MultiAgentGraphConstrainEnv variable-size graph obs + cost    (readme.md:38-41)

One object = `n_envs` independent worlds resident on one B200; `step` is ONE fused
kernel launch through the C ABI (include/gsmarl_b200.h).  torch is used only for device
memory and the current stream.  The reference's per-env return convention (lists of
per-agent arrays) becomes stacked tensors with leading dims [n_envs, n_agents].

The reference source is withheld, so the exact tuple arity/order of its `step` cannot
be checked; the order here is the one BASELINE.json's north_star states:
`obs, graph/adjacency, rewards, costs, dones, infos`.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import abi
from .config import WorldConfig

_TORCH_DT = {np.float32: torch.float32, np.float64: torch.float64, np.int32: torch.int32,
             np.uint32: torch.int32, np.uint8: torch.uint8}


class Box:
    """Shape/dtype descriptor standing in for gym.spaces.Box (gym is not a dependency)."""

    def __init__(self, shape, dtype):
        self.shape, self.dtype = tuple(shape), dtype

    def __repr__(self):
        return f"Box(shape={self.shape}, dtype={np.dtype(self.dtype).name})"


class Discrete:
    def __init__(self, n):
        self.n = n

    def __repr__(self):
        return f"Discrete({self.n})"


class MultiAgentGraphConstrainEnv:
    OUTPUTS = ("obs", "nbr_idx", "nbr_feat", "nbr_cnt", "adj", "reward", "cost", "done", "assign")

    def __init__(self, world: WorldConfig, n_envs: int, device: int = 0, env_offset: int = 0,
                 auto_reset: bool = False, seed: int = 0):
        self.world, self.n_envs, self.device_index = world, int(n_envs), int(device)
        self.env_offset, self.auto_reset = int(env_offset), bool(auto_reset)
        self.lib = abi.load_library()
        if not torch.cuda.is_available():
            raise abi.GsmError("CUDA device required: gs_marl_b200 has no CPU fallback")
        self.device = torch.device("cuda", self.device_index)
        self._c, self._keep = world.to_c()
        self._h = C.c_void_p()
        abi.check(self.lib, self.lib.gsm_create(C.byref(self._c), self.n_envs, self.env_offset,
                                                self.device_index, C.byref(self._h)))
        self._seed = int(seed)
        self._shapes = world.io_shapes(self.n_envs)
        self.buf = {k: self._alloc(k) for k in self.OUTPUTS}
        self._io = self._make_io(self.buf)
        # reference-style attributes (per agent)
        self.n = world.n_agents
        n, K = world.n_agents, world.max_nbrs
        self.observation_space = [Box((abi.GSM_OBS_DIM,), world.np_real)] * n
        self.node_observation_space = [Box((K, abi.GSM_NBR_FEAT_DIM), world.np_real)] * n
        self.adj_observation_space = [Box((world.adj_words,), np.uint32)] * n
        self.share_observation_space = [Box((n * abi.GSM_OBS_DIM,), world.np_real)] * n
        self.action_space = ([Discrete(len(world.discrete_u))] * n
                             if world.action_mode == "discrete" else [Box((2,), world.np_real)] * n)

    # ---- plumbing ---------------------------------------------------------------------
    def _alloc(self, name, lead=()):
        dt, shape = self._shapes[name]
        return torch.zeros(tuple(lead) + tuple(shape), dtype=_TORCH_DT[dt], device=self.device)

    @staticmethod
    def _make_io(bufs: dict, actions: Optional[torch.Tensor] = None) -> abi.GsmStepIO:
        io = abi.GsmStepIO()
        for k in abi.GsmStepIO.FIELDS:
            t = actions if k == "actions" else bufs.get(k)
            setattr(io, k, None if t is None else t.data_ptr())
        return io

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, st):
        abi.check(self.lib, st, self._h)

    def _actions(self, actions) -> torch.Tensor:
        dt, shape = self._shapes["actions"]
        a = torch.as_tensor(actions, device=self.device).to(_TORCH_DT[dt]).contiguous()
        if tuple(a.shape) != tuple(shape):
            raise ValueError(f"actions must have shape {tuple(shape)}, got {tuple(a.shape)}")
        return a

    def _result(self, b):
        graph = {"nbr_idx": b["nbr_idx"], "nbr_feat": b["nbr_feat"], "nbr_cnt": b["nbr_cnt"],
                 "adj": b["adj"]}
        infos = {"assign": b["assign"], "collisions": b["cost"]}
        return b["obs"], graph, b["reward"], b["cost"], b["done"], infos

    # ---- reference API ----------------------------------------------------------------
    def seed(self, seed: int):
        self._seed = int(seed)

    def reset(self, mask: Optional[torch.Tensor] = None):
        """reset() -> obs, graph.  mask: optional uint8/bool [n_envs] (device)."""
        m, stride = None, 1
        if mask is not None:
            mt = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            if tuple(mt.shape) != (self.n_envs,):       # the reset kernel reads one byte per env
                raise ValueError(f"mask must have shape ({self.n_envs},), got {tuple(mt.shape)}")
            m = C.c_void_p(mt.data_ptr())
        with torch.cuda.device(self.device):
            self._check(self.lib.gsm_reset(self._h, self._seed, m, stride, C.byref(self._io),
                                           self._stream()))
        b = self.buf
        return b["obs"], {"nbr_idx": b["nbr_idx"], "nbr_feat": b["nbr_feat"],
                          "nbr_cnt": b["nbr_cnt"], "adj": b["adj"]}

    def step(self, actions):
        """step(actions) -> obs, graph, rewards, costs, dones, infos (device tensors, views of
        buffers that the next step overwrites)."""
        a = self._actions(actions)
        io = self._make_io(self.buf, a)
        with torch.cuda.device(self.device):
            self._check(self.lib.gsm_step(self._h, C.byref(io), self._stream()))
            if self.auto_reset:
                # done envs restart; their obs/graph rows become the first obs of the new
                # episode, reward/cost/done keep the terminal step's values.
                self._check(self.lib.gsm_reset(self._h, self._seed, C.c_void_p(self.buf["done"].data_ptr()),
                                               self.world.n_agents, C.byref(self._io), self._stream()))
        return self._result(self.buf)

    def rollout(self, actions, out: Optional[dict] = None, auto_reset: Optional[bool] = None) -> dict:
        """T steps in one launch (fused kernel, or a CUDA graph for shapes without one); actions
        [T, n_envs, N(,2)]; returns dict of [T, ...] tensors (the rollout-buffer layout,
        SURVEY.md §8 f2).  auto_reset (default: the env's flag): envs that finish inside the
        rollout keep their terminal outputs in that slot and are re-drawn before the next step."""
        dt, shape = self._shapes["actions"]
        a = torch.as_tensor(actions, device=self.device).to(_TORCH_DT[dt]).contiguous()
        T = a.shape[0]
        if tuple(a.shape[1:]) != tuple(shape):
            raise ValueError(f"actions must have shape (T,)+{tuple(shape)}")
        if out is None:
            out = {k: self._alloc(k, (T,)) for k in self.OUTPUTS}
        for k in self.OUTPUTS:                            # the kernel writes T full slots of each
            dt, shape = self._shapes[k]
            o = out[k]
            if tuple(o.shape) != (T,) + tuple(shape) or o.dtype != _TORCH_DT[dt] or o.device != self.device \
                    or not o.is_contiguous():
                raise ValueError(f"out[{k!r}] must be a contiguous {_TORCH_DT[dt]} tensor of shape "
                                 f"{(T,) + tuple(shape)} on {self.device}")
        io = self._make_io(out, a)
        ar = self.auto_reset if auto_reset is None else bool(auto_reset)
        with torch.cuda.device(self.device):
            self._check(self.lib.gsm_set_auto_reset(self._h, int(ar)))
            self._check(self.lib.gsm_rollout(self._h, T, C.byref(io), self._stream()))
        out["actions"] = a
        return out

    def observe(self):
        with torch.cuda.device(self.device):
            self._check(self.lib.gsm_observe(self._h, C.byref(self._io), self._stream()))
        return self._result(self.buf)[:2]

    # ---- state access (parity tests, checkpoint/resume) ---------------------------------
    def state_tensors(self):
        w, r = self.world, _TORCH_DT[self.world.np_real]
        return (torch.zeros((self.n_envs, w.n_agents, 4), dtype=r, device=self.device),
                torch.zeros((self.n_envs, w.n_landmarks, 2), dtype=r, device=self.device),
                torch.zeros((self.n_envs,), dtype=torch.int32, device=self.device))

    def set_state(self, agent_state=None, landmark_pos=None, step_count=None):
        r = _TORCH_DT[self.world.np_real]

        def prep(x, dt):
            return None if x is None else torch.as_tensor(x).to(device=self.device, dtype=dt).contiguous()
        a, l, t = prep(agent_state, r), prep(landmark_pos, r), prep(step_count, torch.int32)
        w = self.world
        # the copies read n_envs rows of each: a smaller array would be read past its end
        for name, x, shape in (("agent_state", a, (self.n_envs, w.n_agents, 4)),
                               ("landmark_pos", l, (self.n_envs, w.n_landmarks, 2)),
                               ("step_count", t, (self.n_envs,))):
            if x is not None and tuple(x.shape) != shape:
                raise ValueError(f"{name} must have shape {shape}, got {tuple(x.shape)}")
        p = [C.c_void_p(x.data_ptr()) if x is not None and x.numel() else None for x in (a, l, t)]
        with torch.cuda.device(self.device):
            self._check(self.lib.gsm_set_state(self._h, p[0], p[1], p[2], self._stream()))
            torch.cuda.current_stream(self.device).synchronize()

    def get_state(self):
        a, l, t = self.state_tensors()
        with torch.cuda.device(self.device):
            self._check(self.lib.gsm_get_state(self._h, a.data_ptr(), l.data_ptr() if l.numel() else None,
                                               t.data_ptr(), self._stream()))
        return a, l, t

    def get_episode(self) -> torch.Tensor:
        """Episode counter per env (keys the reset draws; part of a full checkpoint)."""
        ep = torch.zeros((self.n_envs,), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.gsm_get_episode(self._h, ep.data_ptr(), self._stream()))
        return ep

    def set_episode(self, episode):
        ep = torch.as_tensor(episode).to(device=self.device, dtype=torch.int32).contiguous()
        if tuple(ep.shape) != (self.n_envs,):
            raise ValueError(f"episode must have shape ({self.n_envs},)")
        with torch.cuda.device(self.device):
            self._check(self.lib.gsm_set_episode(self._h, ep.data_ptr(), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()

    @property
    def kernel_launches(self) -> int:
        return int(self.lib.gsm_kernel_launches(self._h))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.gsm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class StreamShardedEnv:
    """`n_envs` worlds of ONE GPU as `n_streams` contiguous sub-shards, each its own handle on its
    own CUDA stream, all writing slices of the SAME output / rollout buffers.

    Why: one fused-rollout launch over the bench batch (16384 envs x 3 agents = 6144 warps) is
    1.5 rounds of the 28 warps/SM the kernel can keep resident, so the second round runs half
    empty and every launch ends with a drained GPU.  Sub-shards are independent (the same
    property the multi-GPU sharding uses; reset draws depend on the GLOBAL env index, so the
    worlds are identical to one handle's), and with `join=False` successive rollouts of different
    shards overlap: the tail of one launch is filled by the body of the next.  Measured on a
    B200 (profiles/README.md): 4.30 -> 3.50 us per env step, 56.5 -> 69.5 % of the HBM peak.

    `reset` / `step` / `rollout(join=True)` return with the CURRENT stream ordered after all
    shard streams, i.e. they behave like MultiAgentGraphConstrainEnv.  `rollout(join=False)`
    leaves the shards running; call `join()` before reading the buffers from the current stream.
    """

    OUTPUTS = MultiAgentGraphConstrainEnv.OUTPUTS

    def __init__(self, world: WorldConfig, n_envs: int, n_streams: int = 4, device: int = 0,
                 env_offset: int = 0, auto_reset: bool = False, seed: int = 0):
        from .env_wrappers import shard_bounds
        self.world, self.n_envs, self.auto_reset = world, int(n_envs), bool(auto_reset)
        self.n_streams = max(1, min(int(n_streams), max(1, self.n_envs)))
        self.env_offset = int(env_offset)
        self.device = torch.device("cuda", int(device))
        self.bounds = [shard_bounds(self.n_envs, self.n_streams, s) for s in range(self.n_streams)]
        self.shards = [MultiAgentGraphConstrainEnv(world, hi - lo, device=device, env_offset=self.env_offset + lo,
                                                   seed=seed) for lo, hi in self.bounds]
        self.streams = [torch.cuda.Stream(device=self.device) for _ in self.shards]
        first = self.shards[0]
        self.lib, self._shapes = first.lib, world.io_shapes(self.n_envs)
        self.buf = {k: self._alloc(k) for k in self.OUTPUTS}
        for sh, (lo, hi) in zip(self.shards, self.bounds):
            sh.buf = {k: v[lo:hi] for k, v in self.buf.items()}     # contiguous env slices
            sh._io = sh._make_io(sh.buf)
            sh._check(self.lib.gsm_set_slot_envs(sh._h, self.n_envs))
        for a in ("n", "observation_space", "node_observation_space", "adj_observation_space",
                  "share_observation_space", "action_space"):
            setattr(self, a, getattr(first, a))

    def _alloc(self, name, lead=()):
        dt, shape = self._shapes[name]
        return torch.zeros(tuple(lead) + tuple(shape), dtype=_TORCH_DT[dt], device=self.device)

    # ---- stream plumbing ----------------------------------------------------------------
    def fork(self):
        """Order every shard stream after what is enqueued on the current stream so far."""
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        for st in self.streams:
            st.wait_event(ev)

    def join(self):
        """Order the current stream after everything enqueued on the shard streams."""
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            cur.wait_stream(st)

    def _each(self, fn):
        self.fork()
        for sh, st, (lo, hi) in zip(self.shards, self.streams, self.bounds):
            with torch.cuda.stream(st):
                fn(sh, lo, hi)

    # ---- reference API ----------------------------------------------------------------------
    def seed(self, seed: int):
        for sh in self.shards:
            sh.seed(seed)

    def reset(self, mask: Optional[torch.Tensor] = None):
        m = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
        self._each(lambda sh, lo, hi: sh.reset(None if m is None else m[lo:hi]))
        self.join()
        return self.shards[0]._result(self.buf)[:2]

    def step(self, actions):
        dt, shape = self._shapes["actions"]
        a = torch.as_tensor(actions, device=self.device).to(_TORCH_DT[dt]).contiguous()
        if tuple(a.shape) != tuple(shape):
            raise ValueError(f"actions must have shape {tuple(shape)}, got {tuple(a.shape)}")

        def one(sh, lo, hi):
            sh.auto_reset = self.auto_reset
            sh.step(a[lo:hi])
        self._each(one)
        self.join()
        return self.shards[0]._result(self.buf)

    def rollout(self, actions, out: Optional[dict] = None, auto_reset: Optional[bool] = None,
                join: bool = True) -> dict:
        """T fused steps per shard, every shard writing its env slice of the [T, n_envs, ...]
        tensors of `out` (gsm_set_slot_envs).  join=False: return with the launches in flight."""
        dt, shape = self._shapes["actions"]
        a = torch.as_tensor(actions, device=self.device).to(_TORCH_DT[dt]).contiguous()
        T = a.shape[0]
        if tuple(a.shape[1:]) != tuple(shape):
            raise ValueError(f"actions must have shape (T,)+{tuple(shape)}")
        if out is None:
            out = {k: self._alloc(k, (T,)) for k in self.OUTPUTS}
        launch = self.rollout_plan(a, out, auto_reset)
        with torch.cuda.device(self.device):
            self.fork()
            launch()
        if join:
            self.join()
        out["actions"] = a
        return out

    def rollout_plan(self, actions: torch.Tensor, out: dict, auto_reset: Optional[bool] = None):
        """Pre-built launch of one T-step fused rollout per shard: returns `launch()`, which only
        enqueues the S kernels on the shard streams (no fork, no join, no per-call Python setup) —
        the collect loop of a caller that replays fixed buffers.  `actions` [T, n_envs, N(,2)] and
        the tensors of `out` must stay alive and in place; order them yourself (`fork`/`join`)."""
        T = actions.shape[0]
        ar = int(self.auto_reset if auto_reset is None else bool(auto_reset))
        ios = [sh._make_io({k: out[k][0, lo:hi] for k in self.OUTPUTS}, actions[0, lo:hi])
               for sh, (lo, hi) in zip(self.shards, self.bounds)]
        streams = [C.c_void_p(st.cuda_stream) for st in self.streams]
        for sh in self.shards:
            sh._check(self.lib.gsm_set_auto_reset(sh._h, ar))
        lib, shards = self.lib, self.shards

        def launch():
            for sh, io, st in zip(shards, ios, streams):
                sh._check(lib.gsm_rollout(sh._h, T, C.byref(io), st))
        return launch

    def get_state(self):
        parts = [sh.get_state() for sh in self.shards]
        return tuple(torch.cat([p[j] for p in parts], 0) for j in range(3))

    def get_episode(self):
        return torch.cat([sh.get_episode() for sh in self.shards], 0)

    def set_episode(self, episode):
        for sh, (lo, hi) in zip(self.shards, self.bounds):
            sh.set_episode(episode[lo:hi])

    def set_state(self, agent_state=None, landmark_pos=None, step_count=None):
        for sh, (lo, hi) in zip(self.shards, self.bounds):
            sh.set_state(*(None if x is None else x[lo:hi] for x in (agent_state, landmark_pos, step_count)))

    @property
    def kernel_launches(self) -> int:
        return sum(sh.kernel_launches for sh in self.shards)

    def close(self):
        for sh in getattr(self, "shards", []):
            sh.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiAgentConstrainEnv(MultiAgentGraphConstrainEnv):
    """Fixed-size observation + cost (readme.md:34-37).  The fixed-size observation is the
    agent's own 6 features followed by its K padded neighbour rows, flattened
    [DECL: the reference's fixed layout is unknown]."""

    def _flat_obs(self, b):
        n_envs, N = self.n_envs, self.world.n_agents
        return torch.cat([b["obs"], b["nbr_feat"].reshape(n_envs, N, -1)], dim=-1)

    def reset(self, mask=None):
        super().reset(mask)
        return self._flat_obs(self.buf)

    def step(self, actions):
        super().step(actions)
        b = self.buf
        return self._flat_obs(b), b["reward"], b["cost"], b["done"], {"assign": b["assign"]}


class MultiAgentEnv(MultiAgentConstrainEnv):
    """Fixed-size observation, no cost (readme.md:29-33)."""

    def step(self, actions):
        obs, rew, _cost, done, infos = super().step(actions)
        return obs, rew, done, infos
