"""Device-resident rollout buffer and collect loop — the rows SURVEY.md §8 marks "next":
f1 `runner/mpe_runner.py` collect loop (GSMARL.egg-info/SOURCES.txt:28) and f2
`utils/graph_separated_buffer.py` insert path (SOURCES.txt:33).  Both are withheld in the
reference; this is the minimal B200-side counterpart: the env kernel writes every step's
outputs DIRECTLY into slot t of the buffer (gsm_step with the io pointers aimed at the slot),
so "insert" is not a copy, and nothing leaves the GPU between policy and env.

Layout (time-major like the lineage's buffers, agents kept as a dimension instead of one
buffer per agent): observations/graph have T+1 slots (slot t = what the policy sees before
action t), rewards/costs/dones/actions have T.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable

import torch

from . import abi
from .environment import MultiAgentGraphConstrainEnv, _TORCH_DT

_OBS_KEYS = ("obs", "nbr_idx", "nbr_feat", "nbr_cnt", "adj", "assign")
_STEP_KEYS = ("reward", "cost", "done")


class GraphRolloutBuffer:
    def __init__(self, env: MultiAgentGraphConstrainEnv, episode_length: int):
        self.env, self.T = env, int(episode_length)
        sh = env._shapes
        dev = env.device
        self.data = {}
        for k in _OBS_KEYS:
            dt, shape = sh[k]
            self.data[k] = torch.zeros((self.T + 1,) + tuple(shape), dtype=_TORCH_DT[dt], device=dev)
        for k in _STEP_KEYS + ("actions",):
            dt, shape = sh[k]
            self.data[k] = torch.zeros((self.T,) + tuple(shape), dtype=_TORCH_DT[dt], device=dev)
        self.data["logp"] = torch.zeros((self.T,) + tuple(sh["reward"][1]), dtype=torch.float32, device=dev)
        # critics' predictions for the observation of slot t (value_preds / cost_preds of the lineage's
        # buffers); slot T is filled by the caller's bootstrap forward on the last observation
        self.data["values"] = torch.zeros((self.T + 1,) + tuple(sh["reward"][1]) + (abi.GSM_POLICY_VALUE_HEADS,),
                                          dtype=torch.float32, device=dev)
        self.step = 0
        # a StreamShardedEnv is S handles over contiguous env ranges, each on its own stream, all
        # filling THIS buffer (their slot stride is the whole env count: gsm_set_slot_envs)
        self._shards = list(getattr(env, "shards", [env]))
        self._bounds = list(getattr(env, "bounds", [(0, env.n_envs)]))
        self._streams = list(getattr(env, "streams", [None] * len(self._shards)))
        # per shard, slot 0 of every tensor at the shard's first env: what gsm_collect takes (it
        # strides through the slots itself)
        self._io_all, self._io_reset = [], []
        for lo, hi in self._bounds:
            io_all, io0 = abi.GsmStepIO(), abi.GsmStepIO()
            for k in _OBS_KEYS + _STEP_KEYS + ("actions",):
                setattr(io_all, k, self.data[k][0, lo:hi].data_ptr())
            for k in _OBS_KEYS:
                setattr(io0, k, self.data[k][0, lo:hi].data_ptr())
            self._io_all.append(io_all)
            self._io_reset.append(io0)
        # one pre-built io struct per step (single-handle envs; `collect` with any torch policy):
        # outputs of step t land in obs-slot t+1 / step-slot t
        self._io = []
        for t in range(self.T if len(self._shards) == 1 else 0):
            io = abi.GsmStepIO()
            io.actions = self.data["actions"][t].data_ptr()
            for k in _OBS_KEYS:
                setattr(io, k, self.data[k][t + 1].data_ptr())
            for k in _STEP_KEYS:
                setattr(io, k, self.data[k][t].data_ptr())
            self._io.append(io)

    def __getitem__(self, k):
        return self.data[k]

    def graph(self, t: int) -> dict:
        return {k: self.data[k][t] for k in ("nbr_idx", "nbr_feat", "nbr_cnt", "adj")}

    def _on_shards(self, fn):
        """fn(shard, shard_index, stream_ptr) on every shard's stream, current stream ordered
        before and after (one handle: just the current stream)."""
        e = self.env
        with torch.cuda.device(e.device):
            if len(self._shards) == 1:
                fn(self._shards[0], 0, self._shards[0]._stream())
                return
            e.fork()
            for j, (sh, st) in enumerate(zip(self._shards, self._streams)):
                fn(sh, j, C.c_void_p(st.cuda_stream))
            e.join()

    def reset_env(self):
        """env.reset() with the first observation written straight into slot 0."""
        self._on_shards(lambda sh, j, st: sh._check(
            sh.lib.gsm_reset(sh._h, sh._seed, None, 1, C.byref(self._io_reset[j]), st)))
        self.step = 0

    def compute_returns(self, gamma: float = 0.99, gae_lambda: float = 0.95, value_norm=None):
        """buffer.compute_returns + compute_cost_returns of the lineage (GAE, SPEC.md §11), one kernel
        for both critics: fills `returns` and `advantages` [T, n_envs, N, 2] from reward / cost / done
        and `values` (slot T must hold the bootstrap prediction for the last observation).  With a
        `learner.ValueNorm` (SPEC.md §15) the values are the critics' normalised outputs: every one is
        denormalised with the normaliser's current affine first (`gsm_gae_normalized`), so returns and
        advantages are in raw units."""
        d, e = self.data, self.env
        for k in ("returns", "advantages"):
            if k not in d:
                d[k] = torch.zeros_like(d["values"][:-1])
        lib = abi.load_library()
        rows = d["reward"][0].numel()
        args = (d["reward"].data_ptr(), d["cost"].data_ptr(), d["values"].data_ptr(), d["done"].data_ptr(), self.T,
                rows, rows, float(gamma), float(gae_lambda), d["returns"].data_ptr(), d["advantages"].data_ptr())
        with torch.cuda.device(e.device):
            stream = C.c_void_p(torch.cuda.current_stream(e.device).cuda_stream)
            if value_norm is None:
                st = lib.gsm_gae(*args, e.device.index or 0, stream)
            else:
                if value_norm.affine.device != d["values"].device:
                    raise ValueError(f"value_norm must live on {d['values'].device}")
                st = lib.gsm_gae_normalized(*args, value_norm.affine.data_ptr(), e.device.index or 0, stream)
        if st != 0:
            raise abi.GsmError(f"{lib.gsm_status_string(st).decode()}: {lib.gsm_policy_last_error().decode()}")
        return d["returns"], d["advantages"]

    def after_update(self):
        """Lineage buffers copy the last observation to slot 0 after an update."""
        for k in _OBS_KEYS:
            self.data[k][0].copy_(self.data[k][self.T])
        self.step = 0


def collect(env: MultiAgentGraphConstrainEnv, policy: Callable, buf: GraphRolloutBuffer) -> GraphRolloutBuffer:
    """One rollout of buf.T steps: actions = policy(obs_t, graph_t) -> [n_envs, N(,2)] device
    tensor; the env step writes reward/cost/done of step t and obs/graph of t+1 into the buffer."""
    if len(buf._shards) != 1:
        raise ValueError("collect() drives one handle; use collect_fused() with a StreamShardedEnv")
    with torch.cuda.device(env.device):
        stream = env._stream()
        for t in range(buf.T):
            a = policy(buf.data["obs"][t], buf.graph(t))
            buf.data["actions"][t].copy_(a)
            env._check(env.lib.gsm_step(env._h, C.byref(buf._io[t]), stream))
            if env.auto_reset:      # finished envs restart; their first observation replaces slot t+1
                env._check(env.lib.gsm_reset(env._h, env._seed, C.c_void_p(buf.data["done"][t].data_ptr()),
                                             env.world.n_agents, C.byref(buf._io[t]), stream))
    buf.step = buf.T
    return buf


def collect_fused(env: MultiAgentGraphConstrainEnv, actor, buf: GraphRolloutBuffer, seed: int = 0,
                  first_step: int = 0, greedy: bool = False, graph: bool = False, with_values: bool = True):
    """The same rollout with the actor forward + sampling as this library's kernel
    (`gsm_collect`: per step one actor launch and one env-step launch, enqueued from C with no
    Python or host sync in between; actions, log-probs and — with_values — the two critics'
    predictions land in the buffer slots).  `actor` is a `policy.GraphAttentionActor` for a
    discrete-action world or a `policy.GaussianGraphActor` (`gsm_collect_gauss`) for a continuous one.  With a `StreamShardedEnv` every sub-shard runs its own
    actor -> env-step chain on its own stream into its env slice of the buffer, so one shard's actor
    kernel (fp32-issue-bound) overlaps another's env step (HBM-bound).  graph=True captures the 2·T launches into a CUDA graph and
    returns it WITHOUT having advanced the env (replay runs the rollout from the env's current
    state and whatever slot 0 holds, with the Philox step counters and the weights baked in at
    capture: re-capture after an optimizer step)."""
    mode, kind = env.world.action_mode, getattr(actor, "action_mode", None)
    if kind is not None and kind != mode:       # other actors: the C side reports a mismatch (GSM_ERR_UNSUPPORTED)
        raise ValueError(f"{type(actor).__name__} samples {kind} actions; the env's action_mode is "
                         f"{mode!r} (use {'GaussianGraphActor' if mode == 'continuous' else 'GraphAttentionActor'})")
    w = actor.packed()
    collect_fn = "gsm_collect_gauss" if isinstance(w, abi.GsmPolicyGaussWeights) else "gsm_collect"
    logp, values = buf.data["logp"], buf.data["values"]
    for sh in buf._shards:          # reset-on-done inside the loop follows the env's flag
        sh._check(sh.lib.gsm_set_auto_reset(sh._h, int(bool(env.auto_reset))))


    def enqueue():
        buf._on_shards(lambda sh, j, st: sh._check(getattr(sh.lib, collect_fn)(
            sh._h, C.byref(w), buf.T, C.byref(buf._io_all[j]),
            C.c_void_p(logp[0, buf._bounds[j][0]:].data_ptr()),
            C.c_void_p(values[0, buf._bounds[j][0]:].data_ptr()) if with_values else None, int(seed), int(first_step),
            int(bool(greedy)), st)))
    with torch.cuda.device(env.device):
        if not graph:
            enqueue()
            buf.step = buf.T
            return buf
        # one eager rollout first (module load / first-launch work must not happen inside a
        # capture); the env state is put back afterwards, slot 0 is never written by a collect
        saved, saved_ep = env.get_state(), env.get_episode()
        enqueue()
        env.set_state(*saved)
        env.set_episode(saved_ep)          # re-draws inside the replay must see the same episode numbers
        torch.cuda.synchronize(env.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            enqueue()
        buf.step = buf.T
        return g
