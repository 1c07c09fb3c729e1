"""Measurement helpers shared by bench.py and the scripts under profiles/.

`RolloutRegion` is the timed region of every device-resident number this repo reports: K env
steps of one handle (or of the S sub-shard handles of a StreamShardedEnv) as fused gsm_rollout
launches, captured ONCE in a CUDA graph and replayed back to back — so no Python / ctypes
launch latency sits between the CUDA events, whatever K is (VERDICT r1: at the driver's
`--steps 20` the old host-launched region was one ~0.1 ms launch per stream and measured the
host, not the kernel).
"""
from __future__ import annotations

import ctypes as C
import math

import torch

GRAPH_CHUNK_STEPS = 2500     # steps held by one CUDA graph (K larger than this is replayed in chunks)


class RolloutRegion:
    """K consecutive env steps of `env` as CUDA graph(s).

    * fused launches of min(T, remaining) steps each (T = slots of the `ring` rollout buffer the
      kernels write: slot s of launch j is ring[s]; the ring is larger than L2),
    * a StreamShardedEnv's shards run on their own streams inside the graph (fork at the graph
      head, join at its tail; consecutive launches of one shard are chained on its stream, shards
      are not joined in between),
    * K <= GRAPH_CHUNK_STEPS: the graph holds c = GRAPH_CHUNK_STEPS // K copies of the K-step
      region (one replay = c regions; c = 1 with pack=False, so that one unit is exactly K
      steps); larger K: a GRAPH_CHUNK_STEPS graph replayed K // chunk times plus one graph with
      the remainder.
    State persists across launches and replays, so with auto-reset on, every env is re-drawn
    in-kernel every `episode_length` steps whatever K and T are: no work is skipped.
    """

    def __init__(self, env, acts, ring, K, T, auto_reset=True, pack=True):
        self.env, self.K, self.T = env, int(K), int(T)
        self.sharded = hasattr(env, "shards")
        self.dev = env.device
        lib = env.lib
        shards = env.shards if self.sharded else [env]
        bounds = env.bounds if self.sharded else [(0, env.n_envs)]
        for sh in shards:
            sh._check(lib.gsm_set_auto_reset(sh._h, int(bool(auto_reset))))
        self._ios = [sh._make_io({k: ring[k][0, lo:hi] for k in env.OUTPUTS}, acts[0, lo:hi])
                     for sh, (lo, hi) in zip(shards, bounds)]
        self._keep = (acts, ring)
        self._shards, self._lib = shards, lib
        self.launches_per_region = len(shards) * math.ceil(self.K / self.T)
        self.launch_steps = []           # steps of every fused launch of one K-step region (one shard)
        d = 0
        while d < self.K:
            m = min(self.T, self.K - d)
            self.launch_steps.append(m)
            d += m
        if self.K <= GRAPH_CHUNK_STEPS:
            self.copies = max(1, GRAPH_CHUNK_STEPS // self.K) if pack else 1
            self.plan = [(self._capture([self.K] * self.copies), 1)]      # (graph, replays per unit)
            self.regions_per_unit = self.copies
            last_segment = self.K
        else:
            q, r = divmod(self.K, GRAPH_CHUNK_STEPS)
            self.copies = 1
            self.plan = [(self._capture([GRAPH_CHUNK_STEPS]), q)]
            if r:
                self.plan.append((self._capture([r]), 1))
            self.regions_per_unit = 1
            last_segment = r or GRAPH_CHUNK_STEPS
        # every fused launch writes ring slots 0, 1, ...: the last step of a unit lands here
        self.last_slot = (last_segment - 1) % self.T

    def _enqueue(self, n_steps, streams):
        done = 0
        while done < n_steps:
            m = min(self.T, n_steps - done)
            for sh, io, st in zip(self._shards, self._ios, streams):
                sh._check(self._lib.gsm_rollout(sh._h, m, C.byref(io), st))
            done += m

    def _capture(self, segments):
        env = self.env
        g = torch.cuda.CUDAGraph()
        with torch.cuda.device(self.dev), torch.cuda.graph(g):
            if self.sharded:
                env.fork()
                streams = [C.c_void_p(st.cuda_stream) for st in env.streams]
            else:
                streams = [C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)]
            for n in segments:
                self._enqueue(n, streams)
            if self.sharded:
                env.join()
        return g

    def replay_unit(self):
        """One unit = `regions_per_unit` K-step regions, enqueued on the current stream."""
        for g, n in self.plan:
            for _ in range(n):
                g.replay()

    def run(self, units):
        """Enqueue `units` units back to back between two CUDA events; returns (ms, regions)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(units):
            self.replay_unit()
        e1.record()
        torch.cuda.synchronize(self.dev)
        return e0.elapsed_time(e1), units * self.regions_per_unit

    def calibrate(self, target_ms):
        """Units needed for a region of at least `target_ms` (one probe unit, already warm)."""
        ms, _ = self.run(1)
        return max(1, math.ceil(target_ms / max(ms, 1e-3)))

    def bytes_per_region(self, cfg):
        """Algorithmic HBM bytes of one K-step region (WorldConfig.bytes_fused per launch)."""
        n_envs = self.env.n_envs
        return sum(cfg.bytes_fused(n_envs, m) for m in self.launch_steps)


def time_rollouts(env, cfg, acts, ring, K, T, auto_reset, target_ms, warm_units=1):
    """step_us, achieved GB/s and the region record of K-step regions of `env` replayed for at
    least target_ms."""
    reg = RolloutRegion(env, acts, ring, K, T, auto_reset)
    for _ in range(warm_units):
        reg.replay_unit()
    torch.cuda.synchronize(env.device)
    units = reg.calibrate(target_ms)
    ms, regions = reg.run(units)
    step_us = ms * 1e3 / (regions * K)
    gbs = reg.bytes_per_region(cfg) * regions / (ms * 1e-3) / 1e9
    return {"step_us": step_us, "achieved": gbs, "regions": regions, "ms": ms,
            "launches": regions * reg.launches_per_region}
