"""Episode statistics (SPEC.md §13): the cost of `EpisodeTracker.update` (`gsm_episode_stats`: the stats
kernel + the fixed-order totals kernel) over a collected rollout buffer, next to the `collect_fused`
rollout that filled the same buffer.

    python profiles/prof_episode_stats.py [--iters 200] [--out FILE]

Workloads: navigation-3 x 16384 envs x T = 25 (the bench's shape), navigation-12 x 65536 x T = 25
(BASELINE configs[4]) and navigation-96 x 4096 x T = 25, fp32, auto-reset, staggered episode ends (random
per-env step counts), so blocks meet completions at most slots.  CUDA events after a warm-up; the update and
the rollout alternate over two rounds and the faster round is kept.  The update is timed twice: its device
time, from a CUDA graph of 20 updates replayed (share_of_collect uses this one), and called from Python in a
loop (eager: the host work of a call is in that number when nothing else keeps
the GPU busy; after a collect it overlaps the collect's kernels).  The update re-reads the same slots
every iteration, so the navigation-3 and navigation-96 buffers (11 / 88 MB) come from L2, as they do right
after the collect that wrote them; navigation-12's 177 MB do not fit.  Bytes: T rows (2 sizeof(real) + 1)
of reward / cost / done plus the carry read and written (2 x 20 B per row).  The GPU's name and power limit
are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from gs_marl_b200 import scenarios
from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
from gs_marl_b200.episodes import EpisodeTracker
from gs_marl_b200.policy import GraphAttentionActor
from gs_marl_b200.rollout import GraphRolloutBuffer, collect_fused


GRAPH_UPDATES = 20


def time_it(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters          # µs per call


def workload(N, envs, T, kw, iters):
    cfg = scenarios.load("navigation").make_world(N, dtype="f32", episode_length=25, **kw)
    env = MultiAgentGraphConstrainEnv(cfg, envs, device=0, seed=1, auto_reset=True)
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    env.set_state(step_count=np.random.default_rng(0).integers(0, 25, envs).astype(np.int32))
    actor = GraphAttentionActor(len(cfg.discrete_u), seed=0)
    tracker = EpisodeTracker(env, agent_cost_limit=1.0, team_cost_limit=float(N))
    step = [0]

    def rollout():
        collect_fused(env, actor, buf, seed=1, first_step=step[0])
        step[0] += T

    def update():
        tracker.update(buf["reward"], buf["cost"], buf["done"])
    rollout()
    update()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()                         # GRAPH_UPDATES updates, replayed: no host enqueue cost
    with torch.cuda.graph(g):
        for _ in range(GRAPH_UPDATES):
            update()
    t_dev, t_upd, t_col = [], [], []
    for _ in range(2):
        t_dev.append(time_it(g.replay, max(2, iters // GRAPH_UPDATES), 2) / GRAPH_UPDATES)
        t_upd.append(time_it(update, iters, 10))
        t_col.append(time_it(rollout, max(3, iters // 40), 2))
    rows = envs * N
    nbytes = T * rows * (2 * 4 + 1) + 2 * rows * 20
    done_frac = float(buf["done"].float().mean())
    td, tu, tc = min(t_dev), min(t_upd), min(t_col)
    s = EpisodeTracker.summary(tracker.update(buf["reward"], buf["cost"], buf["done"]))
    res = {"workload": f"navigation-{N} x {envs} envs x T={T}", "rows": rows, "done_slot_fraction": round(done_frac, 4),
           "update_device_us": [round(x, 2) for x in t_dev], "update_eager_us": [round(x, 2) for x in t_upd],
           "collect_fused_us": [round(x, 1) for x in t_col], "bytes": nbytes,
           "update_GBps": round(nbytes / (td * 1e-6) / 1e9, 1), "share_of_collect": round(td / tc, 5),
           "eager_share_of_collect": round(tu / tc, 5), "agent_episodes_last_call": s["episodes"],
           "team_episodes_last_call": s["team_episodes"]}
    env.close()
    del buf, tracker
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default=None, help="also write the results to this JSON file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("prof_episode_stats.py needs a GPU")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    out = {"gpu": gpu, "results": []}
    print(json.dumps({"gpu": gpu}), flush=True)
    for N, envs, T, kw in ((3, 16384, 25, {}), (12, 65536, 25, {}), (96, 4096, 25, {"max_nbrs": 32})):
        r = workload(N, envs, T, kw, args.iters)
        out["results"].append(r)
        print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
