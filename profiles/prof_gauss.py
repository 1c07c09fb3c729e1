"""The Gaussian actor (SPEC.md §10b / §12b) against the discrete A = 5 actor on the same worlds.

    python profiles/prof_gauss.py [--iters 10] [--warmup 3] [--out gauss.json]

1. Closed loop: `collect_fused` of navigation-3, 16384 envs x T = 25, in-kernel auto-reset, replayed
   from a CUDA graph; the continuous world with GaussianGraphActor against the discrete world with
   GraphAttentionActor(5), the two graphs replayed alternately.
2. Actor kernel alone: navigation-12 x 65536 envs (786 k rows, the reset observation), with and
   without the critics, Gaussian against A = 5.
3. Learner pass: one forward + backward of the example clipped-PPO loss over the 1.23 M rows of (1),
   the kernels against the `dist_autograd` torch formulation, and the A = 5 kernels
   (profiles/prof_learner.py) in the same run.
CUDA events after a warm-up; the GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch

from gs_marl_b200 import scenarios
from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
from gs_marl_b200.policy import GaussianGraphActor, GraphAttentionActor
from gs_marl_b200.rollout import GraphRolloutBuffer, collect_fused
from prof_learner import example_loss, time_it
import prof_learner


def _env(N, envs, mode, T):
    cfg = scenarios.load("navigation").make_world(N, dtype="f32", episode_length=25, action_mode=mode)
    env = MultiAgentGraphConstrainEnv(cfg, envs, device=0, seed=1, auto_reset=True)
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    return env, buf


def closed_loop(iters, warmup):
    T, envs = 25, 16384
    runs = {}
    for name, mode, actor in (("gauss", "continuous", GaussianGraphActor(seed=0)),
                              ("discrete_a5", "discrete", GraphAttentionActor(5, seed=0))):
        env, buf = _env(3, envs, mode, T)
        actor = actor.cuda()
        runs[name] = (env, buf, collect_fused(env, actor, buf, seed=1, graph=True))
    t = {k: [] for k in runs}
    for _ in range(3):
        for k, (_, _, g) in runs.items():
            t[k].append(time_it(g.replay, iters, warmup))
    rows = envs * 3 * T
    res = {"workload": f"navigation-3 x {envs} envs x T={T}, auto-reset, CUDA graph"}
    for k in runs:
        res[f"{k}_ms"] = [round(x, 3) for x in t[k]]
        res[f"{k}_agent_steps_per_s"] = float(f"{rows / (min(t[k]) * 1e-3):.3g}")
    res["gauss_over_discrete"] = round(min(t["gauss"]) / min(t["discrete_a5"]), 3)
    for env, buf, _ in runs.values():
        env.close()
    return res


def actor_alone(iters, warmup):
    env, buf = _env(12, 65536, "discrete", 1)
    obs, g = buf["obs"][0], buf.graph(0)
    rows = obs.shape[0] * obs.shape[1]
    gauss, cat = GaussianGraphActor(seed=0).cuda(), GraphAttentionActor(5, seed=0).cuda()
    res = {"workload": "navigation-12 x 65536 envs (reset observation)", "rows": rows,
           "mean_nbr_cnt": round(float(g["nbr_cnt"].float().mean()), 3)}
    for values in (False, True):
        t = {"gauss": [], "discrete_a5": []}
        for _ in range(3):
            t["gauss"].append(time_it(lambda: gauss.act(obs, g, seed=1, want_values=values), iters, warmup))
            t["discrete_a5"].append(time_it(lambda: cat.act(obs, g, seed=1, want_values=values), iters, warmup))
        tag = "with_critics" if values else "actor_only"
        for k, v in t.items():
            res[f"{k}_{tag}_ms"] = [round(x, 4) for x in v]
        res[f"gauss_over_discrete_{tag}"] = round(min(t["gauss"]) / min(t["discrete_a5"]), 3)
    env.close()
    return res


def learner(iters, warmup):
    T = 25
    env, buf = _env(3, 16384, "continuous", T)
    actor = GaussianGraphActor(seed=0).cuda()
    collect_fused(env, actor, buf, seed=1)
    *_, vT = actor.act(buf["obs"][-1], buf.graph(T), want_values=True)
    buf["values"][-1].copy_(vT)
    ret, adv = buf.compute_returns(0.99, 0.95)
    obs, feat = buf["obs"][:-1].flatten(0, 2), buf["nbr_feat"][:-1].flatten(0, 2)
    cnt, act = buf["nbr_cnt"][:-1].flatten(0, 2), buf["actions"].flatten(0, 2)
    old_lp, ret, adv = buf["logp"].flatten(), ret.flatten(0, 2), adv[..., 0].flatten()
    idx = torch.randperm(cnt.numel(), device="cuda", generator=torch.Generator("cuda").manual_seed(0))

    def kernels():
        actor.zero_grad(set_to_none=True)
        out = actor.evaluate_actions(obs, {"nbr_feat": feat, "nbr_cnt": cnt}, act, rows=idx)
        example_loss(*out, old_lp[idx], adv[idx], ret[idx]).backward()

    def plain_torch():
        actor.zero_grad(set_to_none=True)
        g = {"nbr_feat": feat[idx], "nbr_cnt": cnt[idx]}
        d = actor.dist_autograd(obs[idx], g)
        out = d.log_prob(act[idx]).sum(-1), d.entropy().sum(-1), actor.values_autograd(obs[idx], g)
        example_loss(*out, old_lp[idx], adv[idx], ret[idx]).backward()

    grads = []
    for fn in (kernels, plain_torch):
        fn()
        grads.append(torch.cat([p.grad.reshape(-1) for p in actor.parameters()]).double())
    rel = float((grads[0] - grads[1]).norm() / grads[1].norm())
    t_k, t_t = [], []
    for _ in range(2):
        t_k.append(time_it(kernels, iters, warmup))
        t_t.append(time_it(plain_torch, iters, warmup))
    res = {"workload": f"navigation-3 x 16384 envs x T={T}, continuous", "rows": cnt.numel(),
           "mean_nbr_cnt": round(float(cnt.float().mean()), 3), "kernels_ms": [round(x, 3) for x in t_k],
           "torch_ms": [round(x, 3) for x in t_t], "speedup": round(min(t_t) / min(t_k), 2),
           "grad_rel_diff_vs_torch": rel}
    env.close()
    del buf
    torch.cuda.empty_cache()
    a5 = prof_learner.workload(3, 16384, T, iters, warmup)
    res["discrete_a5_kernels_ms"] = a5["kernels_ms"]
    res["gauss_over_discrete_kernels"] = round(min(t_k) / min(a5["kernels_ms"]), 3)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the results as one JSON file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("prof_gauss.py needs a GPU")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    out = {"gpu": gpu}
    print(json.dumps(out), flush=True)
    for name, fn in (("closed_loop", closed_loop), ("actor_alone", actor_alone), ("learner", learner)):
        out[name] = fn(args.iters, args.warmup)
        print(json.dumps({name: out[name]}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
