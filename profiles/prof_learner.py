"""The learner pass (SPEC.md §12): one forward + backward of `evaluate_actions` against the plain-torch
formulation (`embed_autograd` + head / value + log_softmax), same example clipped-surrogate loss, same
shuffled rows of a collected rollout (so the nbr_cnt distribution is the env's).

    python profiles/prof_learner.py [--iters 10] [--warmup 3]

Workloads: navigation-3 x 16384 envs x T = 25 (1.23 M rows) and BASELINE configs[4], navigation-12 x
65536 envs (one collected slot, 786 k rows).  CUDA events around each path after a warm-up; the GPU's
name and power limit are read in the same run.  FLOPs: the model's forward FMAs per row,
H (6 + NZ) + mean(nbr_cnt) H (7 + NZ) with NZ = A + 2, times 3 for forward + backward, times 2 FLOP per
FMA, over the 72 TFLOP/s FFMA rate profiles/fma_peak.cu measured (the kernels recompute the forward,
so they execute more than this count)."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from gs_marl_b200 import scenarios
from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
from gs_marl_b200.policy import GraphAttentionActor
from gs_marl_b200.rollout import GraphRolloutBuffer, collect_fused

FFMA_PEAK = 72e12
H = 64


def torch_formulation(actor, obs, feat, cnt, act):
    emb = actor.embed_autograd(obs, {"nbr_feat": feat, "nbr_cnt": cnt})
    lp_all = torch.log_softmax(actor.head(emb), -1)
    logp = lp_all.gather(-1, act.long()[..., None])[..., 0]
    return logp, -(lp_all.exp() * lp_all).sum(-1), actor.value(emb)


def example_loss(lp, ent, v, old_lp, adv, ret):
    """An example clipped surrogate + value + entropy loss (the learner's real loss is not part of the library)."""
    ratio = torch.exp(lp - old_lp)
    surr = torch.min(ratio * adv, ratio.clamp(0.8, 1.2) * adv)
    return -surr.mean() + 0.5 * ((ret - v) ** 2).mean() - 0.01 * ent.mean()


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
    return e0.elapsed_time(e1) / iters


def workload(N, envs, T, iters, warmup):
    cfg = scenarios.load("navigation").make_world(N, dtype="f32", episode_length=25)
    env = MultiAgentGraphConstrainEnv(cfg, envs, device=0, seed=1, auto_reset=True)
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    actor = GraphAttentionActor(len(cfg.discrete_u), seed=0).cuda()
    collect_fused(env, actor, buf, seed=1)
    *_, vT = actor.act(buf["obs"][-1], buf.graph(T), want_values=True)
    buf["values"][-1].copy_(vT)
    ret, adv = buf.compute_returns(0.99, 0.95)
    obs, feat = buf["obs"][:-1].flatten(0, 2), buf["nbr_feat"][:-1].flatten(0, 2)
    cnt, act = buf["nbr_cnt"][:-1].flatten(0, 2), buf["actions"].flatten(0, 2)
    old_lp, ret, adv = buf["logp"].flatten(), ret.flatten(0, 2), adv[..., 0].flatten()
    n = cnt.numel()
    idx = torch.randperm(n, device="cuda", generator=torch.Generator("cuda").manual_seed(0))

    def kernels():
        actor.zero_grad(set_to_none=True)
        out = actor.evaluate_actions(obs, {"nbr_feat": feat, "nbr_cnt": cnt}, act, rows=idx)
        example_loss(*out, old_lp[idx], adv[idx], ret[idx]).backward()

    def plain_torch():
        actor.zero_grad(set_to_none=True)
        out = torch_formulation(actor, obs[idx], feat[idx], cnt[idx], act[idx])
        example_loss(*out, old_lp[idx], adv[idx], ret[idx]).backward()

    # the two gradients agree (the bar of tests/test_policy_learner.py), then time alternately
    grads = []
    for fn in (kernels, plain_torch):
        fn()
        grads.append(torch.cat([p.grad.reshape(-1) for p in actor.parameters()]).double())
    rel = float((grads[0] - grads[1]).norm() / grads[1].norm())
    t_k, t_t = [], []
    for _ in range(2):
        t_k.append(time_it(kernels, iters, warmup))
        t_t.append(time_it(plain_torch, iters, warmup))
    mean_cnt = float(cnt.float().mean())
    A = actor.n_actions
    NZ = A + 2
    flops = 2 * 3 * n * (H * (6 + NZ) + mean_cnt * H * (7 + NZ))
    tk, tt = min(t_k), min(t_t)
    res = {"workload": f"navigation-{N} x {envs} envs x T={T}", "rows": n, "max_nbrs": int(feat.shape[-2]),
           "mean_nbr_cnt": round(mean_cnt, 3), "kernels_ms": [round(x, 3) for x in t_k],
           "torch_ms": [round(x, 3) for x in t_t], "speedup": round(tt / tk, 2),
           "model_gflop": round(flops / 1e9, 2), "kernels_share_of_ffma_peak": round(flops / (tk * 1e-3) / FFMA_PEAK, 4),
           "grad_rel_diff_vs_torch": rel}
    env.close()
    del buf
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("prof_learner.py needs a GPU")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"gpu": gpu}))
    for N, envs, T in ((3, 16384, 25), (12, 65536, 1)):
        print(json.dumps(workload(N, envs, T, args.iters, args.warmup)), flush=True)


if __name__ == "__main__":
    main()
