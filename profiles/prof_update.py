"""One PPO-Lagrangian update (SPEC.md §14): `LagrangianPPO.update` (per minibatch gsm_ppo_backward + gsm_adam_step,
three kernels) against the composition it replaces (per minibatch `evaluate_actions` + the §14 loss in torch ops +
autograd through gsm_policy_backward + `clip_grad_norm_` + `torch.optim.Adam(fused=True)`), on the same collected
rollout with the same hyper-parameters and minibatch schedule (ppo_epoch 5, a device permutation per epoch).

    python profiles/prof_update.py [--iters 3] [--warmup 1] [--out update_b200.json]

Workloads: navigation-3 x 16384 envs x T = 25 (1.23 M rows) and BASELINE configs[4] (navigation-12 x 65536 envs,
one collected slot, 786 k rows), each with num_mini_batch 1 and 4.  The two paths alternate, each timed with CUDA
events around whole updates after a warm-up; the GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from gs_marl_b200 import presets, scenarios
from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
from gs_marl_b200.learner import LagrangianPPO
from gs_marl_b200.policy import GraphAttentionActor
from gs_marl_b200.rollout import GraphRolloutBuffer, collect_fused

HP = dict(presets.UNVERIFIED_PPO_LAG, ppo_epoch=5, seed=0)


def composition(actor, trainer, buf, opt, gen):
    """The update written with the differentiable learner pass and torch's loss, clipping and optimiser."""
    x = trainer.inputs(buf)
    n = x["cnt"].numel()
    mb = n // trainer.num_mini_batch
    a = x["adv"].double()
    mu, sd = a.mean(0), a.std(0, unbiased=False)
    lam = trainer.lagrange
    out = []
    for _ in range(trainer.ppo_epoch):
        perm = torch.randperm(n, generator=gen, device="cuda")
        for b in range(trainer.num_mini_batch):
            rows = perm[b * mb:(b + 1) * mb]
            opt.zero_grad(set_to_none=True)
            lp, ent, v = actor.evaluate_actions(x["obs"], {"nbr_feat": x["feat"], "nbr_cnt": x["cnt"]}, x["act"], rows=rows)
            A = ((x["adv"][rows] - mu) / (sd + 1e-5)).float()
            abar = A[:, 0] - lam * A[:, 1]
            rho = torch.exp(lp - x["old_logp"][rows])
            lpi = -torch.min(rho * abar, rho.clamp(1 - trainer.clip, 1 + trainer.clip) * abar).mean()
            ov, R = x["old_v"][rows], x["ret"][rows]
            vc = ov + (v - ov).clamp(-trainer.value_clip, trainer.value_clip)
            lv = torch.max(0.5 * (v - R) ** 2, 0.5 * (vc - R) ** 2).sum(1).mean()
            loss = lpi + trainer.value_coef * lv - trainer.entropy_coef * ent.mean()
            loss.backward()
            out.append(torch.nn.utils.clip_grad_norm_(actor.parameters(), trainer.max_grad_norm))
            opt.step()
    return out


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


def workload(N, envs, T, n_mb, iters, warmup):
    cfg = scenarios.load("navigation").make_world(N, dtype="f32", episode_length=25)
    env = MultiAgentGraphConstrainEnv(cfg, envs, device=0, seed=1, auto_reset=True)
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    actor = GraphAttentionActor(len(cfg.discrete_u), seed=0).cuda()
    collect_fused(env, actor, buf, seed=1)
    *_, vT = actor.act(buf["obs"][-1], buf.graph(T), want_values=True)
    buf["values"][-1].copy_(vT)
    buf.compute_returns(0.99, 0.95)
    trainer = LagrangianPPO(actor, **dict(HP, num_mini_batch=n_mb))
    opt = torch.optim.Adam(actor.parameters(), lr=trainer.lr, betas=trainer.betas, eps=trainer.eps, fused=True)
    gen = torch.Generator(device="cuda").manual_seed(0)
    fused = lambda: trainer.update(buf)
    comp = lambda: composition(actor, trainer, buf, opt, gen)
    t_f, t_c = [], []
    for _ in range(3):                                   # alternate the two paths
        t_f.append(time_it(fused, iters, warmup))
        t_c.append(time_it(comp, iters, warmup))
    # the first minibatch step of both paths from the same parameters: the same loss statistics
    p0 = torch.nn.utils.parameters_to_vector(actor.parameters()).detach().clone()
    st = trainer.update(buf)[0]
    torch.nn.utils.vector_to_parameters(p0.clone(), actor.parameters())
    torch.cuda.synchronize()
    n = buf["nbr_cnt"][:-1].numel()
    tf, tc = min(t_f), min(t_c)
    res = {"workload": f"navigation-{N} x {envs} envs x T={T}", "rows": n, "ppo_epoch": HP["ppo_epoch"],
           "num_mini_batch": n_mb, "fused_update_ms": [round(x, 3) for x in t_f],
           "composition_update_ms": [round(x, 3) for x in t_c], "speedup": round(tc / tf, 3),
           "fused_ms_per_minibatch": round(tf / (HP["ppo_epoch"] * n_mb), 3),
           "composition_ms_per_minibatch": round(tc / (HP["ppo_epoch"] * n_mb), 3),
           "first_step_stats": [round(float(x), 6) for x in st]}
    env.close()
    del buf
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("prof_update.py needs a GPU")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    rec = {"gpu": gpu, "hyper_parameters": HP, "timing": "CUDA events around whole updates, min of 3 alternating "
           f"rounds of {args.iters} updates after {args.warmup} warm-up", "results": []}
    print(json.dumps({"gpu": gpu}), flush=True)
    for N, envs, T in ((3, 16384, 25), (12, 65536, 1)):
        for n_mb in (1, 4):
            r = workload(N, envs, T, n_mb, args.iters, args.warmup)
            rec["results"].append(r)
            print(json.dumps(r), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
