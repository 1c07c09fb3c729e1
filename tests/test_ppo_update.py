"""The PPO-Lagrangian update (SPEC.md §14): `gsm_ppo_backward(_gauss)`, `gsm_adam_step` and `LagrangianPPO`
against the float64 restatement in tests/_ppo_oracle.py, torch autograd and torch.optim.Adam."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from gs_marl_b200 import abi, presets
from gs_marl_b200.learner import LagrangianPPO, STAT_FIELDS
from gs_marl_b200.policy import GaussianGraphActor, GraphAttentionActor
from oracle import policy_oracle as P
from tests import _gauss_oracle as G
from tests import _learner_oracle as L
from tests import _ppo_oracle as O
from tests._util import make_cfg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
DEV = "cuda"
COEFS = dict(clip=0.2, value_clip=0.2, value_coef=0.5, entropy_coef=0.01)
HP = dict(presets.UNVERIFIED_PPO_LAG, value_coef=0.5, seed=0)


# ---- the oracle against torch autograd of the §14 formula (CPU) -----------------------------------------
def _torch_loss(logp, ent, v, old_logp, old_v, R, A, mom, lam, clip, value_clip, value_coef, entropy_coef):
    n = logp.shape[0]
    abar = (A[:, 0] - mom[0]) / (mom[1] + 1e-5) - lam * (A[:, 1] - mom[2]) / (mom[3] + 1e-5)
    rho = torch.exp(logp - old_logp)
    lpi = -torch.min(rho * abar, torch.clamp(rho, 1 - clip, 1 + clip) * abar).sum() / n
    vc = old_v + torch.clamp(v - old_v, -value_clip, value_clip)
    lv = torch.max(0.5 * (v - R) ** 2, 0.5 * (vc - R) ** 2).sum() / n
    return lpi + value_coef * lv - entropy_coef * ent.sum() / n


def _branchy_inputs(n, rng, clip=0.2, value_clip=0.2):
    """logp / values and loss inputs with every branch populated: rho below, inside and above the clip range
    with Abar of both signs, values inside and beyond the value clip on both sides."""
    logp, ent, v = rng.normal(-1.5, 0.5, n), rng.uniform(0.5, 1.5, n), rng.normal(0, 1, (n, 2))
    rho = rng.choice([0.5, 0.7, 0.9, 1.0, 1.1, 1.3, 1.6], n) * rng.uniform(0.97, 1.03, n)
    old_logp = logp - np.log(rho)
    delta = rng.choice([-3, -1.5, -0.5, 0.5, 1.5, 3], (n, 2)) * value_clip * rng.uniform(0.9, 1.1, (n, 2))
    old_v = v - delta
    R = v + rng.normal(0, 0.5, (n, 2))
    A = rng.normal(0, 1, (n, 2))
    return logp, ent, v, old_logp, old_v, R, A


def test_oracle_seeds_equal_autograd_of_the_formula():
    rng = np.random.default_rng(0)
    n = 4000
    logp, ent, v, old_logp, old_v, R, A = _branchy_inputs(n, rng)
    mom, lam = O.adv_moments(A), 0.7
    d_logp, d_ent, d_v, st, rho, abar = O.seeds(logp, ent, v, old_logp, old_v, R, A, mom, lam, **COEFS)
    # every branch is populated
    for lo in (True, False):
        for pos in (True, False):
            sel = (rho < 0.8 if lo else rho > 1.2) & ((abar > 0) == pos)
            assert sel.sum() > 50
    vc_side = v - old_v
    assert (vc_side > 0.2).sum() > 100 and (vc_side < -0.2).sum() > 100 and (np.abs(vc_side) < 0.2).sum() > 100
    assert (d_logp == 0).sum() > 100 and (d_v == 0).sum() > 100
    t = [torch.tensor(x, dtype=torch.float64, requires_grad=i < 3) for i, x in
         enumerate((logp, ent, v, old_logp, old_v, R, A))]
    loss = _torch_loss(*t, torch.tensor(mom), lam, **COEFS)
    loss.backward()
    np.testing.assert_allclose(t[0].grad.numpy(), d_logp, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(t[1].grad.numpy(), d_ent, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(t[2].grad.numpy(), d_v, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(float(loss), st[7], rtol=1e-12)
    assert st[5] == (np.abs(rho - 1) > 0.2).mean()


# ---- the C ABI (CPU) ---------------------------------------------------------------------------------------
def test_loss_io_mirror_matches_the_header_as_compiled_by_gcc(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    fields = [f for f, _ in abi.GsmPpoLossIO._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "gsmarl_b200.h"', 'int main(void) {',
             '  printf("sizeof %zu\\n", sizeof(gsm_ppo_loss_io));',
             '  printf("fields %d\\n", GSM_PPO_STAT_FIELDS);']
    lines += [f'  printf("{f} %zu\\n", offsetof(gsm_ppo_loss_io, {f}));' for f in fields]
    lines += ['  return 0;', '}']
    src = tmp_path / "ppo_layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "ppo_layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o",
                    str(exe)], check=True)
    got = dict(ln.split() for ln in subprocess.run([str(exe)], capture_output=True, text=True,
                                                   check=True).stdout.splitlines())
    assert int(got["sizeof"]) == C.sizeof(abi.GsmPpoLossIO)
    assert int(got["fields"]) == abi.GSM_PPO_STAT_FIELDS == len(STAT_FIELDS) - 1
    for f in fields:
        assert int(got[f]) == getattr(abi.GsmPpoLossIO, f).offset, f


def _host_ios(gauss=False, R=10, K=3):
    """Valid eval and loss ios over HOST arrays: every argument check returns before a pointer is dereferenced."""
    a = {"params": np.zeros(2380, np.float32), "obs": np.zeros((R, 6), np.float32),
         "feat": np.zeros((R, K, 6), np.float32), "cnt": np.zeros(R, np.int32),
         "act": np.zeros((R, 2), np.float32) if gauss else np.zeros(R, np.int32),
         "old_logp": np.zeros(R, np.float32), "old_v": np.zeros((R, 2), np.float32), "ret": np.zeros((R, 2), np.float32),
         "adv": np.zeros((R, 2), np.float32), "mom": np.zeros(4, np.float32), "lam": np.zeros(1, np.float32),
         "stats": np.full(8, 7.0, np.float32), "grad": np.full(2380, 7.0, np.float32)}
    io = (abi.GsmPolicyGaussEvalIO if gauss else abi.GsmPolicyEvalIO)()
    io.struct_size = C.sizeof(type(io))
    if gauss:
        io.action_dim = 2
    else:
        io.n_actions = 5
    io.params, io.obs, io.nbr_feat = a["params"].ctypes.data, a["obs"].ctypes.data, a["feat"].ctypes.data
    io.nbr_cnt, io.actions = a["cnt"].ctypes.data, a["act"].ctypes.data
    io.n_rows, io.max_nbrs = R, K
    loss = abi.GsmPpoLossIO()
    loss.struct_size = C.sizeof(abi.GsmPpoLossIO)
    for f, k in (("old_logp", "old_logp"), ("old_values", "old_v"), ("returns", "ret"), ("advantages", "adv"),
                 ("adv_moments", "mom"), ("lagrange", "lam"), ("stats", "stats")):
        setattr(loss, f, a[k].ctypes.data)
    for k, v in COEFS.items():
        setattr(loss, k, v)
    return io, loss, a


@pytest.mark.parametrize("gauss", [False, True])
def test_ppo_backward_invalid_arguments_return_their_status(gauss):
    lib = abi.load_library()
    fn = lib.gsm_ppo_backward_gauss if gauss else lib.gsm_ppo_backward
    need = lib.gsm_ppo_backward_workspace_gauss(10) if gauss else lib.gsm_ppo_backward_workspace(10, 5)
    assert need > 0
    assert lib.gsm_ppo_backward_workspace(-1, 5) == -1 and lib.gsm_ppo_backward_workspace(10, 7) == -4
    assert lib.gsm_ppo_backward_workspace_gauss(-1) == -1
    ws = np.zeros(need, np.uint8)

    def status(mutate_loss=lambda l: None, mutate_io=lambda io: None, n_bytes=need, workspace=ws.ctypes.data,
               grad=True):
        io, loss, a = _host_ios(gauss)
        mutate_loss(loss)
        mutate_io(io)
        return fn(C.byref(io), C.byref(loss), C.c_void_p(a["grad"].ctypes.data if grad else None),
                  C.c_void_p(workspace), n_bytes, 0, None)
    assert status(lambda l: setattr(l, "struct_size", 8)) == -3
    assert status(mutate_io=lambda io: setattr(io, "struct_size", 8)) == -3
    for f in ("old_logp", "old_values", "returns", "advantages", "adv_moments", "lagrange", "stats"):
        assert status(lambda l: setattr(l, f, None)) == -1, f
    for f, v in (("clip", 0.0), ("clip", -0.1), ("value_clip", 0.0), ("value_coef", -1.0), ("entropy_coef", -1e-3),
                 ("clip", float("nan"))):
        assert status(lambda l: setattr(l, f, v)) == -1, (f, v)
    assert status(grad=False) == -1
    assert status(n_bytes=need - 1) == -1
    assert status(workspace=None) == -1
    assert status(mutate_io=lambda io: setattr(io, "params", None)) == -1
    io, _, a = _host_ios(gauss)
    assert fn(C.byref(io), None, C.c_void_p(a["grad"].ctypes.data), C.c_void_p(ws.ctypes.data), need, 0, None) == -1
    # n_rows == 0 is a no-op: grad and stats untouched
    io, loss, a = _host_ios(gauss)
    io.n_rows = 0
    assert fn(C.byref(io), C.byref(loss), C.c_void_p(a["grad"].ctypes.data), None, 0, 0, None) == 0
    assert (a["grad"] == 7).all() and (a["stats"] == 7).all()


def test_adam_invalid_arguments_return_their_status():
    lib = abi.load_library()
    bufs = [np.zeros(16, np.float32) for _ in range(5)]
    step = np.zeros(1, np.int32)
    good = dict(params=bufs[0].ctypes.data, grad=bufs[1].ctypes.data, m=bufs[2].ctypes.data, v=bufs[3].ctypes.data,
                step=step.ctypes.data, n=16, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, max_grad_norm=1.0,
                grad_norm=bufs[4].ctypes.data)

    def status(**kw):
        a = dict(good, **kw)
        return lib.gsm_adam_step(*(C.c_void_p(a[k]) for k in ("params", "grad", "m", "v", "step")), a["n"], a["lr"],
                                 a["beta1"], a["beta2"], a["eps"], a["max_grad_norm"], C.c_void_p(a["grad_norm"]), 0, None)
    for k in ("params", "grad", "m", "v", "step", "grad_norm"):
        assert status(**{k: None}) == -1, k
    for kw in ({"n": 0}, {"n": -5}, {"beta1": 1.0}, {"beta1": -0.1}, {"beta2": 1.0}, {"beta2": float("nan")},
               {"lr": -1.0}, {"eps": -1.0}, {"max_grad_norm": 0.0}):
        assert status(**kw) == -1, kw
    assert step[0] == 0 and (bufs[0] == 0).all()


def test_trainer_requires_every_hyper_parameter():
    actor = GraphAttentionActor(5, seed=0)
    hp = dict(HP)
    for k in ("clip", "value_clip", "value_coef", "entropy_coef", "lr", "betas", "eps", "max_grad_norm", "ppo_epoch",
              "num_mini_batch", "lagrangian_lr", "cost_limit", "seed"):
        kw = {q: v for q, v in hp.items() if q != k}
        with pytest.raises(TypeError):
            LagrangianPPO(actor, **kw)
    with pytest.raises(TypeError):
        LagrangianPPO(torch.nn.Linear(2, 2), **hp)
    with pytest.raises(ValueError):
        LagrangianPPO(actor, **dict(hp, clip=0.0))
    with pytest.raises(ValueError):
        LagrangianPPO(actor, **dict(hp, betas=(1.0, 0.999)))
    with pytest.raises(abi.GsmError):                 # parameters on the CPU: no fallback
        LagrangianPPO(actor, **hp)


def test_trainer_rejects_a_buffer_without_returns():
    trainer = LagrangianPPO.__new__(LagrangianPPO)     # the input check runs before anything touches a device
    trainer._act_dtype, trainer._act_tail = torch.int32, ()
    buf = {"obs": torch.zeros(3, 4, 6), "nbr_feat": torch.zeros(3, 4, 2, 6), "nbr_cnt": torch.zeros(3, 4, dtype=torch.int32),
           "actions": torch.zeros(2, 4, dtype=torch.int32), "logp": torch.zeros(2, 4), "values": torch.zeros(3, 4, 2)}
    with pytest.raises(ValueError, match="compute_returns"):
        trainer.inputs(buf)
    with pytest.raises(ValueError, match="compute_returns"):
        trainer.update(buf)


# ---- GPU: the fused gradient against the fp64 oracle ---------------------------------------------------
def _synthetic(actor, R, K, seed, clip=0.2, value_clip=0.2):
    """One-slot buffer dict with loss inputs placed so that no row lies within 1e-3 of a branch edge (fp32 and
    fp64 take the same branches), plus the fp64 oracle module and weights."""
    rng = np.random.default_rng(seed)
    gauss = isinstance(actor, GaussianGraphActor)
    obs = rng.normal(0, 1, (R, 6)).astype(np.float32)
    feat = rng.normal(0, 1, (R, K, 6)).astype(np.float32)
    cnt = rng.integers(0, K + 1, R).astype(np.int32)
    cnt[0], cnt[-1] = K, 0
    feat[np.arange(K)[None, :] >= cnt[:, None]] = 0
    if gauss:
        mod, w = G, G.weights_from_state_dict(actor.state_dict())
        act = rng.normal(0, 1.5, (R, 2)).astype(np.float32)
    else:
        mod, w = L, P.weights_from_state_dict(actor.state_dict(), np.float64)
        act = rng.integers(0, actor.n_actions, R).astype(np.int32)
    logp, ent, v = mod.evaluate(w, obs, feat, cnt, act)
    rho = rng.choice([0.6, 0.9, 1.0, 1.1, 1.4], R) * rng.uniform(0.98, 1.02, R)
    rho = np.where(np.abs(np.abs(rho - 1) - clip) < 2e-3, rho + 5e-3, rho)
    old_logp = (logp - np.log(rho)).astype(np.float32)
    delta = rng.choice([-2.0, -0.5, 0.5, 2.0], (R, 2)) * value_clip
    old_v = (v - delta).astype(np.float32)
    c = np.clip(delta, -value_clip, value_clip) - delta              # vc - v
    e1 = rng.normal(0, 0.5, (R, 2))
    e1 = np.where((c != 0) & (np.abs(2 * e1 + c) < 0.05), e1 + 0.2, e1)   # (v-R)^2 vs (vc-R)^2 well apart
    ret = (v - e1).astype(np.float32)
    adv = rng.normal(0, 1, (R, 2)).astype(np.float32)
    mom = np.array([0.1, 1.3, -0.2, 0.7], np.float32)
    lam = np.float32(0.5)
    abar = (adv[:, 0] - mom[0]) / (mom[1] + 1e-5) - lam * (adv[:, 1] - mom[2]) / (mom[3] + 1e-5)
    adv[:, 0] = np.where(np.abs(abar) < 1e-2, adv[:, 0] + 0.1, adv[:, 0])
    d = {k: torch.from_numpy(np.ascontiguousarray(x))[None].to(DEV) for k, x in
         dict(obs=obs, nbr_feat=feat, nbr_cnt=cnt, actions=act, logp=old_logp, values=old_v, returns=ret,
              advantages=adv).items()}
    host = dict(obs=obs, feat=feat, cnt=cnt, act=act, old_logp=old_logp, old_v=old_v, R=ret, A=adv,
                moments=mom.astype(np.float64), lam=float(lam))
    return d, host, mod, w


def _trainer(actor, **kw):
    return LagrangianPPO(actor, **dict(HP, **COEFS, **kw))


def _fused(trainer, d, mom, lam, rows=None):
    trainer.adv_moments.copy_(torch.tensor(mom, dtype=torch.float32))
    trainer.lagrange.fill_(lam)
    stats = torch.full((8,), float("nan"), device=DEV)
    trainer.backward(trainer.inputs(d), rows, stats)
    return trainer.grad.double().cpu().numpy(), stats.double().cpu().numpy()


def _assert_grad_close(got, want, split, bar=1e-4):
    g, w = split(got), split(want)
    bad = []
    for k in g:
        scale = np.linalg.norm(w["att_w" if k == "att_b" else k])
        err = np.linalg.norm(np.asarray(g[k]) - np.asarray(w[k]))
        if not err <= bar * scale:
            bad.append((k, err, scale))
    assert not bad, bad


def _make_actor(kind, seed):
    return (GaussianGraphActor(seed=seed) if kind == "gauss" else GraphAttentionActor(kind, seed=seed)).to(DEV)


@gpu
@pytest.mark.parametrize("kind", [5, 9, "gauss"])
@pytest.mark.parametrize("shuffled", [False, True])
def test_fused_gradient_matches_fp64_oracle(kind, shuffled):
    R, K = 4099, 7
    actor = _make_actor(kind, seed=3)
    d, h, mod, w = _synthetic(actor, R, K, seed=11)
    split = G.split_vector if kind == "gauss" else (lambda v: L.split_vector(v, kind))
    rows = np.random.default_rng(5).permutation(R)[:3001] if shuffled else None
    trainer = _trainer(actor)
    got, st = _fused(trainer, d, h["moments"], h["lam"], None if rows is None else torch.from_numpy(rows).to(DEV))
    want, st0, ex = O.loss_grad(mod, w, h["obs"], h["feat"], h["cnt"], h["act"], h["old_logp"], h["old_v"], h["R"],
                                h["A"], h["moments"], h["lam"], rows=rows, **COEFS)
    assert (ex["d_logp"] == 0).any() and (ex["d_logp"] != 0).any() and (ex["d_v"] == 0).any()
    _assert_grad_close(got, want, split)
    n = len(ex["rho"])
    assert st[5] == np.float32(np.float32((np.abs(ex["rho"] - 1) > 0.2).sum()) / np.float32(n))
    np.testing.assert_allclose(st, st0, rtol=1e-4, atol=1e-6)
    got2, st2 = _fused(trainer, d, h["moments"], h["lam"], None if rows is None else torch.from_numpy(rows).to(DEV))
    assert np.array_equal(got, got2) and np.array_equal(st, st2)


def _nav3_buffer(B=1024, T=8, sharded=False, seed=3, gauss=False):
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv, StreamShardedEnv
    from gs_marl_b200.rollout import GraphRolloutBuffer
    kw = {"action_mode": "continuous"} if gauss else {}
    cfg = make_cfg("navigation", 3, "f32", episode_length=25, **kw)
    env = (StreamShardedEnv(cfg, B, n_streams=4, auto_reset=True, seed=seed) if sharded
           else MultiAgentGraphConstrainEnv(cfg, B, auto_reset=True, seed=seed))
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    return env, buf


def _rollout(env, actor, buf, it):
    from gs_marl_b200.rollout import collect_fused
    collect_fused(env, actor, buf, seed=17, first_step=it * buf.T)
    g = buf.graph(buf.T)
    buf["values"][buf.T] = actor.act(buf["obs"][buf.T], g, seed=0, greedy=True, want_values=True)[-1]
    buf.compute_returns(0.99, 0.95)


@gpu
def test_collected_rollout_matches_evaluate_actions_and_autograd():
    env, buf = _nav3_buffer()
    actor = GraphAttentionActor(5, seed=2).to(DEV)
    _rollout(env, actor, buf, 0)
    trainer = _trainer(actor)
    x = trainer.inputs(buf)
    trainer.set_advantage_moments(x["adv"])
    trainer.lagrange.fill_(0.3)
    rows = torch.randperm(x["cnt"].numel(), generator=torch.Generator(device=DEV).manual_seed(1), device=DEV)[:2000]
    stats = torch.zeros(8, device=DEV)
    trainer.backward(x, rows, stats)
    st = stats.cpu().numpy()
    assert st[4] == 1.0 and st[5] == 0.0 and st[6] == 0.0          # first epoch: rho is exactly 1
    # the composition the fused kernel replaces
    actor.zero_grad(set_to_none=True)
    lp, ent, v = actor.evaluate_actions(x["obs"], {"nbr_feat": x["feat"], "nbr_cnt": x["cnt"]}, x["act"], rows=rows)
    mom = trainer.adv_moments
    loss = _torch_loss(lp, ent, v, x["old_logp"][rows], x["old_v"][rows], x["ret"][rows], x["adv"][rows], mom, 0.3,
                       **COEFS)
    loss.backward()
    ref = torch.nn.utils.parameters_to_vector([p.grad for p in actor.parameters()]).double().cpu().numpy()
    _assert_grad_close(trainer.grad.double().cpu().numpy(), ref, lambda q: L.split_vector(q, 5), bar=1e-5)
    np.testing.assert_allclose(st[7], float(loss.detach()), rtol=1e-5)
    env.close()


# ---- GPU: Adam ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("max_norm", [0.05, 1e3])
def test_adam_matches_torch_over_20_steps(max_norm):
    lib = abi.load_library()
    n = 2380
    g = torch.Generator().manual_seed(0)
    p0 = torch.randn(n, generator=g, dtype=torch.float64)
    grads = [torch.randn(n, generator=g, dtype=torch.float64).float().double() * 0.01 for _ in range(20)]
    ref = torch.nn.Parameter(p0.clone())
    f32 = lambda x: float(np.float32(x))                  # the ABI's hyper-parameters are fp32
    opt = torch.optim.Adam([ref], lr=f32(5e-3), betas=(f32(0.9), f32(0.999)), eps=f32(1e-5))
    p, m, v = p0.float().to(DEV), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    step, norm = torch.zeros(1, dtype=torch.int32, device=DEV), torch.zeros(1, device=DEV)
    norms = []
    for gr in grads:
        ref.grad = gr.clone()
        nref = float(torch.nn.utils.clip_grad_norm_([ref], max_norm))
        opt.step()
        gd = gr.float().to(DEV)
        assert lib.gsm_adam_step(p.data_ptr(), gd.data_ptr(), m.data_ptr(), v.data_ptr(), step.data_ptr(), n, 5e-3,
                                 0.9, 0.999, 1e-5, max_norm, norm.data_ptr(), 0, None) == 0
        np.testing.assert_allclose(float(norm), nref, rtol=1e-6)
        norms.append(nref)
    assert (min(norms) > max_norm) if max_norm < 1 else (max(norms) < max_norm)
    np.testing.assert_allclose(p.double().cpu().numpy(), ref.detach().numpy(), rtol=1e-5, atol=1e-7)
    st = opt.state[ref]
    np.testing.assert_allclose(m.double().cpu().numpy(), st["exp_avg"].numpy(), rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(v.double().cpu().numpy(), st["exp_avg_sq"].numpy(), rtol=1e-5, atol=1e-12)
    assert int(step) == 20


@gpu
def test_adam_skips_a_non_finite_gradient():
    lib = abi.load_library()
    n = 1864
    p, m, v = (torch.randn(n, device=DEV) for _ in range(3))
    v = v.abs()
    step = torch.full((1,), 7, dtype=torch.int32, device=DEV)
    norm = torch.zeros(1, device=DEV)
    before = [t.clone() for t in (p, m, v, step)]
    for bad in (float("nan"), float("inf")):
        gd = torch.randn(n, device=DEV)
        gd[100] = bad
        assert lib.gsm_adam_step(p.data_ptr(), gd.data_ptr(), m.data_ptr(), v.data_ptr(), step.data_ptr(), n, 1e-3,
                                 0.9, 0.999, 1e-8, 1.0, norm.data_ptr(), 0, None) == 0
        assert not torch.isfinite(norm).all()
        for a, b in zip((p, m, v, step), before):
            assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a,
                               b.view(torch.int32) if b.dtype == torch.float32 else b)


# ---- GPU: determinism, capture, sync-free update, guard bands ------------------------------------------
@gpu
def test_two_trainers_are_bit_identical_across_streams():
    env, buf = _nav3_buffer()
    actor = GraphAttentionActor(5, seed=4).to(DEV)
    _rollout(env, actor, buf, 0)
    res = []
    for s in (torch.cuda.current_stream(), torch.cuda.Stream()):
        a = GraphAttentionActor(5, seed=4).to(DEV)
        tr = LagrangianPPO(a, **dict(HP, ppo_epoch=2, num_mini_batch=3))
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            out = tr.update(buf)
        torch.cuda.synchronize()
        res.append((out.cpu(), tr.params.cpu(), tr.m.cpu(), tr.v.cpu(), int(tr.step)))
    (o1, p1, m1, v1, t1), (o2, p2, m2, v2, t2) = res
    assert torch.equal(o1, o2) and torch.equal(p1, p2) and torch.equal(m1, m2) and torch.equal(v1, v2) and t1 == t2 == 6
    assert torch.isfinite(o1).all()
    env.close()


@gpu
def test_captured_minibatch_step_replays_bit_identical_to_eager():
    env, buf = _nav3_buffer()
    actor = GraphAttentionActor(5, seed=6).to(DEV)
    _rollout(env, actor, buf, 0)
    tr = LagrangianPPO(actor, **HP)
    x = tr.inputs(buf)
    tr.set_advantage_moments(x["adv"])
    rows = torch.randperm(x["cnt"].numel(), device=DEV)[:5000]
    saved = [t.clone() for t in (tr.params, tr.m, tr.v, tr.step)]
    eager = torch.zeros(9, device=DEV)
    tr.minibatch_step(x, rows, eager)                      # also allocates the workspace before the capture
    want = [t.clone() for t in (tr.params, tr.m, tr.v, tr.step)]
    for t, s in zip((tr.params, tr.m, tr.v, tr.step), saved):
        t.copy_(s)
    torch.cuda.synchronize()
    cap = torch.zeros(9, device=DEV)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        tr.minibatch_step(x, rows, cap)
    for t, s in zip((tr.params, tr.m, tr.v, tr.step), saved):
        t.copy_(s)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(cap, eager)
    for t, w in zip((tr.params, tr.m, tr.v, tr.step), want):
        assert torch.equal(t, w)
    env.close()


@gpu
@pytest.mark.parametrize("kind", [5, "gauss"])
def test_update_makes_no_host_sync(kind):
    env, buf = _nav3_buffer(gauss=kind == "gauss")
    actor = _make_actor(kind, seed=1)
    _rollout(env, actor, buf, 0)
    tr = LagrangianPPO(actor, **dict(HP, ppo_epoch=2, num_mini_batch=2))
    tr.update(buf)                                          # first call: workspace allocation, module load
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = tr.update(buf)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert out.shape == (4, len(STAT_FIELDS)) and torch.isfinite(out).all()
    env.close()


@gpu
def test_guard_bands_stay_untouched():
    actor = GraphAttentionActor(5, seed=8).to(DEV)
    d, h, _, _ = _synthetic(actor, 2000, 5, seed=2)
    tr = _trainer(actor)
    GB = 1024                                                  # 4 KB of float32 on each side
    sentinel = 12345.0

    def banded(t):
        big = torch.full((t.numel() + 2 * GB,), sentinel, dtype=t.dtype, device=DEV)
        big[GB:GB + t.numel()] = t.reshape(-1)
        return big, big[GB:GB + t.numel()].view_as(t)
    bands = {}
    for k in ("params", "grad", "m", "v"):
        bands[k], view = banded(getattr(tr, k))
        setattr(tr, k, view)
    stats_big, stats = banded(torch.zeros(9, device=DEV))
    need = abi.load_library().gsm_ppo_backward_workspace(2000, 5)
    ws_big = torch.full((need + 8 * GB,), 0x5A, dtype=torch.uint8, device=DEV)
    tr._ws = ws_big[4 * GB:4 * GB + need]
    tr.adv_moments.copy_(torch.tensor(h["moments"], dtype=torch.float32))
    tr.minibatch_step(tr.inputs(d), None, stats)
    torch.cuda.synchronize()
    for k, big in list(bands.items()) + [("stats", stats_big)]:
        assert (big[:GB] == sentinel).all() and (big[-GB:] == sentinel).all(), k
    assert (ws_big[:4 * GB] == 0x5A).all() and (ws_big[-4 * GB:] == 0x5A).all()
    assert torch.isfinite(stats).all() and int(tr.step) == 1


@gpu
def test_update_lagrange_rule():
    actor = GraphAttentionActor(5, seed=0).to(DEV)
    tr = LagrangianPPO(actor, **dict(HP, lagrangian_lr=0.05, cost_limit=2.0, lagrangian_init=1.0))
    tot = torch.zeros(16, dtype=torch.float64, device=DEV)
    tot[8], tot[11] = 4.0, 20.0                               # team cost mean 5: gap 3
    tr.update_lagrange(tot)
    assert float(tr.lagrange) == np.float32(1.0 + 0.05 * 3.0)
    tot[11] = 0.0                                             # gap -2, 50 times: clamped at 0
    for _ in range(50):
        tr.update_lagrange(tot)
    assert float(tr.lagrange) == 0.0
    tr.lagrange.fill_(0.75)
    tr.update_lagrange(torch.zeros(16, dtype=torch.float64, device=DEV))   # no team episode: unchanged
    assert float(tr.lagrange) == 0.75


@gpu
@pytest.mark.parametrize("sharded", [False, True])
def test_three_iteration_training_loop(sharded):
    from gs_marl_b200.episodes import EpisodeTracker
    env, buf = _nav3_buffer(B=2048, T=25, sharded=sharded)
    actor = GraphAttentionActor(5, seed=9).to(DEV)
    p0 = torch.nn.utils.parameters_to_vector(actor.parameters()).detach().clone()
    tr = LagrangianPPO(actor, **dict(HP, ppo_epoch=2, num_mini_batch=4, lagrangian_lr=0.1, cost_limit=0.0))
    tracker = EpisodeTracker(env, agent_cost_limit=0.0, team_cost_limit=0.0)
    tracker.reset()
    outs = []
    for it in range(3):
        _rollout(env, actor, buf, it)
        totals = tracker.update(buf["reward"], buf["cost"], buf["done"])
        outs.append(tr.update(buf))
        tr.update_lagrange(totals)
        actor.pack()
        buf.after_update()
    torch.cuda.synchronize()
    out = torch.cat(outs)
    assert torch.isfinite(out).all() and int(tr.step) == 24
    p1 = torch.nn.utils.parameters_to_vector(actor.parameters()).detach()
    assert torch.isfinite(p1).all() and not torch.equal(p0, p1)
    assert torch.equal(p1, tr.params)
    assert float(tr.lagrange) >= 0
    sd = tr.state_dict()
    tr2 = LagrangianPPO(GraphAttentionActor(5, seed=1).to(DEV), **HP)
    tr2.load_state_dict(sd)
    assert torch.equal(tr2.params, tr.params) and torch.equal(tr2.v, tr.v) and int(tr2.step) == 24
    env.close()
