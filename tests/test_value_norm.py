"""The value normaliser (SPEC.md §15): `gsm_value_norm_update`, `gsm_gae_normalized`,
`gsm_ppo_backward_normalized(_gauss)`, `learner.ValueNorm` and `LagrangianPPO(value_norm=...)` against the
float64 restatement in tests/_value_norm_oracle.py and torch autograd."""
import ctypes as C
import os
import shutil
import subprocess
from fractions import Fraction

import numpy as np
import pytest
import torch

from gs_marl_b200 import abi, presets
from gs_marl_b200.learner import LagrangianPPO, ValueNorm
from gs_marl_b200.policy import GraphAttentionActor
from tests import _gauss_oracle as G
from tests import _learner_oracle as L
from tests import _ppo_oracle as O
from tests import _value_norm_oracle as VO
from tests._util import make_cfg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
DEV = "cuda"
COEFS = dict(clip=0.2, value_clip=0.2, value_coef=0.5, entropy_coef=0.01)
HP = dict(presets.UNVERIFIED_PPO_LAG, value_coef=0.5, seed=0)
VN = presets.UNVERIFIED_VALUE_NORM
AFFINE = np.array([[0.75, 2.5], [-0.4, 0.6]], np.float32)     # (mu_h, sigma_h) of a used normaliser


# ---- the oracle against torch autograd of the §15 + §14 formula (CPU) -----------------------------------
def test_oracle_seeds_on_normalised_targets_equal_autograd_of_the_formula():
    rng = np.random.default_rng(1)
    n = 4000
    logp, ent, v = rng.normal(-1.5, 0.5, n), rng.uniform(0.5, 1.5, n), rng.normal(0, 1, (n, 2))
    old_logp = logp - np.log(rng.choice([0.6, 0.9, 1.0, 1.1, 1.4], n))
    old_v = v - rng.choice([-2.0, -0.5, 0.5, 2.0], (n, 2)) * 0.2
    Rn = v + rng.normal(0, 0.5, (n, 2))
    R = Rn * AFFINE[:, 1] + AFFINE[:, 0]                         # raw returns
    A = rng.normal(0, 1, (n, 2))
    mom, lam = O.adv_moments(A), 0.4
    d_logp, d_ent, d_v, st, _, _ = O.seeds(logp, ent, v, old_logp, old_v, VO.normalize(R, AFFINE), A, mom, lam,
                                           **COEFS)
    assert (d_v == 0).sum() > 100 and (d_v != 0).sum() > 100
    t = [torch.tensor(x, dtype=torch.float64, requires_grad=i < 3) for i, x in
         enumerate((logp, ent, v, old_logp, old_v, R, A))]
    aff = torch.tensor(AFFINE, dtype=torch.float64)
    mu, sd = aff[:, 0], aff[:, 1]
    m = torch.tensor(mom)
    abar = (t[6][:, 0] - m[0]) / (m[1] + 1e-5) - lam * (t[6][:, 1] - m[2]) / (m[3] + 1e-5)
    rho = torch.exp(t[0] - t[3])
    lpi = -torch.min(rho * abar, torch.clamp(rho, 0.8, 1.2) * abar).sum() / n
    target = (t[5] - mu) / sd                                    # §15: normalize(R)
    vc = t[4] + torch.clamp(t[2] - t[4], -0.2, 0.2)
    lv = torch.max(0.5 * (t[2] - target) ** 2, 0.5 * (vc - target) ** 2).sum() / n
    loss = lpi + COEFS["value_coef"] * lv - COEFS["entropy_coef"] * t[1].sum() / n
    loss.backward()
    np.testing.assert_allclose(t[0].grad.numpy(), d_logp, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(t[1].grad.numpy(), d_ent, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(t[2].grad.numpy(), d_v, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(float(loss.detach()), st[7], rtol=1e-12)


def test_oracle_value_norm_is_the_lineage_formula():
    vn = VO.ValueNorm64(**VN)
    np.testing.assert_array_equal(vn.affine(), [[0.0, 0.1], [0.0, 0.1]])     # a fresh normaliser: sigma 0.1
    R = np.random.default_rng(0).normal([3.0, 1.0], [2.0, 0.5], (1000, 2))
    vn.update(R)
    w = 1 - VN["beta"]
    np.testing.assert_allclose(vn.state[:, 0], w * R.mean(0), rtol=1e-14)
    np.testing.assert_allclose(vn.affine()[:, 0], R.mean(0), rtol=1e-9)           # debiased
    np.testing.assert_allclose(vn.affine()[:, 1], R.std(0), rtol=1e-7)


# ---- the C ABI (CPU) ---------------------------------------------------------------------------------------
def test_value_norm_io_mirror_matches_the_header_as_compiled_by_gcc(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    fields = [f for f, _ in abi.GsmValueNormIO._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "gsmarl_b200.h"', 'int main(void) {',
             '  printf("sizeof %zu\\n", sizeof(gsm_value_norm_io));', '  printf("abi %d\\n", GSM_ABI_VERSION);']
    lines += [f'  printf("{f} %zu\\n", offsetof(gsm_value_norm_io, {f}));' for f in fields]
    lines += ['  return 0;', '}']
    src = tmp_path / "vn_layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "vn_layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o",
                    str(exe)], check=True)
    got = dict(ln.split() for ln in subprocess.run([str(exe)], capture_output=True, text=True,
                                                   check=True).stdout.splitlines())
    assert int(got["sizeof"]) == C.sizeof(abi.GsmValueNormIO)
    assert int(got["abi"]) == abi.GSM_ABI_VERSION == 8
    for f in fields:
        assert int(got[f]) == getattr(abi.GsmValueNormIO, f).offset, f


def _host_vn_io(R=64, nmb=2):
    a = {"state": np.zeros(6), "affine": np.full((nmb + 1) * 4, 7.0, np.float32), "ret": np.zeros((R, 2), np.float32),
         "rows": np.arange(R, dtype=np.int64)}
    io = abi.GsmValueNormIO()
    io.struct_size = C.sizeof(abi.GsmValueNormIO)
    io.state, io.affine = a["state"].ctypes.data, a["affine"].ctypes.data
    io.returns, io.rows = a["ret"].ctypes.data, a["rows"].ctypes.data
    io.mb, io.n_mini_batch = R // nmb, nmb
    io.beta, io.epsilon, io.var_floor = VN["beta"], VN["epsilon"], VN["var_floor"]
    return io, a


def test_value_norm_update_invalid_arguments_return_their_status():
    lib = abi.load_library()
    need = lib.gsm_value_norm_update_workspace(32, 2)
    assert need > 0
    for mb, nmb in ((0, 2), (32, 0), (-1, 1), (1, -3)):
        assert lib.gsm_value_norm_update_workspace(mb, nmb) == -1, (mb, nmb)
    ws = np.zeros(need, np.uint8)

    def status(mutate=lambda io: None, n_bytes=need, workspace=ws.ctypes.data):
        io, a = _host_vn_io()
        mutate(io)
        st = lib.gsm_value_norm_update(C.byref(io), C.c_void_p(workspace), n_bytes, 0, None)
        assert (a["state"] == 0).all() and (a["affine"] == 7).all()     # nothing was touched
        return st
    assert lib.gsm_value_norm_update(None, C.c_void_p(ws.ctypes.data), need, 0, None) == -1
    assert status(lambda io: setattr(io, "struct_size", 8)) == -3
    for f in ("state", "affine", "returns", "rows"):
        assert status(lambda io: setattr(io, f, None)) == -1, f
    for f, v in (("beta", 1.0), ("beta", -0.1), ("beta", float("nan")), ("epsilon", 0.0), ("epsilon", -1e-5),
                 ("var_floor", 0.0), ("var_floor", float("nan")), ("mb", 0), ("n_mini_batch", 0)):
        assert status(lambda io: setattr(io, f, v)) == -1, (f, v)
    assert status(n_bytes=need - 1) == -1
    assert status(workspace=None) == -1


def test_normalized_entry_points_require_the_affine():
    lib = abi.load_library()
    f = np.zeros(64, np.float32)
    d = np.zeros(64, np.uint8)
    p = lambda x: C.c_void_p(x.ctypes.data)
    assert lib.gsm_gae_normalized(p(f), p(f), p(f), p(d), 2, 4, 4, 0.99, 0.95, p(f), p(f), None, 0, None) == -1
    assert "value_affine" in lib.gsm_policy_last_error().decode()
    from tests.test_ppo_update import _host_ios
    for gauss in (False, True):
        fn = lib.gsm_ppo_backward_normalized_gauss if gauss else lib.gsm_ppo_backward_normalized
        need = lib.gsm_ppo_backward_workspace_gauss(10) if gauss else lib.gsm_ppo_backward_workspace(10, 5)
        ws = np.zeros(need, np.uint8)
        io, loss, a = _host_ios(gauss)
        assert fn(C.byref(io), C.byref(loss), None, p(a["grad"]), p(ws), need, 0, None) == -1
        assert "value_affine" in lib.gsm_policy_last_error().decode()
        loss.struct_size = 8
        assert fn(C.byref(io), C.byref(loss), p(f), p(a["grad"]), p(ws), need, 0, None) == -3
        assert (a["grad"] == 7).all()


def test_value_norm_requires_its_hyper_parameters():
    for k in VN:
        with pytest.raises(TypeError):
            ValueNorm("cuda", **{q: v for q, v in VN.items() if q != k})
    for bad in (dict(beta=1.0), dict(beta=-0.5), dict(epsilon=0.0), dict(var_floor=-1.0)):
        with pytest.raises(ValueError):
            ValueNorm("cuda", **dict(VN, **bad))
    with pytest.raises(abi.GsmError):                 # no CPU fallback
        ValueNorm("cpu", **VN)


# ---- GPU: the normaliser against the float64 ValueNorm ----------------------------------------------------
def _ulps(got, want):
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    return np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))


def _returns(n, seed):
    rng = np.random.default_rng(seed)
    R = np.stack([rng.normal(5.0, 3.0, n), rng.exponential(0.7, n)], 1).astype(np.float32)
    return R, torch.from_numpy(R).to(DEV)


@gpu
@pytest.mark.parametrize("beta", [VN["beta"], 0.9])
def test_update_matches_the_float64_value_norm(beta):
    n, nmb = 3 * 51_000 + 2, 3                                # 3 x 51 000 rows (25 blocks each) + a remainder of 2
    R, Rd = _returns(n, 0)
    vn = ValueNorm(DEV, beta=beta, epsilon=VN["epsilon"], var_floor=VN["var_floor"])
    ref = VO.ValueNorm64(beta, VN["epsilon"], VN["var_floor"])
    assert torch.equal(vn.affine.cpu(), torch.tensor([[0.0, np.float32(0.1)]] * 2))
    g = torch.Generator(device=DEV).manual_seed(3)
    for ep in range(4):
        perm = torch.randperm(n, generator=g, device=DEV)
        snaps = vn.update(Rd, perm, nmb).cpu().numpy()
        want = VO.epoch(ref, R, perm.cpu().numpy(), nmb)
        assert _ulps(snaps, want).max() <= 1, (ep, snaps, want)
        np.testing.assert_allclose(vn.state.cpu().numpy(), ref.state, rtol=1e-12, atol=0)
        np.testing.assert_array_equal(vn.affine.cpu().numpy(), snaps[-1])
    mu, sd = vn.mean_std()
    assert torch.equal(mu, vn.affine[:, 0]) and torch.equal(sd, vn.affine[:, 1])


@gpu
def test_update_is_bit_identical_across_calls_and_streams():
    n, nmb = 200_003, 4
    _, Rd = _returns(n, 1)
    perms = [torch.randperm(n, generator=torch.Generator(device=DEV).manual_seed(s), device=DEV) for s in range(3)]
    res = []
    for s in (torch.cuda.current_stream(), torch.cuda.Stream(), torch.cuda.current_stream()):
        vn = ValueNorm(DEV, **VN)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            snaps = [vn.update(Rd, p, nmb).clone() for p in perms]
        torch.cuda.synchronize()
        res.append((torch.stack(snaps).cpu(), vn.state.cpu()))
    for snaps, state in res[1:]:
        assert torch.equal(snaps, res[0][0]) and torch.equal(state, res[0][1])


@gpu
def test_normalize_and_denormalize_round_like_the_kernels():
    vn = ValueNorm(DEV, **VN)
    vn.affine.copy_(torch.from_numpy(AFFINE))
    rng = np.random.default_rng(4)
    v = rng.normal(0, 3, (3000, 2)).astype(np.float32)
    got = vn.denormalize(torch.from_numpy(v).to(DEV)).cpu().numpy()
    for i in range(0, 3000, 7):                                # fmaf: the exact v sigma + mu, rounded once
        for h in range(2):
            exact = Fraction(float(v[i, h])) * Fraction(float(AFFINE[h, 1])) + Fraction(float(AFFINE[h, 0]))
            lo = np.float32(float(exact))
            cands = [np.nextafter(lo, np.float32(-np.inf)), lo, np.nextafter(lo, np.float32(np.inf))]
            best = min(cands, key=lambda c: (abs(Fraction(float(c)) - exact), int(np.float32(c).view(np.int32)) & 1))
            assert got[i, h] == best, (v[i, h], h)
    x = torch.from_numpy(v).to(DEV)
    assert torch.equal(vn.normalize(x), (x - vn.affine[:, 0]) / vn.affine[:, 1])


# ---- GPU: GAE on denormalised values -----------------------------------------------------------------------
def _gae_inputs(T=16, rows=2048, seed=0):
    rng = np.random.default_rng(seed)
    h = dict(reward=rng.normal(0, 1, (T, rows)).astype(np.float32), cost=rng.poisson(0.3, (T, rows)).astype(np.float32),
             values=rng.normal(0, 1, (T + 1, rows, 2)).astype(np.float32),
             done=(rng.random((T, rows)) < 0.1).astype(np.uint8))
    return h, {k: torch.from_numpy(x).to(DEV) for k, x in h.items()}


def _gae(d, affine=None, out=None):
    lib = abi.load_library()
    T, rows = d["reward"].shape
    ret, adv = out if out is not None else (torch.full((T, rows, 2), np.nan, device=DEV) for _ in range(2))
    args = [d["reward"].data_ptr(), d["cost"].data_ptr(), d["values"].data_ptr(), d["done"].data_ptr(), T, rows, rows,
            0.99, 0.95, ret.data_ptr(), adv.data_ptr()]
    if affine is None:
        st = lib.gsm_gae(*args, 0, None)
    else:
        st = lib.gsm_gae_normalized(*args, affine.data_ptr(), 0, None)
    assert st == 0
    torch.cuda.synchronize()
    return ret, adv


@gpu
def test_gae_normalized_matches_fp64_and_equals_gsm_gae_at_the_identity():
    h, d = _gae_inputs()
    ret, adv = _gae(d, torch.from_numpy(AFFINE).to(DEV))
    R64, A64 = VO.gae(h["reward"], h["cost"], h["values"], h["done"], np.float32(0.99), np.float32(0.95), AFFINE)
    np.testing.assert_allclose(ret.cpu().numpy(), R64, rtol=1e-5, atol=2e-5)
    np.testing.assert_allclose(adv.cpu().numpy(), A64, rtol=1e-5, atol=2e-5)
    r0, a0 = _gae(d)
    r1, a1 = _gae(d, torch.tensor([[0.0, 1.0], [0.0, 1.0]], device=DEV))
    assert torch.equal(r0, r1) and torch.equal(a0, a1)
    # the buffer entry point: a fresh normaliser denormalises x0.1 (the lineage's start), None is gsm_gae
    env, buf = _nav3_buffer(B=256, T=8)
    buf["values"].normal_()
    buf.compute_returns(0.99, 0.95)
    plain = buf["returns"].clone()
    vn = ValueNorm(DEV, **VN)
    buf.compute_returns(0.99, 0.95, value_norm=vn)
    scaled = buf["returns"].clone()
    buf["values"].mul_(np.float32(0.1))
    buf.compute_returns(0.99, 0.95)
    torch.testing.assert_close(scaled, buf["returns"], rtol=1e-6, atol=1e-6)
    assert not torch.equal(plain, scaled)
    env.close()


# ---- GPU: the normalised backward ----------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("kind", [5, 9, "gauss"])
def test_normalized_backward_matches_fp64_oracle_and_equals_the_plain_one_at_the_identity(kind):
    from tests.test_ppo_update import _assert_grad_close, _make_actor, _synthetic, _trainer
    R, K = 4099, 7
    actor = _make_actor(kind, seed=3)
    d, h, mod, w = _synthetic(actor, R, K, seed=12)
    # _synthetic places the targets away from every branch edge; keep them there in normalised units
    raw = (h["R"].astype(np.float64) * AFFINE[:, 1] + AFFINE[:, 0]).astype(np.float32)
    d["returns"] = torch.from_numpy(raw)[None].to(DEV)
    split = G.split_vector if kind == "gauss" else (lambda v: L.split_vector(v, kind))
    rows = np.random.default_rng(6).permutation(R)[:3001]
    rows_d = torch.from_numpy(rows).to(DEV)
    tr = _trainer(actor)
    tr.adv_moments.copy_(torch.tensor(h["moments"], dtype=torch.float32))
    tr.lagrange.fill_(h["lam"])
    x = tr.inputs(d)
    stats = torch.full((8,), float("nan"), device=DEV)
    tr.backward(x, rows_d, stats, torch.from_numpy(AFFINE).to(DEV))
    got, st = tr.grad.double().cpu().numpy(), stats.double().cpu().numpy()
    want, st0, ex = VO.loss_grad(mod, w, h["obs"], h["feat"], h["cnt"], h["act"], h["old_logp"], h["old_v"], raw,
                                 h["A"], h["moments"], h["lam"], AFFINE, rows=rows, **COEFS)
    assert (ex["d_v"] == 0).any() and (ex["d_v"] != 0).any()
    _assert_grad_close(got, want, split)
    np.testing.assert_allclose(st, st0, rtol=1e-4, atol=1e-6)
    # the identity affine: bit-identical to gsm_ppo_backward(_gauss)
    tr.backward(x, rows_d, stats, torch.tensor([[0.0, 1.0], [0.0, 1.0]], device=DEV))
    g1, s1 = tr.grad.clone(), stats.clone()
    tr.backward(x, rows_d, stats)
    assert torch.equal(g1, tr.grad) and torch.equal(s1, stats)


# ---- GPU: the update with a normaliser -----------------------------------------------------------------------
def _nav3_buffer(B=256, T=8, seed=3):
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
    from gs_marl_b200.rollout import GraphRolloutBuffer
    env = MultiAgentGraphConstrainEnv(make_cfg("navigation", 3, "f32", episode_length=25), B, auto_reset=True,
                                      seed=seed)
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    return env, buf


def _rollout(env, actor, buf, vn, it=0):
    from gs_marl_b200.rollout import collect_fused
    collect_fused(env, actor, buf, seed=17, first_step=it * buf.T)
    buf["values"][buf.T] = actor.act(buf["obs"][buf.T], buf.graph(buf.T), seed=0, greedy=True, want_values=True)[-1]
    buf.compute_returns(0.99, 0.95, value_norm=vn)


@gpu
def test_update_with_a_normaliser_matches_the_fp64_restatement():
    env, buf = _nav3_buffer()
    actor = GraphAttentionActor(5, seed=2).to(DEV)
    vn = ValueNorm(DEV, beta=0.99, epsilon=VN["epsilon"], var_floor=VN["var_floor"])
    _rollout(env, actor, buf, vn)
    n_epoch, nmb = 2, 3
    tr = LagrangianPPO(actor, **dict(HP, **COEFS, ppo_epoch=n_epoch, num_mini_batch=nmb), value_norm=vn)
    tr.lagrange.fill_(0.3)
    gen = torch.Generator(device=DEV)
    gen.set_state(tr.generator.get_state())
    p0 = tr.params.double().cpu().numpy()
    x = {k: t.cpu().numpy() for k, t in tr.inputs(buf).items()}
    out = tr.update(buf).double().cpu().numpy()
    # the restatement: the same permutations, fp64 normaliser / loss / gradient, Adam in float64 torch
    f32 = lambda q: float(np.float32(q))
    ref_p = torch.nn.Parameter(torch.from_numpy(p0.copy()))
    opt = torch.optim.Adam([ref_p], lr=f32(HP["lr"]), betas=tuple(f32(b) for b in HP["betas"]), eps=f32(HP["eps"]))
    ref_vn = VO.ValueNorm64(0.99, VN["epsilon"], VN["var_floor"])
    mom = O.adv_moments(x["adv"])
    n = len(x["cnt"])
    mb = n // nmb
    want_stats = []
    for _ in range(n_epoch):
        perm = torch.randperm(n, generator=gen, device=DEV).cpu().numpy()
        snaps = VO.epoch(ref_vn, x["ret"], perm, nmb)
        for b in range(nmb):
            wts = L.split_vector(ref_p.detach().numpy(), 5)
            g, st, _ = VO.loss_grad(L, wts, x["obs"], x["feat"], x["cnt"], x["act"], x["old_logp"], x["old_v"],
                                    x["ret"], x["adv"], mom, 0.3, snaps[b], rows=perm[b * mb:(b + 1) * mb], **COEFS)
            ref_p.grad = torch.from_numpy(np.asarray(g, np.float64))
            norm = float(torch.nn.utils.clip_grad_norm_([ref_p], f32(HP["max_grad_norm"])))
            opt.step()
            want_stats.append(np.append(st, norm))
    np.testing.assert_allclose(vn.state.cpu().numpy(), ref_vn.state, rtol=1e-12, atol=0)
    assert _ulps(vn.affine.cpu().numpy(), ref_vn.affine().astype(np.float32)).max() <= 1
    want_stats = np.array(want_stats)
    np.testing.assert_allclose(out[0], want_stats[0], rtol=1e-4, atol=1e-6)      # the first step: the §14 bar
    np.testing.assert_allclose(out, want_stats, rtol=2e-3, atol=1e-5)
    got_d, want_d = L.split_vector(tr.params.double().cpu().numpy() - p0, 5), \
        L.split_vector(ref_p.detach().numpy() - p0, 5)
    for k in got_d:
        scale = np.linalg.norm(want_d["att_w" if k == "att_b" else k])
        assert np.linalg.norm(np.asarray(got_d[k]) - np.asarray(want_d[k])) <= 1e-3 * scale, k
    env.close()


@gpu
def test_captured_normaliser_and_minibatch_step_replay_bit_identical_to_eager():
    env, buf = _nav3_buffer()
    actor = GraphAttentionActor(5, seed=6).to(DEV)
    vn = ValueNorm(DEV, **VN)
    _rollout(env, actor, buf, vn)
    tr = LagrangianPPO(actor, **HP, value_norm=vn)
    x = tr.inputs(buf)
    tr.set_advantage_moments(x["adv"])
    n = x["cnt"].numel()
    perm = torch.randperm(n, device=DEV)
    mb = n // 3

    def step(stats):
        snaps = vn.update(x["ret"], perm, 3)
        tr.minibatch_step(x, perm[mb:2 * mb], stats, snaps[1])
    state = [tr.params, tr.m, tr.v, tr.step, vn.state]
    saved = [t.clone() for t in state]
    vn.update(x["ret"], perm, 3)                             # allocates the snapshots and the workspaces
    eager = torch.zeros(9, device=DEV)
    for t, s in zip(state, saved):
        t.copy_(s)
    step(eager)
    want = [t.clone() for t in state] + [vn._snaps.clone()]
    for t, s in zip(state, saved):
        t.copy_(s)
    torch.cuda.synchronize()
    cap = torch.zeros(9, device=DEV)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step(cap)
    for t, s in zip(state, saved):
        t.copy_(s)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(cap, eager)
    for t, w in zip(state + [vn._snaps], want):
        assert torch.equal(t, w)
    env.close()


@gpu
def test_state_dict_round_trip_resumes_bit_identically():
    env, buf = _nav3_buffer()
    actor = GraphAttentionActor(5, seed=7).to(DEV)
    vn = ValueNorm(DEV, **VN)
    _rollout(env, actor, buf, vn)
    hp = dict(HP, ppo_epoch=2, num_mini_batch=3)
    tr = LagrangianPPO(actor, **hp, value_norm=vn)
    tr.update(buf)
    sd = tr.state_dict()
    assert set(sd["value_norm"]) == {"state", "affine"}
    with pytest.raises(ValueError):                          # a trainer without a normaliser refuses it
        LagrangianPPO(GraphAttentionActor(5, seed=1).to(DEV), **hp).load_state_dict(sd)
    out1 = tr.update(buf)
    vn2 = ValueNorm(DEV, **VN)
    tr2 = LagrangianPPO(GraphAttentionActor(5, seed=1).to(DEV), **hp, value_norm=vn2)
    tr2.load_state_dict(sd)
    out2 = tr2.update(buf)
    torch.cuda.synchronize()
    assert torch.equal(out1, out2) and torch.equal(tr.params, tr2.params)
    assert torch.equal(vn.state, vn2.state) and torch.equal(vn.affine, vn2.affine)
    assert torch.isfinite(out1).all()
    env.close()


@gpu
def test_guard_bands_stay_untouched():
    lib = abi.load_library()
    GB = 1024                                                  # 4 KB of fp32 (512 doubles: 4 KB too)

    def banded(n, dtype, fill):
        big = torch.full((n + 2 * GB,), fill, dtype=dtype, device=DEV)
        return big, big[GB:GB + n]
    n, nmb = 40_001, 3
    _, Rd = _returns(n, 2)
    perm = torch.randperm(n, device=DEV)
    mb = n // nmb
    state_big, state = banded(6, torch.float64, 12345.0)
    state.zero_()
    aff_big, aff = banded((nmb + 1) * 4, torch.float32, 12345.0)
    need = lib.gsm_value_norm_update_workspace(mb, nmb)
    ws_big = torch.full((need + 8 * GB,), 0x5A, dtype=torch.uint8, device=DEV)
    io = abi.GsmValueNormIO()
    io.struct_size = C.sizeof(abi.GsmValueNormIO)
    io.state, io.affine, io.returns, io.rows = state.data_ptr(), aff.data_ptr(), Rd.data_ptr(), perm.data_ptr()
    io.mb, io.n_mini_batch = mb, nmb
    io.beta, io.epsilon, io.var_floor = VN["beta"], VN["epsilon"], VN["var_floor"]
    assert lib.gsm_value_norm_update(C.byref(io), ws_big[4 * GB:].data_ptr(), need, 0, None) == 0
    h, d = _gae_inputs(T=8, rows=1000)
    T, rows = 8, 1000
    ret_big, ret = banded(T * rows * 2, torch.float32, 12345.0)
    adv_big, adv = banded(T * rows * 2, torch.float32, 12345.0)
    _gae(d, aff[:4], out=(ret, adv))
    torch.cuda.synchronize()
    for k, big in (("state", state_big), ("affine", aff_big), ("returns", ret_big), ("advantages", adv_big)):
        assert (big[:GB] == 12345.0).all() and (big[-GB:] == 12345.0).all(), k
    assert (ws_big[:4 * GB] == 0x5A).all() and (ws_big[4 * GB + need:] == 0x5A).all()
    assert torch.isfinite(state).all() and torch.isfinite(aff).all() and torch.isfinite(ret).all()
