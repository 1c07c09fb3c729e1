"""SPEC.md §10b / §12b: the Gaussian graph actor for continuous-action worlds — `gsm_policy_act_gauss`,
`gsm_collect_gauss`, `gsm_policy_evaluate_gauss` / `gsm_policy_backward_gauss`, exposed as
`GaussianGraphActor` and `collect_fused`.

CPU: the fp64 oracle (tests/_gauss_oracle.py) against torch autograd of `dist_autograd`, the vector
order and `pack()`, the struct layouts, the entry points' argument checks, the Box-Muller draw.
GPU: the kernels against the oracle, the draw's statistics and sharding invariance, the fused collect
against a stepwise loop (one handle, stream shards, CUDA graph), bit identity of `evaluate_actions` with
what collect wrote, gradients, determinism, capture, a clipped-PPO minibatch, the shared-memory limit."""
import ctypes as C
import math
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from gs_marl_b200 import abi
from gs_marl_b200.policy import GaussianGraphActor, GraphAttentionActor
from oracle import policy_oracle as P
from tests import _gauss_oracle as G
from tests._util import make_cfg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NP = abi.GSM_POLICY_GAUSS_N_PARAMS
SMEM_OPTIN = 232448                    # sm_100: shared memory a block may opt in to (227 KB)
# backward static shared memory: weights, then per row of its 64: obs, dZ (4), dsum, cnt, src, dlog_std (2)
KMAX = (SMEM_OPTIN - (4 * NP + 64 * 4 * (6 + 4 + 1 + 1) + 64 * 8 + 64 * 4 * 2)) // (2 * 4 * 64)
BENCH_ROWS = 16384 * 3 * 25


def synth(R, K, seed=0, act_scale=1.0):
    rng = np.random.default_rng(seed)
    obs = rng.standard_normal((R, 6)).astype(np.float32)
    cnt = rng.integers(0, K + 1, R).astype(np.int32)
    cnt[0] = 0
    cnt[min(1, R - 1)] = K                                    # both ends of the count range
    feat = rng.standard_normal((R, K, 6)).astype(np.float32)
    feat[np.arange(K)[None, :] >= cnt[:, None]] = 0
    act = (rng.standard_normal((R, 2)) * act_scale).astype(np.float32)
    up = (rng.standard_normal(R), rng.standard_normal(R), rng.standard_normal((R, 2)))
    return obs, feat, cnt, act, up


def make_actor(seed, log_std=(-0.5, 0.3), dtype=torch.float32, device="cpu"):
    a = GaussianGraphActor(seed=seed)
    with torch.no_grad():
        a.log_std.weight.copy_(torch.tensor(log_std))
    return a.to(device=device, dtype=dtype)


def torch_reference(actor, obs, feat, cnt, act):
    g = {"nbr_feat": feat, "nbr_cnt": cnt}
    d = actor.dist_autograd(obs, g)
    return d.log_prob(act).sum(-1), d.entropy().sum(-1), actor.values_autograd(obs, g)


# ---- CPU --------------------------------------------------------------------------------------
@pytest.mark.parametrize("R,K", [(96, 8), (40, 1)])
@pytest.mark.parametrize("log_std", [-3.0, 0.0, 2.0])
def test_oracle_matches_torch_autograd_fp64(R, K, log_std):
    actor = make_actor(21, (log_std, log_std * 0.5), torch.float64)
    obs, feat, cnt, act, (dl, de, dv) = synth(R, K, seed=3)
    w = G.weights_from_state_dict(actor.state_dict())
    t = lambda x: torch.from_numpy(x)
    lp, ent, v = torch_reference(actor, t(obs).double(), t(feat).double(), t(cnt), t(act).double())
    loss = (lp * t(dl)).sum() + (ent * t(de)).sum() + (v * t(dv)).sum()
    want = torch.cat([g.reshape(-1) for g in torch.autograd.grad(loss, list(actor.parameters()))]).numpy()
    lp0, ent0, v0 = G.evaluate(w, obs, feat, cnt, act)
    for x, x0 in ((lp, lp0), (ent, ent0), (v, v0)):
        np.testing.assert_allclose(x0, x.detach().numpy(), rtol=1e-9, atol=1e-12)
    got = G.evaluate_backward(w, obs, feat, cnt, act, dl, de, dv)
    assert got.shape == (NP,)
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-12)


def test_vector_order_and_pack_round_trip():
    actor = make_actor(4)
    names = [n for n, _ in actor.named_parameters()]
    assert names == ["ego.weight", "ego.bias", "nbr.weight", "nbr.bias", "att.weight", "att.bias", "head.weight",
                     "head.bias", "log_std.weight", "value.weight", "value.bias"]
    vec = torch.nn.utils.parameters_to_vector(actor.parameters()).detach().numpy()
    assert vec.size == NP == 1479
    np.testing.assert_array_equal(vec, G.to_vector(G.weights_from_state_dict(actor.state_dict(), np.float32)))
    sp = G.split_vector(vec)
    np.testing.assert_array_equal(sp["log_std"], np.float32([-0.5, 0.3]))
    w = actor.pack()
    arr = lambda f: np.ctypeslib.as_array(getattr(w, f))
    packed = {"ego_w": arr("ego_w"), "ego_b": arr("ego_b"), "nbr_w": arr("nbr_w"), "nbr_b": arr("nbr_b"),
              "att_w": arr("att_w"), "att_b": np.float32(w.att_b), "head_w": arr("mean_w"), "head_b": arr("mean_b"),
              "log_std": arr("log_std"), "value_w": arr("value_w"), "value_b": arr("value_b")}
    np.testing.assert_array_equal(G.to_vector(packed).astype(np.float32), vec)
    assert w.struct_size == C.sizeof(abi.GsmPolicyGaussWeights)


def test_gauss_struct_layouts_match_the_header(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    structs = {"gsm_policy_gauss_weights": abi.GsmPolicyGaussWeights, "gsm_policy_gauss_io": abi.GsmPolicyGaussIO,
               "gsm_policy_gauss_eval_io": abi.GsmPolicyGaussEvalIO}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "gsmarl_b200.h"', 'int main(void) {',
             '  printf("dim %d\\n", GSM_POLICY_GAUSS_DIM);', '  printf("np %d\\n", GSM_POLICY_GAUSS_N_PARAMS);']
    for s, cls in structs.items():
        lines.append(f'  printf("{s}.size %zu\\n", sizeof({s}));')
        lines += [f'  printf("{s}.{f} %zu\\n", offsetof({s}, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    (tmp_path / "l.c").write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(tmp_path / "l.c"),
                    "-o", str(tmp_path / "l")], check=True)
    got = dict(ln.split() for ln in subprocess.run([str(tmp_path / "l")], capture_output=True, text=True,
                                                   check=True).stdout.splitlines())
    assert (int(got["dim"]), int(got["np"])) == (abi.GSM_POLICY_GAUSS_DIM, NP)
    for s, cls in structs.items():
        assert int(got[f"{s}.size"]) == C.sizeof(cls), s
        for f, _ in cls._fields_:
            assert int(got[f"{s}.{f}"]) == getattr(cls, f).offset, (s, f)


def test_gauss_bad_arguments_without_device():
    lib = abi.load_library()
    io = abi.GsmPolicyGaussEvalIO()
    assert lib.gsm_policy_evaluate_gauss(None, 0, None) == -1
    assert lib.gsm_policy_evaluate_gauss(C.byref(io), 0, None) == -3            # struct_size 0
    io.struct_size, io.action_dim = C.sizeof(abi.GsmPolicyGaussEvalIO), 3
    assert lib.gsm_policy_evaluate_gauss(C.byref(io), 0, None) == -4
    io.action_dim = 2
    assert lib.gsm_policy_evaluate_gauss(C.byref(io), 0, None) == -1            # NULL pointers
    assert b"required" in lib.gsm_policy_last_error()
    io.params = io.obs = io.nbr_feat = io.nbr_cnt = io.actions = 256
    io.n_rows, io.max_nbrs = 100, 0
    assert lib.gsm_policy_evaluate_gauss(C.byref(io), 0, None) == -1            # max_nbrs < 1
    io.max_nbrs = 8
    need = lib.gsm_policy_backward_workspace_gauss(100)
    assert need > 0 and need % (4 * NP) == 0
    assert lib.gsm_policy_backward_workspace_gauss(-1) == -1
    assert lib.gsm_policy_backward_gauss(C.byref(io), None, None, None, None, 512, need, 0, None) == -1   # grad NULL
    assert lib.gsm_policy_backward_gauss(C.byref(io), None, None, None, 512, 512, need - 1, 0, None) == -1
    assert b"workspace" in lib.gsm_policy_last_error()
    io.struct_size = 8
    assert lib.gsm_policy_backward_gauss(C.byref(io), None, None, None, 512, 512, need, 0, None) == -3
    io.struct_size, io.n_rows = C.sizeof(abi.GsmPolicyGaussEvalIO), 0            # no-op
    assert lib.gsm_policy_evaluate_gauss(C.byref(io), 0, None) == 0
    assert lib.gsm_policy_backward_gauss(C.byref(io), None, None, None, 512, None, 0, 0, None) == 0
    # the actor entry point
    w, aio = abi.GsmPolicyGaussWeights(), abi.GsmPolicyGaussIO()
    assert lib.gsm_policy_act_gauss(None, C.byref(aio), 0, None) == -1
    assert lib.gsm_policy_act_gauss(C.byref(w), C.byref(aio), 0, None) == -3     # struct_size 0
    w.struct_size = C.sizeof(abi.GsmPolicyGaussWeights)
    assert lib.gsm_policy_act_gauss(C.byref(w), C.byref(aio), 0, None) == -1     # NULL pointers
    aio.obs = aio.nbr_feat = aio.nbr_cnt = aio.actions = 256
    aio.n_rows, aio.max_nbrs = 4, 0
    assert lib.gsm_policy_act_gauss(C.byref(w), C.byref(aio), 0, None) == -1     # max_nbrs < 1
    assert lib.gsm_collect_gauss(None, C.byref(w), 1, None, None, None, 0, 0, 0, None) == -1
    if not torch.cuda.is_available():
        aio.max_nbrs = 8
        assert lib.gsm_policy_act_gauss(C.byref(w), C.byref(aio), 0, None) == -5
        with pytest.raises(abi.GsmError):
            GaussianGraphActor().evaluate_actions(torch.zeros(4, 6), {"nbr_feat": torch.zeros(4, 8, 6),
                                                                      "nbr_cnt": torch.zeros(4, dtype=torch.int32)},
                                                  torch.zeros(4, 2))


@pytest.mark.parametrize("seed,row,step", [(0, 0, 0), (7, 12345, 3), (2 ** 40 + 5, 2 ** 33 + 17, 99), (1, 786431, 24)])
def test_box_muller_matches_scalar_restatement(seed, row, step):
    got = G.box_muller_eps(1, seed, step, row_offset=row)[0]
    r = P.philox4x32_10(np.array([row & 0xFFFFFFFF]), np.array([row >> 32]), np.array([step]), np.array([0x80000000]),
                        seed & 0xFFFFFFFF, seed >> 32)
    u0 = (int(r[0][0]) >> 9) * 2.0 ** -23 + 2.0 ** -24
    u1 = (int(r[1][0]) >> 9) * 2.0 ** -23 + 2.0 ** -24
    rho = math.sqrt(-2.0 * math.log(u0))
    assert got[0] == pytest.approx(rho * math.cos(2 * math.pi * u1), rel=1e-15, abs=1e-15)
    assert got[1] == pytest.approx(rho * math.sin(2 * math.pi * u1), rel=1e-15, abs=1e-15)


# ---- GPU --------------------------------------------------------------------------------------
DEV = "cuda"
to = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _chunked(fn, n, chunk=65536):
    outs = [fn(slice(s, min(n, s + chunk))) for s in range(0, n, chunk)]
    return [np.concatenate(z) for z in zip(*outs)]


def _grads(actor):
    return torch.cat([p.grad.reshape(-1) for p in actor.parameters()])


def _assert_grad_close(got, want, bar=1e-4):
    """||g - g_ref|| <= bar ||g_ref|| per parameter tensor; att_b (exact gradient 0) at att_w's scale."""
    g, w = G.split_vector(np.asarray(got, np.float64)), G.split_vector(np.asarray(want, np.float64))
    bad = [(k, np.linalg.norm(g[k] - w[k])) for k in G.VECTOR_ORDER
           if not np.linalg.norm(g[k] - w[k]) <= bar * np.linalg.norm(w["att_w" if k == "att_b" else k])]
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("R,K", [(1, 7), (613, 32), (4099, 1), (786432, 7)])
def test_act_matches_oracle(R, K):
    actor = make_actor(5, device=DEV)
    obs, feat, cnt, _, _ = synth(R, K, seed=6)
    f = feat.copy()
    f[np.arange(K)[None, :] >= cnt[:, None]] = np.nan           # only the valid rows may be read
    g = {"nbr_feat": to(f), "nbr_cnt": to(cnt)}
    a, lp, mu, v = actor.act(to(obs), g, seed=11, step=4, row_offset=100, want_mean=True, want_values=True)
    w = G.weights_from_state_dict(actor.state_dict())
    a0, lp0, mu0, v0 = _chunked(lambda s: G.act(w, obs[s], feat[s], cnt[s], 11, 4, 100 + s.start), R)
    for x, x0, atol in ((mu, mu0, 2e-5), (v, v0, 2e-5), (a, a0, 1e-5), (lp, lp0, 2e-5)):
        assert torch.isfinite(x).all()
        np.testing.assert_allclose(x.cpu().numpy(), x0, rtol=1e-4, atol=atol)
    ag, lpg = actor.act(to(obs), g, seed=11, step=4, greedy=True)
    assert torch.equal(ag, mu)
    np.testing.assert_allclose(lpg.cpu().numpy(), -(np.asarray([-0.5, 0.3]).sum()) - G.LOG_2PI, rtol=1e-6)


@pytest.mark.gpu
def test_draws_are_sharding_invariant_and_change_with_step():
    actor = make_actor(6, device=DEV)
    obs, feat, cnt, _, _ = synth(3000, 5, seed=7)
    o, g = to(obs), {"nbr_feat": to(feat), "nbr_cnt": to(cnt)}
    full, _ = actor.act(o, g, seed=3, step=9)
    lo, _ = actor.act(o[:1234].contiguous(), {k: v[:1234].contiguous() for k, v in g.items()}, seed=3, step=9)
    hi, _ = actor.act(o[1234:].contiguous(), {k: v[1234:].contiguous() for k, v in g.items()}, seed=3, step=9,
                      row_offset=1234)
    assert torch.equal(torch.cat([lo, hi]), full)
    other, _ = actor.act(o, g, seed=3, step=10)
    assert bool((other != full).all(-1).float().mean() > 0.99)


@pytest.mark.gpu
def test_draws_are_standard_normal():
    from scipy import stats
    actor = make_actor(7, log_std=(0.0, 0.0), device=DEV)
    with torch.no_grad():
        actor.head.weight.zero_(); actor.head.bias.zero_()
    R = 1 << 20
    o = torch.zeros(R, 6, device=DEV)
    g = {"nbr_feat": torch.zeros(R, 1, 6, device=DEV), "nbr_cnt": torch.zeros(R, dtype=torch.int32, device=DEV)}
    eps = actor.act(o, g, seed=2024, step=1)[0].double().cpu().numpy()
    for d in range(2):
        assert stats.kstest(eps[:, d], "norm").pvalue > 1e-3, d
    assert abs(np.corrcoef(eps[:, 0], eps[:, 1])[0, 1]) < 5e-3


def _cont_env(scn, N, n_envs, sharded=False, seed=3):
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv, StreamShardedEnv
    cfg = make_cfg(scn, N, "f32", action_mode="continuous").replace(episode_length=4)   # restarts in the rollout
    if sharded:
        return StreamShardedEnv(cfg, n_envs, n_streams=3, seed=seed, auto_reset=True)
    return MultiAgentGraphConstrainEnv(cfg, n_envs, seed=seed, auto_reset=True)


def _stepwise(env, actor, T, seed, first_step):
    """act + gsm_step + reset-on-done per step (rollout.collect with the actor as the torch policy)."""
    from gs_marl_b200.rollout import GraphRolloutBuffer, collect
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    t = [0]

    def policy(obs, graph):
        a, lp, v = actor.act(obs, graph, seed=seed, step=first_step + t[0], want_values=True)
        buf["logp"][t[0]].copy_(lp)
        buf["values"][t[0]].copy_(v)
        t[0] += 1
        return a
    collect(env, policy, buf)
    torch.cuda.synchronize()
    return buf


def _fused(env, actor, T, seed, first_step, graph=False):
    from gs_marl_b200.rollout import GraphRolloutBuffer, collect_fused
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    g = collect_fused(env, actor, buf, seed=seed, first_step=first_step, graph=graph)
    if graph:
        g.replay()
    torch.cuda.synchronize()
    return buf


def _assert_buffers_equal(a, b):
    for k in a.data:
        if k == "values":                                      # slot T is the caller's bootstrap
            assert torch.equal(a[k][:-1], b[k][:-1]), k
        else:
            assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("scn,N", [("navigation", 3), ("navigation", 12), ("polygon", 6), ("line", 6)])
def test_collect_fused_equals_stepwise_loop(scn, N):
    actor = make_actor(8, device=DEV)
    e1, e2 = _cont_env(scn, N, 700), _cont_env(scn, N, 700)
    fused = _fused(e1, actor, 9, seed=5, first_step=20)
    step = _stepwise(e2, actor, 9, seed=5, first_step=20)
    assert bool(fused["done"].any()), "episodes must restart inside the rollout"
    _assert_buffers_equal(fused, step)
    e1.close(); e2.close()


@pytest.mark.gpu
def test_collect_fused_sharded_and_graph_replay_equal_one_handle():
    actor = make_actor(9, device=DEV)
    ref = _fused(_cont_env("navigation", 3, 1000), actor, 7, seed=1, first_step=0)
    shard = _fused(_cont_env("navigation", 3, 1000, sharded=True), actor, 7, seed=1, first_step=0)
    _assert_buffers_equal(ref, shard)
    replay = _fused(_cont_env("navigation", 3, 1000), actor, 7, seed=1, first_step=0, graph=True)
    _assert_buffers_equal(ref, replay)


@pytest.mark.gpu
def test_collect_of_the_wrong_kind_is_unsupported():
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
    from gs_marl_b200.rollout import GraphRolloutBuffer, collect_fused
    gauss, cat = make_actor(1, device=DEV), GraphAttentionActor(5, seed=1).to(DEV)
    cont = _cont_env("navigation", 3, 64)
    disc = MultiAgentGraphConstrainEnv(make_cfg("navigation", 3, "f32"), 64, seed=1)
    for env, right, wrong, fn, w in ((cont, gauss, cat, "gsm_collect", cat.pack()),
                                     (disc, cat, gauss, "gsm_collect_gauss", gauss.pack())):
        buf = GraphRolloutBuffer(env, 2)
        buf.reset_env()
        st = getattr(env.lib, fn)(env._h, C.byref(w), 2, C.byref(buf._io_all[0]), None, None, 0, 0, 0, None)
        assert st == -4
        with pytest.raises(ValueError, match="action_mode"):
            collect_fused(env, wrong, buf)
        collect_fused(env, right, buf)
        env.close()


@pytest.mark.gpu
def test_collect_fused_takes_an_actor_without_action_mode():
    """Any object with packed() works: the weights' type picks the collect, the C side checks the kind."""
    from gs_marl_b200.rollout import collect_fused

    class Wrapped:
        def __init__(self, actor):
            self.packed = actor.packed
    actor = make_actor(2, device=DEV)
    ref = _fused(_cont_env("navigation", 3, 200), actor, 3, seed=4, first_step=0)
    env = _cont_env("navigation", 3, 200)
    got = _fused(env, Wrapped(actor), 3, seed=4, first_step=0)
    _assert_buffers_equal(ref, got)
    with pytest.raises(abi.GsmError, match="discrete actions"):
        collect_fused(env, Wrapped(GraphAttentionActor(5, seed=1).to(DEV)), got)
    env.close()


def _collected(T=6, n_envs=500):
    env = _cont_env("navigation", 3, n_envs)
    actor = make_actor(12, device=DEV)
    buf = _fused(env, actor, T, seed=5, first_step=10)
    return env, buf, actor


@pytest.mark.gpu
def test_evaluate_is_bit_identical_to_collection():
    env, buf, actor = _collected()
    g = {"nbr_feat": buf["nbr_feat"][:-1], "nbr_cnt": buf["nbr_cnt"][:-1]}
    with torch.no_grad():
        lp, ent, v = actor.evaluate_actions(buf["obs"][:-1], g, buf["actions"])
    assert torch.equal(lp, buf["logp"]) and torch.equal(v, buf["values"][:-1])
    assert torch.equal(torch.exp(lp - buf["logp"]), torch.ones_like(lp))          # first-epoch PPO ratio
    idx = torch.randperm(lp.numel(), device=DEV, generator=torch.Generator(DEV).manual_seed(0))
    with torch.no_grad():
        lp2, _, v2 = actor.evaluate_actions(buf["obs"][:-1].flatten(0, 2), {
            "nbr_feat": buf["nbr_feat"][:-1].flatten(0, 2), "nbr_cnt": buf["nbr_cnt"][:-1].flatten(0, 2)},
            buf["actions"].flatten(0, 2), rows=idx)
    assert torch.equal(lp2, buf["logp"].flatten()[idx]) and torch.equal(v2, buf["values"][:-1].flatten(0, 2)[idx])
    env.close()


def _check_against_oracle(actor, obs, feat, cnt, act, up, nan_pad=True):
    f = feat.copy()
    if nan_pad:
        f[np.arange(feat.shape[1])[None, :] >= cnt[:, None]] = np.nan
    actor.zero_grad(set_to_none=True)
    out = actor.evaluate_actions(to(obs), {"nbr_feat": to(f), "nbr_cnt": to(cnt)}, to(act))
    torch.autograd.backward(out, [to(u.astype(np.float32)) for u in up])
    w = G.weights_from_state_dict(actor.state_dict())
    R = obs.shape[0]
    want = _chunked(lambda s: G.evaluate(w, obs[s], feat[s], cnt[s], act[s]), R)
    for x, x0 in zip(out, want):
        np.testing.assert_allclose(x.detach().cpu().numpy(), x0, rtol=1e-4, atol=2e-5)
    up32 = [u.astype(np.float32) for u in up]
    gw = sum(G.evaluate_backward(w, obs[s], feat[s], cnt[s], act[s], *[u[s] for u in up32])
             for s in (slice(i, min(R, i + 65536)) for i in range(0, R, 65536)))
    got = _grads(actor).cpu().numpy()
    return out, got, gw


@pytest.mark.gpu
@pytest.mark.parametrize("R,K", [(1, 7), (997, KMAX), (4099, 1), (BENCH_ROWS, 7)])
def test_evaluate_and_gradients_match_fp64_oracle(R, K):
    actor = make_actor(13, log_std=(0.4, -1.2), device=DEV)
    obs, feat, cnt, act, up = synth(R, K, seed=14)
    with torch.no_grad():                                       # actions around the mean, not around 0
        mu = actor.act(to(obs), {"nbr_feat": to(feat), "nbr_cnt": to(cnt)}, greedy=True)[0].cpu().numpy()
    act = (mu + act * np.exp([0.4, -1.2])).astype(np.float32)
    out, got, want = _check_against_oracle(actor, obs, feat, cnt, act, up)
    assert np.isfinite(got).all()
    _assert_grad_close(got, want)


@pytest.mark.gpu
def test_far_and_nan_actions():
    actor = make_actor(15, device=DEV)
    R, K = 2000, 6
    obs, feat, cnt, act, up = synth(R, K, seed=16)
    with torch.no_grad():
        mu = actor.act(to(obs), {"nbr_feat": to(feat), "nbr_cnt": to(cnt)}, greedy=True)[0].cpu().numpy()
    far = (mu + 50 * np.exp([-0.5, 0.3]) * np.sign(act)).astype(np.float32)   # 50 sigma from the mean
    out, got, want = _check_against_oracle(actor, obs, feat, cnt, far, up)
    assert np.isfinite(got).all()
    _assert_grad_close(got, want)
    nan = far.copy()
    nan[5, 1] = np.nan
    g = {"nbr_feat": to(feat), "nbr_cnt": to(cnt)}
    for dl5, poisoned in ((0.0, False), (1.5, True)):
        d_logp = to(up[0].astype(np.float32))
        d_logp[5] = dl5
        actor.zero_grad(set_to_none=True)
        lp, ent, v = actor.evaluate_actions(to(obs), g, to(nan))
        assert bool(torch.isnan(lp[5])) and bool(torch.isfinite(torch.cat([lp[:5], lp[6:]])).all())
        torch.autograd.backward((lp, ent, v), [d_logp, to(up[1].astype(np.float32)), to(up[2].astype(np.float32))])
        sp = G.split_vector(_grads(actor).double().cpu().numpy())
        assert np.isfinite(sp["value_w"]).all() and np.isfinite(sp["value_b"]).all()   # d_values carry no NaN
        assert np.isnan(sp["head_w"]).any() == poisoned and np.isnan(sp["log_std"]).any() == poisoned
        if not poisoned:
            assert all(np.isfinite(x).all() for x in sp.values())


@pytest.mark.gpu
def test_rows_index_equals_gathered_inputs():
    actor = make_actor(17, device=DEV)
    R, K = 20000, 8
    obs, feat, cnt, act, _ = synth(R, K, seed=18)
    o, g, a = to(obs), {"nbr_feat": to(feat), "nbr_cnt": to(cnt)}, to(act)
    gen = torch.Generator(DEV).manual_seed(1)
    idx = torch.randint(0, R, (7777,), device=DEV, generator=gen)          # repeats included
    up = [torch.randn(7777, device=DEV, generator=gen), torch.randn(7777, device=DEV, generator=gen),
          torch.randn(7777, 2, device=DEV, generator=gen)]
    res = []
    for gathered in (False, True):
        actor.zero_grad(set_to_none=True)
        if gathered:
            out = actor.evaluate_actions(o[idx].contiguous(), {k: v[idx].contiguous() for k, v in g.items()},
                                         a[idx].contiguous())
        else:
            out = actor.evaluate_actions(o, g, a, rows=idx)
        torch.autograd.backward(out, up)
        res.append([x.detach().clone() for x in out] + [_grads(actor).clone()])
    for x, y in zip(*res):
        assert torch.equal(x, y)
    with pytest.raises(IndexError):
        actor.evaluate_actions(o, g, a, rows=torch.tensor([0, R], device=DEV))
    with pytest.raises(TypeError):
        actor.evaluate_actions(o, g, a.to(torch.int32))
    with pytest.raises(ValueError):
        actor.evaluate_actions(o, g, a[:, :1].contiguous())


@pytest.mark.gpu
def test_backward_is_deterministic_and_capturable():
    actor = make_actor(19, device=DEV)
    R, K = 30000, 8
    obs, feat, cnt, act, up = synth(R, K, seed=20)
    o, g, a = to(obs), {"nbr_feat": to(feat), "nbr_cnt": to(cnt)}, to(act)
    idx = torch.randperm(R, device=DEV, generator=torch.Generator(DEV).manual_seed(2))[:12345]
    ups = [to(u[:12345].astype(np.float32)) for u in up]

    def step():
        actor.zero_grad(set_to_none=True)
        out = actor.evaluate_actions(o, g, a, rows=idx)
        torch.autograd.backward(out, ups)
        return [x.detach() for x in out] + [_grads(actor)]
    e1 = [x.clone() for x in step()]
    e2 = [x.clone() for x in step()]
    for x, y in zip(e1, e2):
        assert torch.equal(x, y)                                            # bit-identical grad
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cap = step()
    for p in actor.parameters():
        p.grad = None
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(e1, cap):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_clipped_ppo_minibatch_gradients_match_torch_formulation():
    """An EXAMPLE clipped-surrogate loss with the Gaussian logp on a shuffled minibatch of a collected
    rollout: gradients through the kernels == through dist_autograd."""
    env, buf, actor = _collected(T=8, n_envs=2000)
    with torch.no_grad():                                  # the learner has moved since collection
        for p in actor.parameters():
            p.add_(torch.randn(p.shape, device=DEV, generator=torch.Generator(DEV).manual_seed(p.numel())) * 3e-3)
    *_, vT = actor.act(buf["obs"][-1], buf.graph(buf.T), want_values=True)
    buf["values"][-1].copy_(vT)
    ret, adv = buf.compute_returns(0.99, 0.95)
    src = {k: buf[k][:-1].flatten(0, 2) for k in ("obs", "nbr_feat", "nbr_cnt")}
    acts = buf["actions"].flatten(0, 2)
    old_lp, ret, adv = buf["logp"].flatten(), ret.flatten(0, 2), adv[..., 0].flatten()
    idx = torch.randperm(old_lp.numel(), device=DEV, generator=torch.Generator(DEV).manual_seed(3))[:16384]

    def loss(lp, ent, v):
        ratio = torch.exp(lp - old_lp[idx])
        surr = torch.min(ratio * adv[idx], ratio.clamp(0.8, 1.2) * adv[idx])
        return -surr.mean() + 0.5 * ((ret[idx] - v) ** 2).mean() - 0.01 * ent.mean()

    grads = []
    for kernel in (True, False):
        actor.zero_grad(set_to_none=True)
        if kernel:
            out = actor.evaluate_actions(src["obs"], {"nbr_feat": src["nbr_feat"], "nbr_cnt": src["nbr_cnt"]},
                                         acts, rows=idx)
        else:
            out = torch_reference(actor, src["obs"][idx], src["nbr_feat"][idx], src["nbr_cnt"][idx], acts[idx])
        loss(*out).backward()
        grads.append(_grads(actor).double().cpu().numpy())
    _assert_grad_close(grads[0], grads[1])
    env.close()


@pytest.mark.gpu
def test_too_large_max_nbrs_is_reported_and_cleared():
    actor = make_actor(22, device=DEV)
    obs, feat, cnt, act, up = synth(70, KMAX + 1, seed=23)
    o, a = to(obs), to(act)
    out = actor.evaluate_actions(o, {"nbr_feat": to(feat), "nbr_cnt": to(cnt)}, a)
    with pytest.raises(abi.GsmError):
        torch.autograd.backward(out, [to(u.astype(np.float32)) for u in up])
    ok = actor.evaluate_actions(o, {"nbr_feat": to(feat[:, :KMAX]).contiguous(),
                                    "nbr_cnt": to(np.minimum(cnt, KMAX))}, a)
    actor.zero_grad(set_to_none=True)
    torch.autograd.backward(ok, [to(u.astype(np.float32)) for u in up])      # the next launch is not poisoned
    torch.cuda.synchronize()
    assert torch.isfinite(_grads(actor)).all()
