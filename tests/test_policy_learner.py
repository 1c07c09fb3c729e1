"""SPEC.md §12: the learner pass of the declared graph actor — `gsm_policy_evaluate` (log-prob of given
actions, entropy, both critics) and `gsm_policy_backward` (gradient w.r.t. the parameter vector),
exposed as `GraphAttentionActor.evaluate_actions`.

CPU: the fp64 numpy oracle (tests/_learner_oracle.py: forward and analytic backward) against torch
autograd of the plain-torch formulation (`embed_autograd`), the vector order, the C entry points' argument checks.  GPU: the kernels
against the oracle, bit identity with what collection wrote, `rows` indexing, determinism, CUDA-graph
capture, a clipped-PPO minibatch against the torch formulation, guard bands."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from gs_marl_b200 import abi
from gs_marl_b200.policy import GraphAttentionActor
from oracle import policy_oracle as P
from tests import _learner_oracle as L
from tests._util import make_cfg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def synth(R, K, n_actions, seed=0):
    rng = np.random.default_rng(seed)
    obs = rng.standard_normal((R, 6)).astype(np.float32)
    cnt = rng.integers(0, K + 1, R).astype(np.int32)
    cnt[0] = 0
    cnt[min(1, R - 1)] = K                                    # both ends of the count range
    feat = rng.standard_normal((R, K, 6)).astype(np.float32)
    feat[np.arange(K)[None, :] >= cnt[:, None]] = 0
    act = rng.integers(0, n_actions, R).astype(np.int32)
    up = (rng.standard_normal(R), rng.standard_normal(R), rng.standard_normal((R, 2)))
    return obs, feat, cnt, act, up


def torch_reference(actor, obs, feat, cnt, act):
    """The plain-torch formulation: embed_autograd + head / value + log_softmax."""
    emb = actor.embed_autograd(obs, {"nbr_feat": feat, "nbr_cnt": cnt})
    lp_all = torch.log_softmax(actor.head(emb), -1)
    logp = lp_all.gather(-1, act.long()[..., None])[..., 0]
    ent = -(lp_all.exp() * lp_all).sum(-1)
    return logp, ent, actor.value(emb)


def per_tensor(vec, n_actions):
    return L.split_vector(np.asarray(vec, np.float64), n_actions)


# ---- CPU --------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_actions,R,K", [(5, 96, 8), (9, 96, 8), (5, 40, 1)])
def test_oracle_learner_matches_torch_autograd_fp64(n_actions, R, K):
    actor = GraphAttentionActor(n_actions, seed=21).double()
    obs, feat, cnt, act, (dl, de, dv) = synth(R, K, n_actions, seed=3)
    w = P.weights_from_state_dict(actor.state_dict(), np.float64)
    lp, ent, v = torch_reference(actor, torch.from_numpy(obs).double(), torch.from_numpy(feat).double(),
                                 torch.from_numpy(cnt), torch.from_numpy(act))
    loss = (lp * torch.from_numpy(dl)).sum() + (ent * torch.from_numpy(de)).sum() + (v * torch.from_numpy(dv)).sum()
    want = torch.cat([g.reshape(-1) for g in torch.autograd.grad(loss, list(actor.parameters()))]).numpy()
    lp0, ent0, v0 = L.evaluate(w, obs, feat, cnt, act)
    np.testing.assert_allclose(lp0, lp.detach().numpy(), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(ent0, ent.detach().numpy(), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(v0, v.detach().numpy(), rtol=1e-9, atol=1e-12)
    got = L.evaluate_backward(w, obs, feat, cnt, act, dl, de, dv)
    assert got.shape == (abi.policy_n_params(n_actions),)
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("n_actions,size", [(5, 1864), (9, 2380)])
def test_vector_order_is_parameters_to_vector(n_actions, size):
    actor = GraphAttentionActor(n_actions, seed=4)
    vec = torch.nn.utils.parameters_to_vector(actor.parameters()).detach().numpy()
    assert vec.size == size == abi.policy_n_params(n_actions)
    np.testing.assert_array_equal(vec, L.to_vector(P.weights_from_state_dict(actor.state_dict())).astype(np.float32))
    sp = per_tensor(vec, n_actions)
    np.testing.assert_array_equal(sp["head_w"], actor.head.weight.detach().numpy())
    assert float(sp["att_b"]) == float(actor.att.bias.detach())


def test_eval_io_layout_matches_the_header(tmp_path):
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    fields = [n for n, _ in abi.GsmPolicyEvalIO._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "gsmarl_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(gsm_policy_eval_io));',
             '  printf("np5 %d\\n", GSM_POLICY_N_PARAMS(5));', '  printf("np9 %d\\n", GSM_POLICY_N_PARAMS(9));']
    lines += [f'  printf("{f} %zu\\n", offsetof(gsm_policy_eval_io, {f}));' for f in fields]
    lines += ['  return 0;', '}']
    (tmp_path / "l.c").write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(tmp_path / "l.c"),
                    "-o", str(tmp_path / "l")], check=True)
    got = dict(ln.split() for ln in subprocess.run([str(tmp_path / "l")], capture_output=True, text=True,
                                                   check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(abi.GsmPolicyEvalIO) == 96
    assert (int(got["np5"]), int(got["np9"])) == (1864, 2380)
    for f in fields:
        assert int(got[f]) == getattr(abi.GsmPolicyEvalIO, f).offset, f


def test_learner_bad_arguments_without_device():
    lib = abi.load_library()
    io = abi.GsmPolicyEvalIO()
    assert lib.gsm_policy_evaluate(None, 0, None) == -1
    assert lib.gsm_policy_evaluate(C.byref(io), 0, None) == -3                # struct_size 0
    io.struct_size, io.n_actions = C.sizeof(abi.GsmPolicyEvalIO), 4
    assert lib.gsm_policy_evaluate(C.byref(io), 0, None) == -4
    assert b"5 and 9" in lib.gsm_policy_last_error()
    io.n_actions = 5
    assert lib.gsm_policy_evaluate(C.byref(io), 0, None) == -1                # NULL pointers
    assert b"required" in lib.gsm_policy_last_error()
    # non-NULL placeholders: every check below fails before a pointer is dereferenced or a device touched
    io.params = io.obs = io.nbr_feat = io.nbr_cnt = io.actions = 256
    io.n_rows, io.max_nbrs = 100, 0
    assert lib.gsm_policy_evaluate(C.byref(io), 0, None) == -1                # max_nbrs < 1
    io.max_nbrs = 8
    need = lib.gsm_policy_backward_workspace(100, 5)
    assert need > 0 and need % (4 * 1864) == 0
    assert lib.gsm_policy_backward_workspace(100, 4) == -4 and lib.gsm_policy_backward_workspace(-1, 5) == -1
    assert lib.gsm_policy_backward(C.byref(io), None, None, None, None, 512, need, 0, None) == -1   # grad NULL
    assert lib.gsm_policy_backward(C.byref(io), None, None, None, 512, 512, need - 1, 0, None) == -1
    assert b"workspace" in lib.gsm_policy_last_error()
    assert lib.gsm_policy_backward(C.byref(io), None, None, None, 512, None, need, 0, None) == -1
    io.struct_size = 8
    assert lib.gsm_policy_backward(C.byref(io), None, None, None, 512, 512, need, 0, None) == -3
    io.struct_size, io.n_actions = C.sizeof(abi.GsmPolicyEvalIO), 9
    assert lib.gsm_policy_backward_workspace(100, 9) == need // 1864 * 2380
    io.n_rows = 0                                                            # no-op
    assert lib.gsm_policy_evaluate(C.byref(io), 0, None) == 0
    assert lib.gsm_policy_backward(C.byref(io), None, None, None, 512, None, 0, 0, None) == 0
    if not torch.cuda.is_available():
        io.n_rows = 4
        assert lib.gsm_policy_evaluate(C.byref(io), 0, None) == -5
        with pytest.raises(abi.GsmError):
            GraphAttentionActor(5).evaluate_actions(torch.zeros(4, 6), {"nbr_feat": torch.zeros(4, 8, 6),
                                                                        "nbr_cnt": torch.zeros(4, dtype=torch.int32)},
                                                    torch.zeros(4, dtype=torch.int32))


# ---- GPU --------------------------------------------------------------------------------------
DEV = "cuda"


def _gpu_inputs(R, K, n_actions, seed, nan_pad=False):
    obs, feat, cnt, act, up = synth(R, K, n_actions, seed)
    f = feat.copy()
    if nan_pad:
        f[np.arange(K)[None, :] >= cnt[:, None]] = np.nan
    to = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
    return (obs, feat, cnt, act, up), (to(obs), {"nbr_feat": to(f), "nbr_cnt": to(cnt)}, to(act),
                                      [to(u.astype(np.float32)) for u in up])


def _grads(actor):
    return torch.cat([p.grad.reshape(-1) for p in actor.parameters()])


def _assert_grad_close(got, want, n_actions, bar=1e-4):
    """||g - g_ref|| <= bar ||g_ref|| per parameter tensor.  The exact gradient of att_b is zero (the
    attention softmax is shift-invariant: sum_r ds_r = 0), so its fp32 value is rounding noise: it is held
    to the scale of the attention gradient it belongs to, ||g_ref[att_w]||."""
    g, w = per_tensor(got, n_actions), per_tensor(want, n_actions)
    bad = []
    for k in L.VECTOR_ORDER:
        err = np.linalg.norm(g[k] - w[k])
        ref = np.linalg.norm(w["att_w" if k == "att_b" else k])
        if not err <= bar * ref:
            bad.append((k, err, ref))
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("n_actions,R,K", [(5, 49152, 8), (9, 4097, 5), (5, 31, 1), (5, 1, 23)])
def test_evaluate_matches_oracle(n_actions, R, K):
    actor = GraphAttentionActor(n_actions, seed=5).to(DEV)
    (obs, feat, cnt, act, _), (o, g, a, _) = _gpu_inputs(R, K, n_actions, seed=6, nan_pad=True)
    with torch.no_grad():
        lp, ent, v = actor.evaluate_actions(o, g, a)
    lp0, ent0, v0 = L.evaluate(P.weights_from_state_dict(actor.state_dict()), obs, feat, cnt, act)
    for x, x0 in ((lp, lp0), (ent, ent0), (v, v0)):
        assert torch.isfinite(x).all()
        np.testing.assert_allclose(x.cpu().numpy(), x0, rtol=1e-4, atol=2e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("n_actions,R,K", [(5, 49152, 8), (9, 4097, 5), (5, 31, 1)])
def test_gradients_match_fp64_oracle(n_actions, R, K):
    """NaN in the padded rows (only the nbr_cnt valid rows may be read), random upstream gradients."""
    actor = GraphAttentionActor(n_actions, seed=7).to(DEV)
    (obs, feat, cnt, act, up), (o, g, a, ups) = _gpu_inputs(R, K, n_actions, seed=8, nan_pad=True)
    out = actor.evaluate_actions(o, g, a)
    torch.autograd.backward(out, ups)
    got = _grads(actor).cpu().numpy()
    assert np.isfinite(got).all()
    want = L.evaluate_backward(P.weights_from_state_dict(actor.state_dict()), obs, feat, cnt, act,
                               *[u.astype(np.float32) for u in up])
    _assert_grad_close(got, want, n_actions)


def _collected(scn, N, T=6, n_envs=500, seed=12):
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
    from gs_marl_b200.rollout import GraphRolloutBuffer, collect_fused
    cfg = make_cfg(scn, N, "f32").replace(episode_length=4)        # episodes restart inside the rollout
    actor = GraphAttentionActor(len(cfg.discrete_u), seed=seed).to(DEV)
    env = MultiAgentGraphConstrainEnv(cfg, n_envs, seed=3, auto_reset=True)
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    collect_fused(env, actor, buf, seed=5, first_step=10)
    torch.cuda.synchronize()
    return env, buf, actor


@pytest.mark.gpu
@pytest.mark.parametrize("scn,N", [("navigation", 3), ("polygon", 6)])
def test_evaluate_is_bit_identical_to_collection(scn, N):
    """logp and values over the buffer's slots == what gsm_collect wrote: PPO's first-epoch ratio is 1."""
    env, buf, actor = _collected(scn, N)
    with torch.no_grad():
        lp, ent, v = actor.evaluate_actions(buf["obs"][:-1], {"nbr_feat": buf["nbr_feat"][:-1],
                                                              "nbr_cnt": buf["nbr_cnt"][:-1]}, buf["actions"])
    assert torch.equal(lp, buf["logp"])
    assert torch.equal(v, buf["values"][:-1])
    assert bool((ent > 0).all())
    # the same through a shuffled row index over the flattened slots
    idx = torch.randperm(buf["logp"].numel(), device=DEV, generator=torch.Generator(DEV).manual_seed(0))
    with torch.no_grad():
        lp2, _, v2 = actor.evaluate_actions(buf["obs"][:-1].flatten(0, 2), {
            "nbr_feat": buf["nbr_feat"][:-1].flatten(0, 2), "nbr_cnt": buf["nbr_cnt"][:-1].flatten(0, 2)},
            buf["actions"].flatten(0, 2), rows=idx)
    assert torch.equal(lp2, buf["logp"].flatten()[idx]) and torch.equal(v2, buf["values"][:-1].flatten(0, 2)[idx])
    env.close()


@pytest.mark.gpu
def test_rows_index_equals_gathered_inputs():
    n_actions, R, K = 9, 20000, 8
    actor = GraphAttentionActor(n_actions, seed=9).to(DEV)
    _, (o, g, a, _) = _gpu_inputs(R, K, n_actions, seed=10, nan_pad=True)
    gen = torch.Generator(DEV).manual_seed(1)
    idx = torch.randint(0, R, (7777,), device=DEV, generator=gen)          # repeats included
    up = [torch.randn(7777, device=DEV, generator=gen), torch.randn(7777, device=DEV, generator=gen),
          torch.randn(7777, 2, device=DEV, generator=gen)]
    res = []
    for gathered in (False, True):
        actor.zero_grad(set_to_none=True)
        if gathered:
            out = actor.evaluate_actions(o[idx].contiguous(), {"nbr_feat": g["nbr_feat"][idx].contiguous(),
                                                               "nbr_cnt": g["nbr_cnt"][idx].contiguous()},
                                         a[idx].contiguous())
        else:
            out = actor.evaluate_actions(o, g, a, rows=idx)
        torch.autograd.backward(out, up)
        res.append([x.detach().clone() for x in out] + [_grads(actor).clone()])
    for x, y in zip(*res):
        assert torch.equal(x, y)
    with pytest.raises(IndexError):
        actor.evaluate_actions(o, g, a, rows=torch.tensor([0, R], device=DEV))
    with pytest.raises(ValueError):
        actor.evaluate_actions(o, g, a, rows=torch.tensor([0, 1], device=DEV, dtype=torch.int32))


@pytest.mark.gpu
def test_backward_is_deterministic_and_capturable():
    n_actions, R, K = 5, 30000, 8
    actor = GraphAttentionActor(n_actions, seed=11).to(DEV)
    _, (o, g, a, ups) = _gpu_inputs(R, K, n_actions, seed=12)
    idx = torch.randperm(R, device=DEV, generator=torch.Generator(DEV).manual_seed(2))[:12345]
    up = [u[:12345].contiguous() for u in ups]

    def step():
        actor.zero_grad(set_to_none=True)
        out = actor.evaluate_actions(o, g, a, rows=idx)
        torch.autograd.backward(out, up)
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
    """An EXAMPLE clipped-surrogate loss (the learner's loss is not part of this library) on a shuffled
    minibatch of a collected rollout: gradients through the kernels == through embed_autograd."""
    env, buf, actor = _collected("navigation", 3, T=8, n_envs=2000)
    with torch.no_grad():                                  # the learner has moved since collection
        for p in actor.parameters():
            p.add_(torch.randn(p.shape, device=DEV, generator=torch.Generator(DEV).manual_seed(p.numel())) * 3e-3)
    *_, vT = actor.act(buf["obs"][-1], buf.graph(buf.T), want_values=True)
    buf["values"][-1].copy_(vT)
    ret, adv = buf.compute_returns(0.99, 0.95)
    src = {"obs": buf["obs"][:-1].flatten(0, 2), "nbr_feat": buf["nbr_feat"][:-1].flatten(0, 2),
           "nbr_cnt": buf["nbr_cnt"][:-1].flatten(0, 2), "actions": buf["actions"].flatten(0, 2)}
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
                                         src["actions"], rows=idx)
        else:
            out = torch_reference(actor, src["obs"][idx], src["nbr_feat"][idx], src["nbr_cnt"][idx], src["actions"][idx])
        loss(*out).backward()
        grads.append(_grads(actor).double().cpu().numpy())
    _assert_grad_close(grads[0], grads[1], actor.n_actions)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_rows", [1, 127, 129])
def test_learner_kernels_write_nothing_outside_their_buffers(n_rows):
    """compute-sanitizer is not available: 4 KB guard bands around every output, grad and the workspace."""
    lib = abi.load_library()
    n_actions, R, K, G = 9, 300, 7, 4096
    actor = GraphAttentionActor(n_actions, seed=13).to(DEV)
    _, (o, g, a, _) = _gpu_inputs(R, K, n_actions, seed=14, nan_pad=True)
    params = torch.nn.utils.parameters_to_vector(actor.parameters()).detach().contiguous()
    rows = torch.randint(0, R, (n_rows,), device=DEV, generator=torch.Generator(DEV).manual_seed(4))
    nbytes = {"logp": 4 * n_rows, "entropy": 4 * n_rows, "values": 8 * n_rows, "grad": 4 * params.numel(),
              "ws": lib.gsm_policy_backward_workspace(n_rows, n_actions)}
    raw = {k: torch.full((n + 2 * G,), 0xA5, dtype=torch.uint8, device=DEV) for k, n in nbytes.items()}
    ptr = {k: r.data_ptr() + G for k, r in raw.items()}
    io = abi.GsmPolicyEvalIO()
    io.struct_size, io.n_actions = C.sizeof(abi.GsmPolicyEvalIO), n_actions
    io.params, io.obs, io.nbr_feat, io.nbr_cnt = params.data_ptr(), o.data_ptr(), g["nbr_feat"].data_ptr(), g["nbr_cnt"].data_ptr()
    io.actions, io.rows, io.n_rows, io.max_nbrs = a.data_ptr(), rows.data_ptr(), n_rows, K
    io.logp, io.entropy, io.values = ptr["logp"], ptr["entropy"], ptr["values"]
    st = torch.cuda.current_stream().cuda_stream
    d = [torch.randn(n_rows, device=DEV), torch.randn(n_rows, device=DEV), torch.randn(n_rows, 2, device=DEV)]
    assert lib.gsm_policy_evaluate(C.byref(io), 0, C.c_void_p(st)) == 0
    assert lib.gsm_policy_backward(C.byref(io), d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), ptr["grad"],
                                   ptr["ws"], nbytes["ws"], 0, C.c_void_p(st)) == 0
    torch.cuda.synchronize()
    for k, r in raw.items():
        assert bool((r[:G] == 0xA5).all()) and bool((r[-G:] == 0xA5).all()), f"{k}: guard band overwritten"
        if k != "ws":
            assert torch.isfinite(r[G:-G].view(torch.float32)).all(), k
