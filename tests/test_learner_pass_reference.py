"""The CUDA learner pass (`GraphAttentionActor.evaluate_actions`: gsm_policy_evaluate forward, gsm_policy_backward
backward) against a float64 torch reference on the CPU.

The reference is the module's own plain-torch definition (`embed_autograd`, `head`, `value`) on a float64 copy of
the actor, followed by log_softmax, the log-prob of the given action and the entropy; its gradients come from
torch.autograd.  The actor has ReLU units and two softmaxes (attention over the neighbour rows, the action
distribution): no tanh, so "saturation" here means softmaxes that are one-hot to fp32 and fp64 alike.  The
kernels return a gradient for the parameter vector only (obs / nbr_feat / actions are data, not parameters).

Tolerances (fp32 kernels, fp32 accumulation over at most 2H + 1 = 129 products per output):
  * forward: rtol 1e-4 and atol 2e-5 * max(1, max |logit|) (SPEC §12; the absolute part follows the scale of
    the logits, since log-probabilities are differences of logits);
  * backward: per parameter tensor ||g - g64|| <= 1e-4 ||g64|| (SPEC §12), att_b against ||g64[att_w]|| because
    its exact gradient is 0 (the attention softmax is shift-invariant).
"""
import numpy as np
import pytest
import torch

from gs_marl_b200 import abi
from gs_marl_b200.policy import GraphAttentionActor

H = abi.GSM_POLICY_HIDDEN
NAMES = ("ego.weight", "ego.bias", "nbr.weight", "nbr.bias", "att.weight", "att.bias", "head.weight", "head.bias",
         "value.weight", "value.bias")
BENCH_ROWS = 16384 * 3 * 25            # bench.py: 16384 envs x 3 agents x T = 25 slots of the rollout buffer
SMEM_OPTIN = 232448                    # sm_100: shared memory a block may opt in to (227 KB)


def max_nbrs_limit(n_actions):
    """The largest max_nbrs the backward kernel can launch with: its static shared memory (the weights and
    per-row state of 64 rows) plus 2 floats per neighbour row of its 64 rows must fit the opt-in limit."""
    n_params = abi.policy_n_params(n_actions)
    static = 4 * n_params + 64 * 4 * (6 + n_actions + 2 + 1 + 1) + 64 * 8
    return (SMEM_OPTIN - static) // (2 * 4 * 64)


# ---- inputs and the float64 reference ----------------------------------------------------------
def make_inputs(R, K, n_actions, seed, scale=1.0):
    """Rows whose neighbour counts cover 0 (no neighbour in range), K (every other entity seen) and values in
    between; actions biased to the ends of the range; per-row random loss weights."""
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(R, 6, generator=g) * scale
    feat = torch.randn(R, K, 6, generator=g) * scale
    cnt = torch.randint(0, K + 1, (R,), generator=g, dtype=torch.int32)
    kind = torch.randint(0, 4, (R,), generator=g)
    cnt = torch.where(kind == 0, 0, torch.where(kind == 1, K, cnt)).to(torch.int32)
    cnt[0] = K
    if R > 1:
        cnt[1] = 0
    feat[torch.arange(K)[None, :] >= cnt[:, None].long()] = 0
    act = torch.randint(0, n_actions, (R,), generator=g, dtype=torch.int32)
    edge = torch.randint(0, 3, (R,), generator=g)
    act = torch.where(edge == 0, 0, torch.where(edge == 1, n_actions - 1, act)).to(torch.int32)
    w = (torch.randn(R, generator=g), torch.randn(R, generator=g), torch.randn(R, 2, generator=g))
    return obs, feat, cnt, act, w


def reference(actor, obs, feat, cnt, act, w=None, chunk=65536):
    """float64 CPU: (logp, entropy, values, max |logit|) and, with loss weights w, the gradient of
    sum_i w0_i logp_i + w1_i entropy_i + w2_i . values_i for every parameter (dict by name)."""
    ref = GraphAttentionActor(actor.n_actions).double()
    ref.load_state_dict({k: v.detach().cpu().double() for k, v in actor.state_dict().items()})
    outs, zmax = [], 0.0
    for lo in range(0, obs.shape[0], chunk):
        sl = slice(lo, lo + chunk)
        emb = ref.embed_autograd(obs[sl].double(), {"nbr_feat": feat[sl].double(), "nbr_cnt": cnt[sl]})
        z = ref.head(emb)
        lp_all = torch.log_softmax(z, -1)
        logp = lp_all.gather(-1, act[sl].long()[:, None])[:, 0]
        ent = -(lp_all.exp() * lp_all).sum(-1)
        v = ref.value(emb)
        if w is not None:
            ((logp * w[0][sl].double()).sum() + (ent * w[1][sl].double()).sum() + (v * w[2][sl].double()).sum()).backward()
        outs.append([x.detach() for x in (logp, ent, v)])
        zmax = max(zmax, float(z.detach().abs().max()))
    res = [torch.cat(x) for x in zip(*outs)] + [zmax]
    if w is not None:
        res.append({n: p.grad.clone() for n, p in ref.named_parameters()})
    return res


def assert_grads_close(got, want, bar=1e-4):
    bad = []
    for n in NAMES:
        err = float((got[n].double().cpu() - want[n]).norm())
        scale = float(want["att.weight" if n == "att.bias" else n].norm())
        if not err <= bar * scale:
            bad.append((n, err, scale))
    assert not bad, bad


# ---- CPU: the reference itself -------------------------------------------------------------------
@pytest.mark.parametrize("n_actions,K", [(5, 1), (9, 7)])
def test_reference_matches_the_numpy_oracle(n_actions, K):
    """The torch reference against tests/_learner_oracle.py (fp64 numpy, analytic backward): two independent
    restatements of SPEC §12 agree to rounding, on rows with no neighbour and rows that see all K."""
    from oracle import policy_oracle as P
    from tests import _learner_oracle as L
    actor = GraphAttentionActor(n_actions, seed=2)
    obs, feat, cnt, act, w = make_inputs(301, K, n_actions, seed=3)
    assert (cnt == 0).any() and (cnt == K).any() and (act == 0).any() and (act == n_actions - 1).any()
    lp, ent, v, _, grads = reference(actor, obs, feat, cnt, act, w)
    wd = P.weights_from_state_dict(actor.state_dict(), np.float64)
    lp0, ent0, v0 = L.evaluate(wd, obs.numpy(), feat.numpy(), cnt.numpy(), act.numpy())
    for x, x0 in ((lp, lp0), (ent, ent0), (v, v0)):
        np.testing.assert_allclose(x.numpy(), x0, rtol=1e-12, atol=1e-12)
    g0 = L.evaluate_backward(wd, obs.numpy(), feat.numpy(), cnt.numpy(), act.numpy(), *[x.numpy() for x in w])
    got = torch.cat([grads[n].reshape(-1) for n in NAMES]).numpy()
    np.testing.assert_allclose(got, g0, rtol=1e-9, atol=1e-11)


# ---- GPU ------------------------------------------------------------------------------------------
DEV = "cuda"


def gpu(test):
    """A CUDA test: marked `gpu`, skipped where no device is visible (the reference-only tests above still run)."""
    return pytest.mark.gpu(pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")(test))


def kernel_pass(actor, obs, feat, cnt, act, w, nan_pad=True):
    """evaluate_actions + backward with the loss weights w: (logp, entropy, values, {name: grad})."""
    f = feat.clone()
    if nan_pad:                                         # only the nbr_cnt valid rows may be read
        f[torch.arange(f.shape[1])[None, :] >= cnt[:, None].long()] = float("nan")
    actor.zero_grad(set_to_none=True)
    lp, ent, v = actor.evaluate_actions(obs.to(DEV), {"nbr_feat": f.to(DEV), "nbr_cnt": cnt.to(DEV)}, act.to(DEV))
    torch.autograd.backward((lp, ent, v), [x.to(DEV).float() for x in w])
    return lp.detach().cpu(), ent.detach().cpu(), v.detach().cpu(), {n: p.grad.detach().clone() for n, p in actor.named_parameters()}


def assert_forward_close(got, want, zmax, ctx=""):
    atol = 2e-5 * max(1.0, zmax)
    for name, x, x0 in zip(("logp", "entropy", "values"), got, want):
        assert torch.isfinite(x).all(), (ctx, name)
        np.testing.assert_allclose(x.double().numpy(), x0.numpy(), rtol=1e-4, atol=atol, err_msg=f"{ctx} {name}")


SHAPES = [(5, 1, 1), (9, 1, "max"), (5, 997, 1), (9, 997, 7), (5, 997, "max"), (9, 613, "max"), (5, 4099, 7)]


@gpu
@pytest.mark.parametrize("n_actions,R,K", SHAPES)
def test_forward_and_backward_match_fp64_reference(n_actions, R, K):
    """Batch 1, batches that are not a multiple of the 32-lane warp, the 64-row backward tile or the 128-row
    forward block; neighbour counts 1, 7 and the largest the backward kernel can launch with.  Gradients of two
    identical calls must be bit-identical (the kernels are deterministic: no atomics, fixed reduction order)."""
    K = max_nbrs_limit(n_actions) if K == "max" else K
    actor = GraphAttentionActor(n_actions, seed=R + K).to(DEV)
    obs, feat, cnt, act, w = make_inputs(R, K, n_actions, seed=K)
    *want, zmax, gw = reference(actor, obs, feat, cnt, act, w)
    lp, ent, v, g1 = kernel_pass(actor, obs, feat, cnt, act, w)
    assert_forward_close((lp, ent, v), want, zmax, f"A={n_actions} R={R} K={K}")
    assert_grads_close(g1, gw)
    g2 = kernel_pass(actor, obs, feat, cnt, act, w)[3]
    for n in NAMES:
        assert torch.equal(g1[n], g2[n]), n


@gpu
def test_bench_sized_batch_matches_fp64_reference():
    """The rollout buffer of bench.py's workload in one pass: 16384 envs x 3 agents x 25 steps, K = 8."""
    actor = GraphAttentionActor(5, seed=1).to(DEV)
    obs, feat, cnt, act, w = make_inputs(BENCH_ROWS, 8, 5, seed=1)
    *want, zmax, gw = reference(actor, obs, feat, cnt, act, w)
    lp, ent, v, g = kernel_pass(actor, obs, feat, cnt, act, w)
    assert_forward_close((lp, ent, v), want, zmax, "bench rows")
    assert_grads_close(g, gw)


@gpu
@pytest.mark.parametrize("n_actions", [5, 9])
def test_saturated_softmaxes_match_fp64_reference(n_actions):
    """Inputs x300: logits hundreds apart (log-softmax one-hot, log-probs of -1e2..-1e3, entropy ~ 0) and attention
    scores hundreds apart (one neighbour row takes all the weight)."""
    actor = GraphAttentionActor(n_actions, seed=5).to(DEV)
    obs, feat, cnt, act, w = make_inputs(2051, 8, n_actions, seed=6, scale=300.0)
    *want, zmax, gw = reference(actor, obs, feat, cnt, act, w)
    assert zmax > 100 and float(want[0].min()) < -100 and float(want[1].min()) < 1e-6
    lp, ent, v, g = kernel_pass(actor, obs, feat, cnt, act, w)
    assert_forward_close((lp, ent, v), want, zmax, "saturated")
    assert_grads_close(g, gw)


@gpu
@pytest.mark.parametrize("n_actions", [5, 9])
def test_actions_outside_the_range(n_actions):
    """SPEC §12: an action outside [0, A) has no log-prob (NaN) and poisons the gradient only through its
    log-prob term: with that term's weight 0 the gradient is the reference's without those rows' log-prob."""
    actor = GraphAttentionActor(n_actions, seed=8).to(DEV)
    obs, feat, cnt, act, w = make_inputs(515, 5, n_actions, seed=9)
    bad = torch.zeros(515, dtype=torch.bool)
    bad[::5] = True
    act_bad = act.clone()
    act_bad[bad] = torch.tensor([-1, n_actions, 1 << 30, -(1 << 31)], dtype=torch.int32).repeat(200)[:int(bad.sum())]
    w0 = (torch.where(bad, 0.0, w[0]), w[1], w[2])
    *want, zmax, gw = reference(actor, obs, feat, cnt, act, w0)
    lp, ent, v, g = kernel_pass(actor, obs, feat, cnt, act_bad, w0)
    assert torch.isnan(lp[bad]).all()
    assert_forward_close((lp[~bad], ent, v), (want[0][~bad], want[1], want[2]), zmax, "out-of-range actions")
    assert_grads_close(g, gw)
    g_nan = kernel_pass(actor, obs, feat, cnt, act_bad, w)[3]               # the log-prob term has weight != 0
    assert torch.isnan(g_nan["head.weight"]).any()


@gpu
def test_max_nbrs_beyond_the_backward_limit_raises_and_leaves_the_library_usable():
    """One neighbour row more than the backward kernel's shared memory holds: a clean error before any launch,
    and the next calls work."""
    n_actions = 5
    K = max_nbrs_limit(n_actions)
    actor = GraphAttentionActor(n_actions, seed=3).to(DEV)
    obs, feat, cnt, act, w = make_inputs(70, K + 1, n_actions, seed=4)
    with pytest.raises(abi.GsmError):
        kernel_pass(actor, obs, feat, cnt, act, w)
    obs, feat, cnt, act, w = make_inputs(70, 3, n_actions, seed=4)
    *want, zmax, gw = reference(actor, obs, feat, cnt, act, w)
    lp, ent, v, g = kernel_pass(actor, obs, feat, cnt, act, w)
    assert_forward_close((lp, ent, v), want, zmax, "after the error")
    assert_grads_close(g, gw)
