"""TEST INFRASTRUCTURE — fp64 numpy restatement of the PPO-Lagrangian loss (SPEC.md §14) that
gs_marl_b200/csrc/gsm_policy.cu fuses into backward_kernel<NA, KIND, true>: the seeds d_logp, d_entropy, d_values the loss
passes into the §12 chain, the loss statistics, and the gradient through tests/_learner_oracle.py or
tests/_gauss_oracle.py `evaluate_backward`.  numpy only; pinned to torch autograd of the §14 formula by
tests/test_ppo_update.py.
"""
from __future__ import annotations

import numpy as np

STAT_FIELDS = ("policy_loss", "value_loss_reward", "value_loss_cost", "entropy", "ratio", "clip_fraction",
               "approx_kl", "loss")


def adv_moments(adv):
    """(mu_0, sigma_0, mu_1, sigma_1): mean and population std over all rows, per head."""
    a = np.asarray(adv, np.float64).reshape(-1, 2)
    return np.array([a[:, 0].mean(), a[:, 0].std(), a[:, 1].mean(), a[:, 1].std()])


def seeds(logp, ent, v, old_logp, old_v, R, A, moments, lam, clip, value_clip, value_coef, entropy_coef):
    """-> d_logp [n], d_entropy [n], d_values [n, 2], stats [8], and the per-row rho and normalised advantage."""
    logp, ent, v = (np.asarray(x, np.float64) for x in (logp, ent, v))
    old_logp, old_v, R, A = (np.asarray(x, np.float64) for x in (old_logp, old_v, R, A))
    mu0, s0, mu1, s1 = (float(x) for x in moments)
    n = logp.shape[0]
    abar = (A[:, 0] - mu0) / (s0 + 1e-5) - lam * (A[:, 1] - mu1) / (s1 + 1e-5)
    rho = np.exp(logp - old_logp)
    surr1, surr2 = rho * abar, np.clip(rho, 1 - clip, 1 + clip) * abar
    d_logp = np.where(surr1 <= surr2, -surr1 / n, 0.0)
    vc = old_v + np.clip(v - old_v, -value_clip, value_clip)
    e1, e2 = v - R, vc - R
    inside = np.abs(v - old_v) <= value_clip          # the clipped branch's gradient passes where clip is inactive
    d_v = np.where(e1 ** 2 >= e2 ** 2, value_coef * e1 / n, np.where(inside, value_coef * e2 / n, 0.0))
    d_ent = np.full(n, -entropy_coef / n)
    lv = 0.5 * np.maximum(e1 ** 2, e2 ** 2)
    st = [-np.minimum(surr1, surr2).mean(), lv[:, 0].mean(), lv[:, 1].mean(), ent.mean(), rho.mean(),
          (np.abs(rho - 1) > clip).mean(), (old_logp - logp).mean()]
    st.append(st[0] + value_coef * (st[1] + st[2]) - entropy_coef * st[3])
    return d_logp, d_ent, d_v, np.array(st), rho, abar


def loss_grad(oracle, w, obs, feat, cnt, act, old_logp, old_v, R, A, moments, lam, rows=None, **coefs):
    """The §14 loss over source rows `rows` (None = all) with the fp64 actor oracle `oracle` (_learner_oracle or
    _gauss_oracle): (grad in vector order, stats [8], extras dict)."""
    idx = np.arange(len(cnt)) if rows is None else np.asarray(rows)
    g = lambda x: np.asarray(x)[idx]
    obs, feat, cnt, act = g(obs), g(feat), g(cnt), g(act)
    logp, ent, v = oracle.evaluate(w, obs, feat, cnt, act)
    d_logp, d_ent, d_v, st, rho, abar = seeds(logp, ent, v, g(old_logp), g(old_v), g(R), g(A), moments, lam, **coefs)
    grad = oracle.evaluate_backward(w, obs, feat, cnt, act, d_logp, d_ent, d_v)
    return grad, st, dict(logp=logp, ent=ent, v=v, rho=rho, abar=abar, d_logp=d_logp, d_v=d_v)
