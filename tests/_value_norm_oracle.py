"""TEST INFRASTRUCTURE — float64 numpy restatement of the value normaliser (SPEC.md §15): the lineage's
ValueNorm (utils/popart.py) per critic head, GAE on denormalised values, and the §14 seeds on normalised
targets through tests/_ppo_oracle.py.  gs_marl_b200/csrc/gsm_value_norm.cu, gae_kernel<true> and
backward_kernel<NA, KIND, LOSS_PPO_VNORM> are checked against it by tests/test_value_norm.py.
"""
from __future__ import annotations

import numpy as np

from tests import _ppo_oracle as O


class ValueNorm64:
    """running_mean, running_mean_sq, debiasing_term per head [2], all from 0."""

    def __init__(self, beta, epsilon, var_floor):
        self.beta, self.epsilon, self.var_floor = float(beta), float(epsilon), float(var_floor)
        self.state = np.zeros((2, 3))

    def update(self, R):
        """One update from a batch of returns R [n, 2]."""
        R = np.asarray(R, np.float64)
        b = self.beta
        mean, mean_sq = R.mean(0), (R ** 2).mean(0)
        self.state[:, 0] = b * self.state[:, 0] + (1 - b) * mean
        self.state[:, 1] = b * self.state[:, 1] + (1 - b) * mean_sq
        self.state[:, 2] = b * self.state[:, 2] + (1 - b)

    def affine(self):
        """[2, 2] (mu_h, sigma_h) in float64."""
        d = np.maximum(self.state[:, 2], self.epsilon)
        mu = self.state[:, 0] / d
        var = np.maximum(self.state[:, 1] / d - mu ** 2, self.var_floor)
        return np.stack([mu, np.sqrt(var)], 1)


def epoch(vn, returns, rows, num_mini_batch):
    """vn.update per minibatch of rows (the remainder left out): the fp32 affine snapshots [nmb, 2, 2]."""
    R = np.asarray(returns, np.float64).reshape(-1, 2)
    mb = len(rows) // num_mini_batch
    snaps = []
    for b in range(num_mini_batch):
        vn.update(R[np.asarray(rows[b * mb:(b + 1) * mb])])
        snaps.append(vn.affine().astype(np.float32))
    return np.array(snaps)


def normalize(R, affine):
    """(R - mu_h) / sigma_h in float64 with the (fp32) affine [2, 2]."""
    a = np.asarray(affine, np.float64)
    return (np.asarray(R, np.float64) - a[:, 0]) / a[:, 1]


def gae(reward, cost, values, done, gamma, lam, affine=None):
    """SPEC.md §11 in float64 over [T, rows] slots (values [T + 1, rows, 2]); with an affine the values are
    denormalised first, V * sigma_h + mu_h.  -> returns, advantages [T, rows, 2]."""
    v = np.asarray(values, np.float64)
    if affine is not None:
        a = np.asarray(affine, np.float64)
        v = v * a[:, 1] + a[:, 0]
    T = v.shape[0] - 1
    r = np.stack([np.asarray(reward, np.float64), np.asarray(cost, np.float64)], -1)
    mask = 1.0 - np.asarray(done, np.float64)[..., None]
    adv = np.zeros_like(r)
    g = np.zeros_like(r[0])
    for t in range(T - 1, -1, -1):
        delta = r[t] + gamma * v[t + 1] * mask[t] - v[t]
        g = delta + gamma * lam * mask[t] * g
        adv[t] = g
    return adv + v[:T], adv


def loss_grad(oracle, w, obs, feat, cnt, act, old_logp, old_v, R, A, moments, lam, affine, rows=None, **coefs):
    """tests/_ppo_oracle.py loss_grad with the value targets normalised by `affine` (§15)."""
    return O.loss_grad(oracle, w, obs, feat, cnt, act, old_logp, old_v, normalize(R, affine), A, moments, lam,
                       rows=rows, **coefs)
