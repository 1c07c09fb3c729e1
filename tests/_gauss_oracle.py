"""TEST INFRASTRUCTURE — fp64 numpy restatement of the Gaussian graph actor (SPEC.md §10b / §12b) that
gs_marl_b200/csrc/gsm_policy.cu implements as gsm_policy_act_gauss / gsm_policy_evaluate_gauss /
gsm_policy_backward_gauss: the sampled action (Box-Muller on the numpy Philox of
oracle.policy_oracle), the log-prob of given actions, the entropy, the two critics and the ANALYTIC
gradient of  sum_i d_logp[i] logp[i] + d_entropy[i] entropy[i] + d_values[i] . values[i]  with respect
to the parameter vector.  Independent of the product package (numpy only); pinned to torch autograd
of `GaussianGraphActor.dist_autograd` by tests/test_policy_gauss.py.
"""
from __future__ import annotations

import numpy as np

from oracle import policy_oracle as P

# Parameter-vector order = parameters_to_vector(GaussianGraphActor): log_std between head and critics.
VECTOR_ORDER = ("ego_w", "ego_b", "nbr_w", "nbr_b", "att_w", "att_b", "head_w", "head_b", "log_std",
                "value_w", "value_b")
D = 2
LOG_2PI = np.log(2 * np.pi)


def weights_from_state_dict(sd, dtype=np.float64):
    """oracle.policy_oracle's weights dict (head = the mean) plus log_std."""
    w = P.weights_from_state_dict(sd, dtype)
    ls = sd["log_std.weight"]
    w["log_std"] = np.asarray(ls.detach().cpu().numpy() if hasattr(ls, "detach") else ls, dtype)
    return w


def to_vector(w):
    return np.concatenate([np.asarray(w[k], np.float64).reshape(-1) for k in VECTOR_ORDER])


def split_vector(vec, H=64):
    shapes = {"ego_w": (H, 6), "ego_b": (H,), "nbr_w": (H, 6), "nbr_b": (H,), "att_w": (H,), "att_b": (),
              "head_w": (D, 2 * H), "head_b": (D,), "log_std": (D,), "value_w": (2, 2 * H), "value_b": (2,)}
    out, o = {}, 0
    for k in VECTOR_ORDER:
        n = int(np.prod(shapes[k], dtype=np.int64))
        out[k] = np.asarray(vec[o:o + n]).reshape(shapes[k])
        o += n
    assert o == len(vec), (o, len(vec))
    return out


def box_muller_eps(n_rows, seed, step, row_offset=0):
    """eps [R, 2] the kernel draws: words 0 and 1 of Philox4x32-10 with counter (row lo, row hi, step,
    0x80000000) and key (seed lo, seed hi), u = (x >> 9) 2^-23 + 2^-24 (exact), rho = sqrt(-2 log u0),
    eps = rho (cos 2 pi u1, sin 2 pi u1); fp64."""
    g = np.uint64(row_offset) + np.arange(n_rows, dtype=np.uint64)
    r = P.philox4x32_10(g & P.MASK, g >> np.uint64(32), np.full(n_rows, step & 0xFFFFFFFF, np.uint64),
                        np.full(n_rows, 0x80000000, np.uint64), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    u0, u1 = ((x >> np.uint32(9)).astype(np.float64) * 2.0 ** -23 + 2.0 ** -24 for x in r[:2])
    rho = np.sqrt(-2 * np.log(u0))
    return np.stack([rho * np.cos(2 * np.pi * u1), rho * np.sin(2 * np.pi * u1)], -1)


def _forward(w, obs, nbr_feat, nbr_cnt):
    w = {k: np.asarray(v, np.float64) for k, v in w.items()}
    obs, feat = np.asarray(obs, np.float64), np.asarray(nbr_feat, np.float64)
    K = feat.shape[1]
    cnt = np.clip(np.asarray(nbr_cnt), 0, K)
    valid = np.arange(K)[None, :] < cnt[:, None]
    feat = np.where(valid[..., None], feat, 0.0)                       # padded rows are never read
    pe = obs @ w["ego_w"].T + w["ego_b"]
    e = np.maximum(pe, 0)
    u = feat @ w["nbr_w"].T + w["nbr_b"]                                # [R,K,H]
    m = np.maximum(u, 0)
    sc = np.where(valid, m @ w["att_w"] + w["att_b"], -np.inf)
    mx = np.where(cnt > 0, sc.max(1, initial=-np.inf), 0.0)
    pr = np.where(valid, np.exp(sc - mx[:, None]), 0.0)
    a = pr / np.where(cnt > 0, pr.sum(1), 1.0)[:, None]                 # zero rows when cnt == 0
    h = np.concatenate([e, (a[..., None] * m).sum(1)], 1)
    return dict(w=w, obs=obs, feat=feat, valid=valid, pe=pe, u=u, m=m, a=a, h=h,
                mu=h @ w["head_w"].T + w["head_b"], v=h @ w["value_w"].T + w["value_b"])


def _logp(mu, log_std, actions):
    delta = (np.asarray(actions, np.float64) - mu) * np.exp(-log_std)
    return (-0.5 * delta ** 2 - log_std).sum(-1) - LOG_2PI, delta


def act(w, obs, nbr_feat, nbr_cnt, seed=0, step=0, row_offset=0, greedy=False):
    """SPEC.md §10b -> actions [R, 2], logp [R], mean [R, 2], values [R, 2] (fp64)."""
    f = _forward(w, obs, nbr_feat, nbr_cnt)
    mu, ls = f["mu"], f["w"]["log_std"]
    a = mu if greedy else mu + np.exp(ls) * box_muller_eps(mu.shape[0], seed, step, row_offset)
    return a, _logp(mu, ls, a)[0], mu, f["v"]


def evaluate(w, obs, nbr_feat, nbr_cnt, actions):
    """SPEC.md §12b forward -> logp [R] (of the given actions), entropy [R], values [R, 2] (fp64)."""
    f = _forward(w, obs, nbr_feat, nbr_cnt)
    ls = f["w"]["log_std"]
    ent = np.full(f["mu"].shape[0], (ls + 0.5 * (1 + LOG_2PI)).sum())
    return _logp(f["mu"], ls, actions)[0], ent, f["v"]


def evaluate_backward(w, obs, nbr_feat, nbr_cnt, actions, d_logp, d_entropy, d_values):
    """Analytic gradient (VECTOR_ORDER) of sum_i d_logp[i] logp[i] + d_entropy[i] entropy[i] +
    d_values[i] . values[i], fp64."""
    f = _forward(w, obs, nbr_feat, nbr_cnt)
    w, H = f["w"], f["pe"].shape[1]
    ls = w["log_std"]
    d_logp, d_entropy = np.asarray(d_logp, np.float64), np.asarray(d_entropy, np.float64)
    dv = np.asarray(d_values, np.float64)
    _, delta = _logp(f["mu"], ls, actions)
    dmu = d_logp[:, None] * delta * np.exp(-ls)
    g = {"head_w": dmu.T @ f["h"], "head_b": dmu.sum(0),
         "log_std": (d_logp[:, None] * (delta ** 2 - 1) + d_entropy[:, None]).sum(0),
         "value_w": dv.T @ f["h"], "value_b": dv.sum(0)}
    dh = dmu @ w["head_w"] + dv @ w["value_w"]
    de = dh[:, :H] * (f["pe"] > 0)                                      # ReLU'(0) = 0
    dg = dh[:, H:]
    g["ego_w"], g["ego_b"] = de.T @ f["obs"], de.sum(0)
    a, m = f["a"], f["m"]
    q = (m * dg[:, None, :]).sum(-1)                                    # m_r . dg
    ds = a * (q - (a * q).sum(1, keepdims=True))                        # softmax backward; 0 on padded rows
    dm = a[..., None] * dg[:, None, :] + ds[..., None] * w["att_w"]
    du = dm * (f["u"] > 0) * f["valid"][..., None]
    g["nbr_w"] = np.einsum("rkh,rkf->hf", du, f["feat"])
    g["nbr_b"] = du.sum((0, 1))
    g["att_w"] = (ds[..., None] * m).sum((0, 1))
    g["att_b"] = ds.sum()
    return to_vector(g)
