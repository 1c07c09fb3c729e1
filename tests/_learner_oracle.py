"""TEST INFRASTRUCTURE — fp64 numpy restatement of the learner pass (SPEC.md §12) that
gs_marl_b200/csrc/gsm_policy.cu implements as gsm_policy_evaluate / gsm_policy_backward: the
log-prob of given actions, the entropy and the two critics of the declared actor (SPEC.md §10),
and the ANALYTIC gradient of  sum_i d_logp[i] logp[i] + d_entropy[i] entropy[i] + d_values[i] . values[i]
with respect to the parameter vector.  Independent of the product package (numpy only); pinned to
torch autograd of the plain-torch formulation by tests/test_policy_learner.py.  Weights come as the
dict of oracle.policy_oracle.weights_from_state_dict.
"""
from __future__ import annotations

import numpy as np

# Parameter-vector order = parameters_to_vector(GraphAttentionActor).
VECTOR_ORDER = ("ego_w", "ego_b", "nbr_w", "nbr_b", "att_w", "att_b", "head_w", "head_b", "value_w", "value_b")


def to_vector(w):
    """weights dict -> the flat parameter vector (fp64)."""
    return np.concatenate([np.asarray(w[k], np.float64).reshape(-1) for k in VECTOR_ORDER])


def split_vector(vec, n_actions, H=64):
    """flat vector -> {name: array} with the shapes of weights_from_state_dict."""
    shapes = {"ego_w": (H, 6), "ego_b": (H,), "nbr_w": (H, 6), "nbr_b": (H,), "att_w": (H,), "att_b": (),
              "head_w": (n_actions, 2 * H), "head_b": (n_actions,), "value_w": (2, 2 * H), "value_b": (2,)}
    out, o = {}, 0
    for k in VECTOR_ORDER:
        n = int(np.prod(shapes[k], dtype=np.int64))
        out[k] = np.asarray(vec[o:o + n]).reshape(shapes[k])
        o += n
    assert o == len(vec), (o, len(vec))
    return out


def _learner_forward(w, obs, nbr_feat, nbr_cnt, actions):
    w = {k: np.asarray(v, np.float64) for k, v in w.items()}
    obs, feat = np.asarray(obs, np.float64), np.asarray(nbr_feat, np.float64)
    R, K = feat.shape[0], feat.shape[1]
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
    z = h @ w["head_w"].T + w["head_b"]
    v = h @ w["value_w"].T + w["value_b"]
    zm = z.max(1, keepdims=True)
    lse = zm[:, 0] + np.log(np.exp(z - zm).sum(1))
    logp_all = z - lse[:, None]
    p = np.exp(logp_all)
    ent = -(p * logp_all).sum(1)
    logp = logp_all[np.arange(R), np.asarray(actions)]
    return dict(w=w, obs=obs, feat=feat, valid=valid, pe=pe, e=e, u=u, m=m, a=a, h=h, p=p,
                logp_all=logp_all, logp=logp, ent=ent, v=v)


def evaluate(w, obs, nbr_feat, nbr_cnt, actions):
    """SPEC.md §12 forward, fp64 -> logp [R] (of the given actions), entropy [R], values [R, 2]."""
    f = _learner_forward(w, obs, nbr_feat, nbr_cnt, actions)
    return f["logp"], f["ent"], f["v"]


def evaluate_backward(w, obs, nbr_feat, nbr_cnt, actions, d_logp, d_entropy, d_values):
    """Analytic gradient of sum_i d_logp[i] logp[i] + d_entropy[i] entropy[i] + d_values[i] . values[i]
    with respect to the parameter vector (VECTOR_ORDER), fp64."""
    f = _learner_forward(w, obs, nbr_feat, nbr_cnt, actions)
    w, H = f["w"], f["e"].shape[1]
    R, A = f["p"].shape
    d_logp, d_entropy = np.asarray(d_logp, np.float64), np.asarray(d_entropy, np.float64)
    dv = np.asarray(d_values, np.float64)
    onehot = np.zeros((R, A))
    onehot[np.arange(R), np.asarray(actions)] = 1.0
    p = f["p"]
    dz = d_logp[:, None] * (onehot - p) - d_entropy[:, None] * p * (f["logp_all"] + f["ent"][:, None])
    g = {"head_w": dz.T @ f["h"], "head_b": dz.sum(0), "value_w": dv.T @ f["h"], "value_b": dv.sum(0)}
    dh = dz @ w["head_w"] + dv @ w["value_w"]
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
