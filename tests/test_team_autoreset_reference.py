"""The polygon / line kernel (env_team_kernel: G lanes per env, the per-step linear assignment, polygon-6 through
the exhaustive enumeration lsa_enum6 with scipy's procedure as the fallback) in fp32 with in-kernel auto-reset,
against the float64 restatement of SPEC.md §1-8 in tests/_env_reference.py (RefTeam: slots, cost matrix and
scipy.optimize.linear_sum_assignment).

The CPU tests pin the reference to the C oracle (oracle/gsm_oracle.py), tie-heavy starts included; the GPU tests
compare one fused launch of the kernel with it slot by slot (check_fused_f32), at bench.py's sizes.

The assignment is checked on the kernel's own post-step positions (obs[..., 2:4], exact fp32 values) and the
known markers, in fp64 with scipy.  The kernel solves the fp32 matrix, so where two assignments are within fp32
rounding of each other it may legitimately pick the other one (SPEC §9): there its fp64 total may exceed the
optimum by at most `near_tie_bound`, and obs[..., 4:6] and the reward must be those of its own assignment.
"""
import numpy as np
import pytest
import torch

from tests._env_reference import RefTeam, check_fused_f32, env_sample, squeezed_start, tie_heavy_start
from tests._util import make_cfg, random_actions

TEAMS = [("polygon", 3), ("polygon", 4), ("polygon", 5), ("polygon", 6), ("polygon", 12),
         ("line", 3), ("line", 4), ("line", 5), ("line", 6), ("line", 12)]


# ---- CPU: the reference against the C oracle -------------------------------------------------
@pytest.mark.parametrize("name,N", TEAMS)
@pytest.mark.parametrize("kw", [{}, {"share_reward": True, "max_nbrs": 2, "action_mode": "continuous"}])
def test_team_reference_rollout_equals_the_oracle(name, N, kw):
    """25 fp64 steps with staggered episode ends and re-draws (which move the markers and so the slots), from
    squeezed draws and tie-heavy starts (agents halfway between slots, agents on the slots in reversed order;
    nobody moves on the first step): integers bit-exact, reals within 1e-12."""
    from oracle import gsm_oracle as O
    cfg = make_cfg(name, N, "f64", episode_length=6, **kw)
    B, T, seed = 48, 25, 5
    ag, lm, t0 = squeezed_start(cfg, B, seed, np.arange(B) % 7)
    tie_heavy_start(cfg, ag, lm, np.arange(0, 8), np.arange(8, 16))
    t0[:16] = 0
    o = O.OracleEnv(cfg, B)
    o.set_state(ag, lm, t0)
    ref = RefTeam(cfg, ag, lm, t0, np.zeros(B), seed)
    acts = random_actions(cfg, np.random.default_rng(N), (T, B))
    acts[0, :16] = 0
    for s in range(T):
        want = o.step(acts[s])
        got = ref.step(acts[s])
        for k in ("nbr_idx", "nbr_cnt", "adj", "done", "assign", "cost"):
            assert (np.asarray(got[k]) == np.asarray(want[k]).astype(np.asarray(got[k]).dtype)).all(), (s, k)
        for k in ("obs", "nbr_feat", "reward"):
            np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=1e-12, err_msg=f"t={s} {k}")
        fin = ref.t >= cfg.episode_length
        ref.redraw(fin)
        if fin.any():
            o.reset(seed, fin.astype(np.uint8))
        np.testing.assert_allclose(ref.ag, o.agent_state, rtol=1e-12, atol=1e-12)
        assert (ref.lm == o.landmark_pos).all() and (ref.t == o.step_count).all() and (ref.ep == o.episode).all()


def test_team_reference_resolves_ties_like_the_oracle():
    """On the tie-heavy starts themselves (every optimum tied), RefTeam's assignment equals the oracle's
    restatement of scipy's procedure, for every team."""
    from oracle import gsm_oracle as O
    for name, N in TEAMS:
        cfg = make_cfg(name, N, "f64")
        B = 20
        ag, lm, t0 = squeezed_start(cfg, B, 3, np.zeros(B))
        tie_heavy_start(cfg, ag, lm, np.arange(10), np.arange(10, 20))
        ref = RefTeam(cfg, ag, lm, t0, np.zeros(B), 3)
        o = O.OracleEnv(cfg, B)
        o.set_state(ag, lm, t0)
        assert (ref.observe()["assign"] == o.evaluate()["assign"]).all(), (name, N)


# ---- GPU --------------------------------------------------------------------------------------
def gpu(test):
    """A CUDA test: marked `gpu`, skipped where no device is visible (the reference-only tests above still run)."""
    return pytest.mark.gpu(pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")(test))


def near_tie_bound(cfg, agent_pos, lm):
    """How far the fp64 total of an assignment the kernel found optimal on its fp32 matrix may exceed the fp64
    optimum, per env [B].  With X the largest coordinate magnitude in play (positions, markers, marker + radius)
    and u = 2^-23 max(X, 1) (one ulp of X, or of 1 for the unit-scale slot table):
      * an fp32 entry C32[i][k] = sqrt(dx^2 + dy^2) differs from the fp64 entry of the same fp32 positions by at
        most ~8u: the slot (R * table, rounded table and product: 1.5u; + marker: 0.5u), the difference dx
        (0.5u), the squares and sum with FMA (relative 1.5 ulp of C <= 3u for C <= 2X) and the IEEE sqrt (0.5u);
      * the two assignments' totals each sum N entries: |total32 - total64| <= 8Nu for either, so an fp32 optimum
        is within 16Nu of the fp64 one (2N entries);
      * the fp32 solver itself (scipy's procedure with rounded duals, one rounding per path-cost update and N
        augmentations) may stop above the fp32 optimum by ~8u per row: another 8Nu.
    Total 24Nu: 3.5e-5 for N = 6 at X = 2, while swapping two agents' slots away from a tie costs a fraction of
    a slot spacing (0.26 for polygon-12)."""
    X = np.abs(agent_pos).max((1, 2))
    X = np.maximum(X, np.abs(lm).max((1, 2)) + (cfg.polygon_radius if cfg.scenario == "polygon" else 0.0))
    return 24 * cfg.n_agents * 2.0 ** -23 * np.maximum(X, 1.0)


class AssignmentCheck:
    """assign_of hook of check_fused_f32: the kernel's assignment of each slot against scipy's on the kernel's
    own post-step positions.  Records the env-slots where the two differ (near-ties)."""

    def __init__(self, got):
        self.got, self.near_ties, self.env_slots = got, 0, 0

    def __call__(self, s, ref):
        a_k = self.got["assign"][s]
        N = a_k.shape[1]
        assert (np.sort(a_k, 1) == np.arange(N)).all(), f"t={s}: assign is not a permutation"
        P = self.got["obs"][s][..., 2:4].astype(np.float64)
        C = ref.cost_matrix(P)
        a_ref = RefTeam.solve(C)
        diff = (a_k != a_ref).any(1)
        if diff.any():
            tot = lambda a: np.take_along_axis(C[diff], a[diff][..., None].astype(np.int64), 2)[..., 0].sum(1)
            excess = tot(a_k) - tot(a_ref)
            bound = near_tie_bound(ref.cfg, P[diff], ref.lm[diff])
            bad = np.flatnonzero(excess > bound)
            assert bad.size == 0, (f"t={s}: {bad.size} envs with an assignment worse than scipy's by more than fp32 "
                                   f"rounding, e.g. excess {excess[bad[0]]:.3e} > {bound[bad[0]]:.3e}: "
                                   f"{a_k[diff][bad[0]]} vs {a_ref[diff][bad[0]]}")
        self.near_ties += int(diff.sum())
        self.env_slots += diff.size
        return np.where(diff[:, None], a_k, a_ref)      # score obs[..., 4:6] and reward with the kernel's own


CONFIGS3 = 16384                                        # bench.py configs[3]: polygon / line-6 / 12 x 16384

# (name, N, B, kw, env vars, envs the reference follows (0: all))
TEAM_CASES = [
    pytest.param("polygon", 6, CONFIGS3, {}, {}, 2048, id="polygon6-16384-enum6"),
    pytest.param("line", 6, CONFIGS3, {}, {}, 2048, id="line6-16384"),
    pytest.param("polygon", 12, CONFIGS3, {}, {}, 2048, id="polygon12-16384"),
    pytest.param("line", 12, CONFIGS3, {}, {}, 2048, id="line12-16384"),
    # G = 1 / G = 2 instances at a ragged batch
    *[pytest.param(n, N, 1001, {}, {}, 0, id=f"{n}{N}-1001") for n in ("polygon", "line") for N in (3, 4, 5)],
    # the non-default lane groupings
    pytest.param("polygon", 6, 1001, {}, {"GSM_TEAM_G": "2"}, 0, id="polygon6-G2"),
    pytest.param("polygon", 6, 1001, {}, {"GSM_TEAM_G": "3"}, 0, id="polygon6-G3"),
    pytest.param("line", 6, 1001, {}, {"GSM_TEAM_G": "2"}, 0, id="line6-G2"),
    pytest.param("line", 6, 1001, {}, {"GSM_TEAM_G": "3"}, 0, id="line6-G3"),
    pytest.param("polygon", 12, 1001, {}, {"GSM_TEAM_G": "6"}, 0, id="polygon12-G6"),
    pytest.param("line", 12, 1001, {}, {"GSM_TEAM_G": "6"}, 0, id="line12-G6"),
    # the switches
    pytest.param("polygon", 6, 1001, {"share_reward": True, "max_nbrs": 2}, {}, 0, id="polygon6-share-k2"),
    pytest.param("line", 6, 1001, {"action_mode": "continuous"}, {}, 0, id="line6-continuous"),
]


@gpu
@pytest.mark.parametrize("name,N,B,kw,env_vars,n_ref", TEAM_CASES)
def test_team_fused_auto_reset_rollout_f32_vs_reference(name, N, B, kw, env_vars, n_ref, monkeypatch):
    """One fused 25-step launch with auto-reset, episodes of 25 steps ending in every slot (counters 0..24), the
    first 80 envs on tie-heavy starts (nobody moves on the first step) so that polygon-6's enumeration falls back
    to scipy's procedure in warps that also re-draw.  Physics, graph, cost, done and the re-draw slot by slot,
    the assignment as the module docstring says; then the final state and counters."""
    for k, v in env_vars.items():
        monkeypatch.setenv(k, v)
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
    cfg = make_cfg(name, N, "f32", episode_length=25, **kw)
    T, seed = 25, 41
    t0 = np.arange(B) % 25
    ag, lm, t0 = squeezed_start(cfg, B, seed + 1, t0, scale=0.6)
    n_tie = min(80, B // 4)
    tie_heavy_start(cfg, ag, lm, np.arange(0, n_tie // 2), np.arange(n_tie // 2, n_tie))
    idx = env_sample(B, n_ref, t0, 128, seed=N)
    idx = np.union1d(idx, np.arange(n_tie))
    env = MultiAgentGraphConstrainEnv(cfg, B, seed=seed)
    env.reset()
    env.set_state(ag, lm, t0)
    ep = env.get_episode().cpu().numpy()
    ref = RefTeam(cfg, ag[idx], lm[idx], t0[idx], ep[idx], seed, genv=idx)
    acts = random_actions(cfg, np.random.default_rng(N), (T, B))
    acts[0, :n_tie] = 0
    out = env.rollout(acts, auto_reset=True)
    ti = torch.as_tensor(idx, device="cuda")
    got = {k: v.index_select(1, ti).cpu().numpy() for k, v in out.items()}
    got["adj"] = got["adj"].view(np.uint32)
    del out
    final = [x.index_select(0, ti).cpu().numpy() for x in list(env.get_state()) + [env.get_episode()]]
    env.close()
    chk = AssignmentCheck(got)
    checked, rows, ends = check_fused_f32(ref, got, acts[:, idx], f"{name}-{N} B={B}", assign_of=chk)
    print(f"[team f32 auto-reset] {name}-{N} B={B} {kw} {env_vars}: reference follows {idx.size} envs "
          f"({idx.size / B:.3f} of the batch), rows checked {checked / rows:.4f}, re-draws {int(ends.sum())}, "
          f"assignment near-ties {chk.near_ties} of {chk.env_slots} env-slots")
    assert checked > 0.5 * rows, (checked, rows)
    assert (ends > 0).all(), f"slots without a re-drawn env: {np.flatnonzero(ends == 0)}"
    assert chk.near_ties < 0.01 * chk.env_slots, (chk.near_ties, chk.env_slots)
    np.testing.assert_allclose(final[0], ref.ag, rtol=1e-4, atol=2e-5)
    assert (final[1] == ref.lm).all() and (final[2] == ref.t).all() and (final[3] == ref.ep).all()
