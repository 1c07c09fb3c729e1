"""The wide kernel's counted hot loop with in-kernel auto-reset, on the fp32 bulk path at the benchmark's size.

A fused rollout runs each warp's steps in segments that end at the first episode end in the warp; the
re-draw and the prologue pass that follows it happen inside the launch.  One-step rollouts from the same
state take none of those segment boundaries mid-launch.  Both must give the same bits.  Both paths share the
re-draw itself (Philox counters, extents), so an error there is caught by the oracle tests of
test_gpu_parity.py, not here."""
import numpy as np
import pytest
import torch

from tests._util import make_cfg, random_actions

pytestmark = pytest.mark.gpu

OUT_KEYS = ("obs", "nbr_idx", "nbr_feat", "nbr_cnt", "adj", "reward", "cost", "done", "assign")


@pytest.mark.parametrize("T", [25, 20])
def test_fused_auto_reset_equals_one_step_rollouts(T):
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
    cfg = make_cfg("navigation", 3, "f32", episode_length=25)
    B = 16384
    env = MultiAgentGraphConstrainEnv(cfg, B, seed=7)
    env.reset()
    # every env of a warp (4 envs) ends its episode at another step: several segments per launch
    ag0, lm0, _ = env.get_state()
    t0 = torch.arange(B, dtype=torch.int32) % cfg.episode_length
    env.set_state(ag0, lm0, t0)
    ag0, lm0, t0 = (x.clone() for x in env.get_state())
    ep0 = env.get_episode().clone()
    acts = random_actions(cfg, np.random.default_rng(T), (T, B))

    fused = {k: v.clone() for k, v in env.rollout(acts, auto_reset=True).items()}
    fused_state = [x.clone() for x in env.get_state()] + [env.get_episode().clone()]

    env.set_state(ag0, lm0, t0)
    env.set_episode(ep0)
    single = {k: [] for k in OUT_KEYS}
    for t in range(T):
        r = env.rollout(acts[t:t + 1], auto_reset=True)
        for k in OUT_KEYS:
            single[k].append(r[k].clone())
    single_state = [x.clone() for x in env.get_state()] + [env.get_episode().clone()]
    env.close()

    # env b ends its episode after step 25 - t0[b]: T of every 25 envs do so inside the rollout
    assert int(fused["done"].sum()) >= B * cfg.n_agents * (T - 1) // cfg.episode_length, "too few episode ends"
    for k in OUT_KEYS:
        s = torch.cat(single[k], 0)
        assert fused[k].shape == s.shape, k
        assert torch.equal(fused[k], s), (T, k, int((fused[k] != s).sum()))
    for name, a, b in zip(("agent_state", "landmark_pos", "t", "episode"), fused_state, single_state):
        assert torch.equal(a, b), (T, name)
