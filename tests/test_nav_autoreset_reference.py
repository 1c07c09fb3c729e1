"""The navigation kernels with in-kernel auto-reset against the float64 numpy restatement of SPEC.md §2-8 in
tests/_env_reference.py:
  * the wide kernel (env_wide_kernel: navigation with 3, 4 or 5 agents), fp64 and fp32;
  * the lane kernel (env_lane_kernel: one lane per agent, N >= 6), fp32, with and without CARRY (the contact force
    of step s + 1 summed in the graph phase of step s; on for N >= 48), at the sizes bench.py runs it.

The reference shares no code with the kernels or with the C oracle: Philox4x32-10, the spawn draw, the contact
force, the integration, the graph, reward, cost, done and the auto-reset rule are all restated there, vectorised
over envs.  The CPU tests pin it to the C oracle (oracle/gsm_oracle.py), so a fault in the reference cannot hide
a fault in the kernel; the GPU tests compare the kernel with it over multi-step rollouts.

Auto-reset conventions (environment.py):
  * fused rollout (`rollout(auto_reset=True)`): an env that finishes on step s keeps its TERMINAL outputs in
    slot s and starts step s + 1 from the SPEC §8 draw of its episode counter, which then advances;
  * `step()` with `auto_reset=True`: reward, cost and done are the terminal step's, obs and graph rows of a
    finished env are the FIRST observation of its new episode.
"""
import numpy as np
import pytest
import torch

from tests._env_reference import (F32_TOL, RefNav, assert_step, check_fused_f32, env_sample, philox4x32_10,
                                  ref_fused_rollout, spawn_draw, squeezed_start)
from tests._util import make_cfg, random_actions

# fp64 kernels round every SPEC operation once (-fmad=false); they differ from this reference only in libm's
# last ulp and in the order in which pair forces are summed, which the stiff contacts amplify over 25 steps
# to well below 1e-9 (SPEC §9).
F64_TOL = dict(rtol=1e-9, atol=1e-9)
BENCH_ENVS = 16384                     # bench.py ENVS_PER_GPU: navigation-3, one launch of T = 25


# ---- CPU: the reference against the C oracle -------------------------------------------------
def test_philox_and_spawn_draw_equal_the_oracle():
    from oracle import gsm_oracle as O
    rng = np.random.default_rng(0)
    c = rng.integers(0, 2 ** 32, (6, 257), dtype=np.uint64)
    c[:, 0] = 0
    c[:, 1] = 2 ** 32 - 1
    got = np.stack(philox4x32_10(*c)).astype(np.uint32)                 # [4, 257]
    for i in range(c.shape[1]):
        assert (got[:, i] == O.philox(*[int(x) for x in c[:, i]])).all(), i
    for N in (3, 4, 5):
        cfg = make_cfg("navigation", N, "f64")
        o = O.OracleEnv(cfg, 37, env_offset=2 ** 32 - 5)                  # global env index crosses 2^32
        o.episode[:] = rng.integers(0, 1000, 37)
        ep0 = o.episode.copy()
        mask = (np.arange(37) % 3 != 1).astype(np.uint8)
        o.reset(2 ** 40 + 77, mask)
        ref = RefNav(cfg, np.zeros((37, N, 4)), np.zeros((37, cfg.n_landmarks, 2)), np.full(37, 9), ep0,
                     2 ** 40 + 77, env_offset=2 ** 32 - 5)
        ref.redraw(mask.astype(bool))
        m = mask.astype(bool)
        assert (ref.ag[m] == o.agent_state[m]).all() and (ref.lm[m] == o.landmark_pos[m]).all()
        assert (ref.ep == o.episode).all() and (ref.t[m] == 0).all() and (ref.t[~m] == 9).all()


@pytest.mark.parametrize("N,kw", [(3, {}), (4, {"share_reward": True}), (5, {"max_nbrs": 6}),
                                  (3, {"max_nbrs": 3, "own_goal_always": False, "cost_obstacles": False}),
                                  # the lane kernel's teams: 6, 12, 24; 33 with 66 entities (3 adjacency words,
                                  # K > 32); 48 with 144 entities (5 words) and K truncation at 32
                                  (6, {}), (12, {}), (24, {}), (33, {"n_obstacles": 0, "max_nbrs": 65}),
                                  (48, {"max_nbrs": 32}),
                                  (12, {"share_reward": True, "own_goal_always": False, "cost_obstacles": False,
                                        "action_mode": "continuous"})])
def test_reference_rollout_equals_the_oracle(N, kw):
    """25 fp64 steps with staggered episode ends and re-draws: the reference against the C oracle."""
    from oracle import gsm_oracle as O
    cfg = make_cfg("navigation", N, "f64", episode_length=6, **kw)
    B, T, seed = 64, 25, 3
    ag, lm, t0 = squeezed_start(cfg, B, seed, np.arange(B) % 7)
    o = O.OracleEnv(cfg, B)
    o.set_state(ag, lm, t0)
    ref = RefNav(cfg, ag, lm, t0, np.zeros(B), seed)
    acts = random_actions(cfg, np.random.default_rng(N), (T, B))
    acts[:, 0] = -1                                                     # out of range: no control
    hits = 0
    for s in range(T):
        want = o.step(acts[s])
        got = ref.step(acts[s])
        for k in ("nbr_idx", "nbr_cnt", "adj", "done", "assign", "cost"):
            assert (np.asarray(got[k]) == np.asarray(want[k]).astype(np.asarray(got[k]).dtype)).all(), (s, k)
        for k in ("obs", "nbr_feat", "reward"):
            np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=1e-12, err_msg=f"t={s} {k}")
        hits += int(want["cost"].sum())
        fin = ref.t >= cfg.episode_length
        ref.redraw(fin)
        if fin.any():
            o.reset(seed, fin.astype(np.uint8))
        np.testing.assert_allclose(ref.ag, o.agent_state, rtol=1e-12, atol=1e-12)
        assert (ref.lm == o.landmark_pos).all() and (ref.t == o.step_count).all() and (ref.ep == o.episode).all()
    assert hits > 0, "no collision: the contact term was never exercised"


# ---- GPU --------------------------------------------------------------------------------------
def gpu(test):
    """A CUDA test: marked `gpu`, skipped where no device is visible (the reference-only tests above still run)."""
    return pytest.mark.gpu(pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")(test))


def _env(cfg, B, **kw):
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
    return MultiAgentGraphConstrainEnv(cfg, B, **kw)


def _np(bufs, idx=None):
    """Host copies of [T, B, ...] outputs, only the envs `idx` (gathered on the device) if given."""
    out = {}
    for k, v in bufs.items():
        if idx is not None:
            v = v.index_select(1, torch.as_tensor(idx, device=v.device))
        a = v.detach().cpu().numpy()
        out[k] = a.view(np.uint32) if k == "adj" else a
    return out


def _state(env, idx=None):
    """(agent_state, landmark_pos, t, episode) as numpy, only the envs `idx` if given."""
    xs = list(env.get_state()) + [env.get_episode()]
    if idx is not None:
        xs = [x.index_select(0, torch.as_tensor(idx, device=x.device)) for x in xs]
    return [x.cpu().numpy() for x in xs]


def _staggered_env(cfg, B, seed, t0, idx=None):
    """An env at a squeezed SPEC §8 draw with step counters t0, and the reference of its envs `idx` (all)."""
    env = _env(cfg, B, seed=seed)
    ag, lm, t = squeezed_start(cfg, B, seed + 1, t0)
    env.reset()
    env.set_state(ag, lm, t)
    idx = np.arange(B) if idx is None else np.asarray(idx)
    return env, RefNav(cfg, ag[idx], lm[idx], t[idx], env.get_episode().cpu().numpy()[idx], seed, genv=idx)


def _lane_envs_per_cta(N):
    return 1 if N > 32 else 32 // N * 4            # gsm_kernels_lane.cuh lane_geom


def _setenv(monkeypatch, env_vars):
    for k, v in env_vars.items():
        monkeypatch.setenv(k, v)


@gpu
@pytest.mark.parametrize("B", [1, 37, 1000])
@pytest.mark.parametrize("N,kw", [(3, {}), (4, {"share_reward": True}), (5, {}), (3, {"max_nbrs": 3})])
def test_fused_auto_reset_rollout_f64_vs_reference(N, kw, B):
    """fp64 instance, one fused launch of 25 steps with episodes of 6 steps ending at staggered steps
    (counters 0..7: some envs start at or past their end): every output of every slot, the final state,
    the step and episode counters.  B = 1 and 37 leave warps partly idle; 1000 is not a multiple of the envs
    per CTA (16 / 8 / 8 for N = 3 / 4 / 5)."""
    cfg = make_cfg("navigation", N, "f64", episode_length=6, **kw)
    T = 25
    env, ref = _staggered_env(cfg, B, 11 + B, np.arange(B) % 8)
    acts = random_actions(cfg, np.random.default_rng(B + N), (T, B))
    got = _np(env.rollout(acts, auto_reset=True))
    want, redrawn = ref_fused_rollout(ref, acts)
    ok = np.ones((B, N), bool)
    for s in range(T):
        assert_step({k: got[k][s] for k in got}, want[s], ok, F64_TOL, f"N={N} B={B} t={s}")
    ag, lm, t = (x.cpu().numpy() for x in env.get_state())
    np.testing.assert_allclose(ag, ref.ag, **F64_TOL)
    assert (lm == ref.lm).all() and (t == ref.t).all()
    assert (env.get_episode().cpu().numpy() == ref.ep).all()
    assert np.stack(redrawn).sum() >= B * (T // 6), "too few episode ends"
    env.close()


# lane-kernel instances: (N, kw, env vars) -> what the case reaches
LANE_12 = (12, {}, {})                                                 # 2 envs per warp
LANE_48 = (48, {"max_nbrs": 32}, {})                                   # CARRY, env spans 2 warps
LANE_12_CARRY = (12, {}, {"GSM_LANE_CARRY_MIN_N": "6"})                # CARRY, envs of a warp end on different steps


@gpu
@pytest.mark.parametrize("dtype,N,kw,env_vars", [
    pytest.param("f64", 3, {}, {}, id="f64-3"), pytest.param("f64", 4, {}, {}, id="f64-4"),
    pytest.param("f64", 5, {}, {}, id="f64-5"), pytest.param("f64", *LANE_12, id="f64-lane12"),
    pytest.param("f32", 3, {}, {}, id="f32-3"), pytest.param("f32", 4, {}, {}, id="f32-4"),
    pytest.param("f32", 5, {}, {}, id="f32-5"), pytest.param("f32", *LANE_12, id="f32-lane12"),
    pytest.param("f32", 24, {"max_nbrs": 32}, {}, id="f32-lane24"), pytest.param("f32", *LANE_48, id="f32-lane48-carry"),
    pytest.param("f32", *LANE_12_CARRY, id="f32-lane12-carry")])
def test_only_finished_envs_are_redrawn(dtype, N, kw, env_vars, monkeypatch):
    """Half of the envs finish on step 2 of a 5-step launch, the other half never: the finished ones restart
    from the SPEC §8 draw of their episode (bit for bit: the draw is integer + exact fp64 arithmetic, rounded to
    the state's precision), the others are untouched — every output and the final state equal the same launch
    without auto-reset.  fp64 runs free against the reference, fp32 slot by slot (check_fused_f32)."""
    _setenv(monkeypatch, env_vars)
    cfg = make_cfg("navigation", N, dtype, episode_length=10, **kw)
    B, T, seed = 203, 5, 21
    fin_env = np.arange(B) % 2 == 0
    t0 = np.where(fin_env, 8, 0)                                     # 8 + 2 = 10: done on step index 1
    env, ref = _staggered_env(cfg, B, seed, t0)
    ag0, lm0, tt0 = (x.clone() for x in env.get_state())
    ep0 = env.get_episode().clone()
    acts = random_actions(cfg, np.random.default_rng(N), (T, B))
    ar = _np(env.rollout(acts, auto_reset=True))
    ar_state = _state(env)
    env.set_state(ag0, lm0, tt0)
    env.set_episode(ep0)
    plain = _np(env.rollout(acts, auto_reset=False))
    plain_state = _state(env)
    env.close()

    if dtype == "f64":
        want, redrawn = ref_fused_rollout(ref, acts)
        for s in range(T):
            assert_step({k: ar[k][s] for k in ar}, want[s], np.ones((B, N), bool), F64_TOL, f"N={N} t={s}")
        redrawn = [r.sum() for r in redrawn]
    else:
        checked, rows, redrawn = check_fused_f32(ref, ar, acts, f"N={N}")
        assert checked > 0.5 * rows, (checked, rows)
    assert redrawn[1] == fin_env.sum() and sum(redrawn) == redrawn[1]
    # the re-draw itself: finished envs end the launch at t = 3 from positions drawn in episode ep0 + 0
    draw = spawn_draw(cfg, np.arange(B), ep0.cpu().numpy(), seed).astype(cfg.np_real)
    assert (ar_state[1][fin_env] == draw[fin_env, N:]).all(), "landmarks of a finished env are not its re-draw"
    assert (ar_state[1][~fin_env] == lm0.cpu().numpy()[~fin_env]).all(), "an unfinished env's landmarks moved"
    assert (ar_state[2] == np.where(fin_env, T - 2, t0 + T)).all()
    assert (ar_state[3] == ep0.cpu().numpy() + fin_env).all(), "episode counters"
    # slot 1 of a finished env holds its terminal observation, slot 2 the first step of the new episode
    assert ar["done"][1][fin_env].all() and not ar["done"][1][~fin_env].any()
    assert (ar["obs"][1] == plain["obs"][1]).all(), "the terminal observation must stay in its slot"
    # envs that never finish: bit-identical to the plain instance in every slot and in the final state
    for k in ar:
        assert (ar[k][:, ~fin_env] == plain[k][:, ~fin_env]).all(), k
    for a, p in zip(ar_state[:3], plain_state[:3]):
        assert (a[~fin_env] == p[~fin_env]).all()


@gpu
@pytest.mark.parametrize("N", [3, 4, 5])
def test_step_api_auto_reset_returns_the_reset_observation(N):
    """`step()` with auto_reset: reward / cost / done of the terminal step, obs and graph rows of the finished
    envs from the first state of the new episode, the other envs' rows from the step."""
    cfg = make_cfg("navigation", N, "f64", episode_length=4)
    B, seed = 45, 8
    t0 = np.arange(B) % 4
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
    env = MultiAgentGraphConstrainEnv(cfg, B, seed=seed, auto_reset=True)
    env.reset()
    ag, lm, t = squeezed_start(cfg, B, seed + 1, t0)
    env.set_state(ag, lm, t)
    ref = RefNav(cfg, ag, lm, t, env.get_episode().cpu().numpy(), seed)
    rng = np.random.default_rng(N)
    for s in range(6):
        a = random_actions(cfg, rng, (B,))
        obs, graph, rew, cost, done, infos = env.step(a)
        got = _np(dict(obs=obs, reward=rew, cost=cost, done=done, assign=infos["assign"], **graph))
        want = ref.step(a)
        fin = ref.t >= cfg.episode_length
        ref.redraw(fin)
        first = ref.observe()
        for k in ("obs", "nbr_idx", "nbr_feat", "nbr_cnt", "adj"):
            want[k] = np.where(fin.reshape((B,) + (1,) * (want[k].ndim - 1)), first[k], want[k])
        assert_step(got, want, np.ones((B, N), bool), F64_TOL, f"N={N} step {s}")
        assert (got["done"].all(1) == fin).all()
    env.close()


@gpu
@pytest.mark.parametrize("N,B,kw,env_vars,T", [
    pytest.param(3, BENCH_ENVS, {}, {}, 25, id="25"), pytest.param(3, BENCH_ENVS, {}, {}, 7, id="7"),
    pytest.param(6, 1001, {}, {}, 25, id="lane6-1001"), pytest.param(12, 8192, {}, {}, 25, id="lane12-8192"),
    pytest.param(24, 4096, {"max_nbrs": 32}, {}, 25, id="lane24-4096"),
    pytest.param(48, 4096, {"max_nbrs": 32}, {}, 25, id="lane48-4096-carry"),
    pytest.param(96, 4096, {"max_nbrs": 32}, {}, 25, id="lane96-4096-carry"),
    pytest.param(*LANE_12_CARRY[:1], 1003, *LANE_12_CARRY[1:], 25, id="lane12-1003-carry")])
def test_auto_reset_instance_equals_plain_instance_when_nothing_finishes(N, B, kw, env_vars, T, monkeypatch):
    """The benchmark's instances (wide <float, 3, 6, auto-reset, K = 8>; lane <float, auto-reset, CARRY>) against
    the plain ones at the bench sizes: with no episode ending inside the launch, the two must give the same bits
    in every output and the final state."""
    _setenv(monkeypatch, env_vars)
    cfg = make_cfg("navigation", N, "f32", episode_length=1000, **kw)
    env = _env(cfg, B, seed=4)
    env.reset()
    rng = np.random.default_rng(T)
    env.set_state(None, None, rng.integers(0, 1000 - T, B).astype(np.int32))
    s0 = [x.clone() for x in env.get_state()]
    acts = random_actions(cfg, rng, (T, B))
    res = []
    for ar in (True, False):
        env.set_state(*s0)
        out = env.rollout(acts, auto_reset=ar)
        res.append([v.clone() for k, v in sorted(out.items()) if k != "actions"] + [x.clone() for x in env.get_state()])
        del out
    env.close()
    assert not bool(res[0][sorted(env.OUTPUTS).index("done")].any())
    for k, a, b in zip(sorted(env.OUTPUTS) + ["agent_state", "landmark_pos", "t"], *res):
        assert torch.equal(a, b), k


# fp32 cases: (N, B, kw, env vars, envs the reference follows (0: all)) -> what the case reaches
F32_CASES = [
    pytest.param(3, BENCH_ENVS, {}, {}, 0, id="3-16384"), pytest.param(3, 1, {}, {}, 0, id="3-1"),
    pytest.param(4, 1001, {}, {}, 0, id="4-1001"), pytest.param(5, 999, {}, {}, 0, id="5-999"),
    # lane kernel, plain: 5 envs per warp with 2 idle lanes and a ragged last CTA; 2 envs per warp at configs[4]'s
    # share and ragged (the 16 + 8-byte row stores); one env per warp (configs[2]); an env over 2 warps with 31
    # idle lanes, 3 adjacency words, K = 65 > 32
    pytest.param(6, 1001, {}, {}, 0, id="lane6-1001"),
    pytest.param(12, 8192, {}, {}, 512, id="lane12-8192"), pytest.param(12, 1003, {}, {}, 0, id="lane12-1003"),
    pytest.param(24, 4096, {"max_nbrs": 32}, {}, 256, id="lane24-4096"),
    pytest.param(33, 67, {"n_obstacles": 0, "max_nbrs": 65}, {}, 0, id="lane33-67"),
    # CARRY + auto-reset (configs[2]): multi-warp envs, 5 / 9 adjacency words, K truncation at 32
    pytest.param(48, 4096, {"max_nbrs": 32}, {}, 256, id="lane48-4096-carry"),
    pytest.param(96, 4096, {"max_nbrs": 32}, {}, 256, id="lane96-4096-carry"),
    # CARRY with several envs per warp that finish on different steps
    pytest.param(*LANE_12_CARRY[:1], 1003, *LANE_12_CARRY[1:], 0, id="lane12-1003-carry"),
    pytest.param(24, 1024, {"max_nbrs": 32}, {"GSM_LANE_CARRY_MIN_N": "6"}, 256, id="lane24-1024-carry"),
    # CARRY instance with carry_ok false (contact reach beyond the sensing radius: sweep every step)
    pytest.param(48, 512, {"max_nbrs": 32, "sensing_radius": 0.33}, {}, 128, id="lane48-carry-sweep"),
    # col_in_nb false: the candidate test also takes the contact distance
    pytest.param(24, 1024, {"max_nbrs": 32, "sensing_radius": 0.3}, {}, 256, id="lane24-contact-candidates"),
    # a re-draw after every step: the carried force is never valid
    pytest.param(48, 512, {"max_nbrs": 32, "episode_length": 1}, {}, 128, id="lane48-carry-ep1"),
    # the switches
    pytest.param(12, 1003, {"share_reward": True, "action_mode": "continuous", "cost_obstacles": False,
                            "own_goal_always": False}, {}, 0, id="lane12-switches"),
]


@gpu
@pytest.mark.parametrize("N,B,kw,env_vars,n_ref", F32_CASES)
def test_fused_auto_reset_rollout_f32_vs_reference(N, B, kw, env_vars, n_ref, monkeypatch):
    """fp32 production instances over one 25-step fused launch with staggered episode ends (the benchmark's
    shapes: navigation-3 x 16384 on the wide kernel, navigation-12 / 24 / 48 / 96 on the lane kernel), slot by
    slot against the reference (check_fused_f32: one reference step from the kernel's own state of the slot
    before).  At the large sizes the kernel runs the whole batch and the reference follows a seeded sample of
    n_ref envs that includes the last CTA's envs and envs that finish in every slot.  Then the final state, step
    and episode counters of those envs."""
    _setenv(monkeypatch, env_vars)
    kw = dict(kw)
    cfg = make_cfg("navigation", N, "f32", episode_length=kw.pop("episode_length", 25), **kw)
    T, seed = 25, 31
    t0 = np.arange(B) % cfg.episode_length
    idx = env_sample(B, n_ref, t0, _lane_envs_per_cta(N) if N >= 6 else 16, seed=N)
    env, ref = _staggered_env(cfg, B, seed, t0, idx)
    acts = random_actions(cfg, np.random.default_rng(N), (T, B))
    got = _np(env.rollout(acts, auto_reset=True), idx)
    final = _state(env, idx)
    env.close()
    checked, rows, ends = check_fused_f32(ref, got, acts[:, idx], f"N={N} B={B}")
    print(f"[f32 auto-reset] N={N} B={B} {kw} {env_vars}: reference follows {idx.size} envs "
          f"({idx.size / B:.3f} of the batch), rows checked {checked / rows:.4f}, re-draws {int(ends.sum())}")
    assert checked > 0.5 * rows, (checked, rows)
    if idx.size >= cfg.episode_length:
        assert (ends > 0).all(), f"slots without a re-drawn env: {np.flatnonzero(ends == 0)}"
    else:
        assert ends.sum() >= idx.size * (T - 1) // cfg.episode_length
    # final state: restarted-and-stepped envs within fp32 rounding, the counters exactly
    np.testing.assert_allclose(final[0], ref.ag, **F32_TOL)
    assert (final[1] == ref.lm).all() and (final[2] == ref.t).all() and (final[3] == ref.ep).all()


@gpu
def test_env_host_checks_reject_wrong_shapes():
    """set_state / reset(mask) / rollout(out=...) copy or write n_envs (x T) rows: a wrong shape must raise
    before anything touches the device."""
    cfg = make_cfg("navigation", 3, "f32")
    env = _env(cfg, 20)
    env.reset()
    with pytest.raises(ValueError):
        env.set_state(np.zeros((19, 3, 4), np.float32))
    with pytest.raises(ValueError):
        env.set_state(None, np.zeros((20, 5, 2), np.float32))
    with pytest.raises(ValueError):
        env.set_state(None, None, np.zeros(21, np.int32))
    with pytest.raises(ValueError):
        env.reset(torch.ones(10, dtype=torch.uint8, device="cuda"))
    acts = np.zeros((4, 20, 3), np.int32)
    good = {k: env._alloc(k, (4,)) for k in env.OUTPUTS}
    for k, bad in (("obs", env._alloc("obs", (3,))), ("reward", good["reward"].double()),
                   ("nbr_feat", good["nbr_feat"].transpose(1, 2))):
        with pytest.raises(ValueError):
            env.rollout(acts, out={**good, k: bad})
    env.rollout(acts, out=good)                                   # the right buffers still work
    env.close()
