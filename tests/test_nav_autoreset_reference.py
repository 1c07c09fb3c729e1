"""The wide navigation kernel (env_wide_kernel: navigation with 3, 4 or 5 agents) and its in-kernel auto-reset,
against a float64 numpy restatement of SPEC.md §2-4 and §6-8 written in this file.

The reference shares no code with the kernels or with the C oracle: Philox4x32-10, the spawn draw, the contact
force, the integration, the graph, reward, cost, done and the auto-reset rule are all restated here, vectorised
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

from tests._util import make_cfg, near_threshold_rows, random_actions

# fp64 kernels round every SPEC operation once (-fmad=false); they differ from this reference only in libm's
# last ulp and in the order in which pair forces are summed, which the stiff contacts amplify over 25 steps
# to well below 1e-9 (SPEC §9).
F64_TOL = dict(rtol=1e-9, atol=1e-9)
# fp32 production bar (SPEC §9): 1e-4 relative; atol 2e-5 covers values that cross zero (positions, deltas)
# with ~2 ulp of the unit-scale state
F32_TOL = dict(rtol=1e-4, atol=2e-5)
BENCH_ENVS = 16384                     # bench.py ENVS_PER_GPU: navigation-3, one launch of T = 25


# ---- float64 reference ------------------------------------------------------------------------
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on uint64 arrays holding 32-bit words -> (r0, r1, r2, r3)."""
    c0, c1, c2, c3, k0, k1 = (np.asarray(x, np.uint64) & _M32 for x in (c0, c1, c2, c3, k0, k1))
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
        k0 = (k0 + np.uint64(0x9E3779B9)) & _M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & _M32
    return c0, c1, c2, c3


def spawn_draw(cfg, genv, ep, seed):
    """SPEC §8: positions [n, E, 2] (fp64) of every entity of global envs `genv` in episodes `ep`."""
    E = cfg.n_entities
    g = np.asarray(genv, np.uint64)[:, None]
    e = np.arange(E, dtype=np.uint64)[None, :]
    r0, r1, r2, r3 = philox4x32_10(g & _M32, g >> np.uint64(32), np.asarray(ep, np.int64)[:, None].astype(np.uint64),
                                   e, np.uint64(seed) & _M32, np.uint64(seed) >> np.uint64(32))
    u = lambda hi, lo: ((hi >> np.uint64(5)).astype(np.float64) * 67108864.0 + (lo >> np.uint64(6)).astype(np.float64)) / 2.0 ** 53
    ext = np.asarray(cfg.spawn_extent, np.float64)[np.asarray(cfg.type)][None, :]
    return np.stack([-ext + (2.0 * ext) * u(r0, r1), -ext + (2.0 * ext) * u(r2, r3)], -1)


class RefNav:
    """Batched navigation world in float64: state, one step, observation, the SPEC §8 re-draw.  `real` is the
    precision of the state the kernel holds: a re-drawn position is rounded to it, as the kernel stores it."""

    def __init__(self, cfg, agent_state, landmark_pos, t, episode, seed, env_offset=0):
        assert cfg.scenario == "navigation"
        self.cfg, self.seed, self.env_offset = cfg, int(seed), int(env_offset)
        self.real = np.float32 if cfg.dtype == "f32" else np.float64
        self.ag = np.array(agent_state, np.float64)            # [B, N, 4]: x, y, vx, vy
        self.lm = np.array(landmark_pos, np.float64)            # [B, L, 2]
        self.t = np.array(t, np.int64)
        self.ep = np.array(episode, np.int64)
        c = cfg
        self.size = np.asarray(c.size, np.float64)
        self.collide = np.asarray(c.collide, bool)
        self.type = np.asarray(c.type, np.int64)
        self.u = np.asarray(c.discrete_u, np.float64)

    @property
    def B(self):
        return self.ag.shape[0]

    def redraw(self, mask):
        """SPEC §8 for the envs in `mask` [B]: spawn draw of (env, ep), v = 0, t = 0, then ep += 1."""
        idx = np.flatnonzero(mask)
        if idx.size == 0:
            return
        N = self.cfg.n_agents
        p = spawn_draw(self.cfg, self.env_offset + idx, self.ep[idx], self.seed).astype(self.real).astype(np.float64)
        self.ag[idx, :, :2] = p[:, :N]
        self.ag[idx, :, 2:] = 0.0
        self.lm[idx] = p[:, N:]
        self.t[idx] = 0
        self.ep[idx] += 1

    def _geometry(self):
        N = self.cfg.n_agents
        pos = np.concatenate([self.ag[..., :2], self.lm], 1)                      # [B, E, 2]
        d = pos[:, None, :, :] - pos[:, :N, None, :]                              # [B, N, E, 2]: p_e - p_i
        dist = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1])
        return pos, d, dist

    def step(self, actions):
        """SPEC §2-4, then the outputs of the new state (§6-7)."""
        c, N = self.cfg, self.cfg.n_agents
        a = np.asarray(actions)
        if c.action_mode == "discrete":
            ok = (a >= 0) & (a < len(self.u))
            ctrl = np.where(ok[..., None], self.u[np.clip(a, 0, len(self.u) - 1)], 0.0)
        else:
            ctrl = a.astype(np.float64)
        F = np.asarray(c.accel, np.float64)[None, :, None] * ctrl                    # [B, N, 2]
        _, d, dist = self._geometry()
        pair = self.collide[:N, None] & self.collide[None, :]
        pair[np.arange(N), np.arange(N)] = False
        x = -(dist - (self.size[:N, None] + self.size[None, :])[None]) / c.contact_margin
        pen = np.logaddexp(0.0, x) * c.contact_margin
        with np.errstate(invalid="ignore", divide="ignore"):
            f = np.where(pair[None, ..., None], c.contact_force * (-d) / dist[..., None] * pen[..., None], 0.0)
        F = F + f.sum(2)
        v = self.ag[..., 2:] * (1.0 - c.damping) + (F / np.asarray(c.mass, np.float64)[None, :, None]) * c.dt
        ms = np.asarray(c.max_speed, np.float64)[None, :]
        sp = np.sqrt(v[..., 0] * v[..., 0] + v[..., 1] * v[..., 1])
        clamp = (ms > 0) & (sp > ms)
        v = np.where(clamp[..., None], v / np.where(clamp, sp, 1.0)[..., None] * ms[..., None], v)
        self.ag[..., 2:] = v
        self.ag[..., :2] = self.ag[..., :2] + v * c.dt
        self.t += 1
        return self.observe()

    def observe(self):
        c, N, K, E = self.cfg, self.cfg.n_agents, self.cfg.max_nbrs, self.cfg.n_entities
        B = self.B
        pos, d, dist = self._geometry()
        vel = np.concatenate([self.ag[..., 2:], np.zeros_like(self.lm)], 1)       # [B, E, 2]
        ar = np.arange(N)
        nb = dist < c.sensing_radius
        if c.own_goal_always:
            nb[:, ar, N + ar] = True
        nb[:, ar, ar] = False
        rank = np.cumsum(nb, 2) - 1
        keep = nb & (rank < K)
        bi, ii, ee = np.nonzero(keep)
        kk = rank[bi, ii, ee]
        out = {"nbr_idx": np.full((B, N, K), -1, np.int32), "nbr_feat": np.zeros((B, N, K, 6))}
        out["nbr_idx"][bi, ii, kk] = ee
        dv = vel[:, None, :, :] - vel[:, :N, None, :]
        out["nbr_feat"][bi, ii, kk] = np.stack([d[..., 0], d[..., 1], dv[..., 0], dv[..., 1], dist,
                                                np.broadcast_to(self.type[None, None, :].astype(np.float64), dist.shape)],
                                               -1)[bi, ii, ee]
        out["nbr_cnt"] = np.minimum(nb.sum(2), K).astype(np.int32)
        out["adj"] = (nb.astype(np.uint64) << np.arange(E, dtype=np.uint64)).sum(2).astype(np.uint32)[..., None]   # E <= 32: one word
        g = d[:, ar, N + ar]                                                        # goal i = landmark i
        gd = dist[:, ar, N + ar]
        out["obs"] = np.concatenate([self.ag[..., 2:], self.ag[..., :2], g], -1)
        r = (0.0 - c.w_dist * gd) + np.where(gd < c.goal_tol, c.w_goal, 0.0)
        if c.share_reward:
            s = r[:, 0].copy()
            for i in range(1, N):
                s = s + r[:, i]
            r = np.repeat((s / N)[:, None], N, 1)
        out["reward"] = r
        counted = (self.type == 0) | ((self.type == 2) & bool(c.cost_obstacles))
        counted = np.broadcast_to(counted[None, :], (N, E)).copy()
        counted[ar, ar] = False
        hit = dist < (self.size[:N, None] + self.size[None, :])[None]
        out["cost"] = (hit & counted[None]).sum(2).astype(np.float64)
        out["done"] = np.repeat((self.t >= c.episode_length)[:, None], N, 1)
        out["assign"] = np.broadcast_to(ar[None, :], (B, N)).astype(np.int32)
        return out


def ref_fused_rollout(ref, acts, auto_reset=True):
    """The fused-rollout convention: outputs of every slot (terminal rows stay), then the re-draw of the envs that
    finished.  Returns (per-slot outputs, per-slot bool [B] of the envs re-drawn after that slot)."""
    outs, redrawn = [], []
    for s in range(len(acts)):
        outs.append(ref.step(acts[s]))
        fin = ref.t >= ref.cfg.episode_length if auto_reset else np.zeros(ref.B, bool)
        ref.redraw(fin)
        redrawn.append(fin)
    return outs, redrawn


def squeezed_start(cfg, B, seed, t0, scale=0.45):
    """A SPEC §8 draw pulled towards the origin (contacts from the first step on), at step counters t0."""
    p = spawn_draw(cfg, np.arange(B), np.zeros(B, np.int64), seed) * scale
    p = p.astype(np.float32 if cfg.dtype == "f32" else np.float64).astype(np.float64)
    N = cfg.n_agents
    ag = np.concatenate([p[:, :N], np.zeros_like(p[:, :N])], -1)
    return ag, p[:, N:], np.asarray(t0, np.int64)


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
                                  (3, {"max_nbrs": 3, "own_goal_always": False, "cost_obstacles": False})])
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


def _np(bufs):
    out = {}
    for k, v in bufs.items():
        a = v.detach().cpu().numpy()
        out[k] = a.view(np.uint32) if k == "adj" else a
    return out


INT_KEYS = ("nbr_idx", "nbr_cnt", "adj", "done", "assign", "cost")
REAL_KEYS = ("obs", "nbr_feat", "reward")


def _assert_step(got, want, ok, tol, ctx):
    """Integer outputs (and the cost count) exact on the rows `ok` [B, N], reals within `tol` there."""
    for k in INT_KEYS:
        g, w = np.asarray(got[k])[ok], np.asarray(want[k])[ok].astype(np.asarray(got[k]).dtype)
        bad = np.argwhere(g != w)
        assert bad.size == 0, f"{ctx} {k}: {len(bad)} rows differ"
    for k in REAL_KEYS:
        np.testing.assert_allclose(got[k][ok], want[k][ok], **tol, err_msg=f"{ctx} {k}")


def _staggered_env(cfg, B, seed, t0):
    env = _env(cfg, B, seed=seed)
    ag, lm, t = squeezed_start(cfg, B, seed + 1, t0)
    env.reset()
    env.set_state(ag, lm, t)
    return env, RefNav(cfg, ag, lm, t, env.get_episode().cpu().numpy(), seed)


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
        _assert_step({k: got[k][s] for k in got}, want[s], ok, F64_TOL, f"N={N} B={B} t={s}")
    ag, lm, t = (x.cpu().numpy() for x in env.get_state())
    np.testing.assert_allclose(ag, ref.ag, **F64_TOL)
    assert (lm == ref.lm).all() and (t == ref.t).all()
    assert (env.get_episode().cpu().numpy() == ref.ep).all()
    assert np.stack(redrawn).sum() >= B * (T // 6), "too few episode ends"
    env.close()


@gpu
@pytest.mark.parametrize("N", [3, 4, 5])
def test_only_finished_envs_are_redrawn_f64(N):
    """Half of the envs finish on step 2 of a 5-step launch, the other half never: the finished ones restart
    from the SPEC §8 draw of their episode (bit for bit: the draw is integer + exact fp64 arithmetic), the others
    are untouched — every output and the final state equal the same launch without auto-reset."""
    cfg = make_cfg("navigation", N, "f64", episode_length=10)
    B, T, seed = 203, 5, 21
    fin_env = np.arange(B) % 2 == 0
    t0 = np.where(fin_env, 8, 0)                                     # 8 + 2 = 10: done on step index 1
    env, ref = _staggered_env(cfg, B, seed, t0)
    ag0, lm0, tt0 = (x.clone() for x in env.get_state())
    ep0 = env.get_episode().clone()
    acts = random_actions(cfg, np.random.default_rng(N), (T, B))
    ar = _np(env.rollout(acts, auto_reset=True))
    ar_state = [x.cpu().numpy() for x in env.get_state()] + [env.get_episode().cpu().numpy()]
    env.set_state(ag0, lm0, tt0)
    env.set_episode(ep0)
    plain = _np(env.rollout(acts, auto_reset=False))
    plain_state = [x.cpu().numpy() for x in env.get_state()] + [env.get_episode().cpu().numpy()]
    env.close()

    want, redrawn = ref_fused_rollout(ref, acts)
    assert (redrawn[1] == fin_env).all() and not any(r.any() for i, r in enumerate(redrawn) if i != 1)
    for s in range(T):
        _assert_step({k: ar[k][s] for k in ar}, want[s], np.ones((B, N), bool), F64_TOL, f"N={N} t={s}")
    # the re-draw itself: finished envs end the launch at t = 3 from positions drawn in episode ep0 + 0
    draw = spawn_draw(cfg, np.arange(B), ep0.cpu().numpy(), seed)
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
        _assert_step(got, want, np.ones((B, N), bool), F64_TOL, f"N={N} step {s}")
        assert (got["done"].all(1) == fin).all()
    env.close()


@gpu
@pytest.mark.parametrize("T", [25, 7])
def test_auto_reset_instance_equals_plain_instance_when_nothing_finishes(T):
    """The benchmark's instance (<float, 3, 6, auto-reset, K = 8>) against the plain one at the bench size: with
    no episode ending inside the launch, the two must give the same bits in every output and the final state."""
    cfg = make_cfg("navigation", 3, "f32", episode_length=1000)
    B = BENCH_ENVS
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
    env.close()
    assert not bool(res[0][sorted(env.OUTPUTS).index("done")].any())
    for a, b in zip(*res):
        assert torch.equal(a, b)


@gpu
@pytest.mark.parametrize("N,B", [(3, BENCH_ENVS), (3, 1), (4, 1001), (5, 999)])
def test_fused_auto_reset_rollout_f32_vs_reference(N, B):
    """fp32 production instances over one 25-step fused launch with staggered episode ends (the benchmark's
    shape for N = 3).  fp32 and fp64 trajectories part at the stiff contacts, so each slot is checked against ONE
    reference step from the kernel's own state of the slot before: the agent state is exactly obs[..., :4] of
    that slot, the landmarks only change in a re-draw, which the reference makes itself (fp64 draw rounded to
    fp32, as the kernel stores it).  Integer outputs must match except on rows with a predicate within 1e-4 of
    its threshold (SPEC §9) or a goal distance within 1e-4 of goal_tol (the reward's step); after a re-draw the positions are the draw's exact fp32 values."""
    cfg = make_cfg("navigation", N, "f32", episode_length=25)
    T, seed = 25, 31
    t0 = np.arange(B) % 25
    env, ref = _staggered_env(cfg, B, seed, t0)
    acts = random_actions(cfg, np.random.default_rng(N), (T, B))
    got = _np(env.rollout(acts, auto_reset=True))
    final = [x.cpu().numpy() for x in env.get_state()] + [env.get_episode().cpu().numpy()]
    env.close()
    checked = ends = 0
    for s in range(T):
        want = ref.step(acts[s])
        gd = np.hypot(want["obs"][..., 4], want["obs"][..., 5])
        ok = ~near_threshold_rows(cfg, ref.ag, ref.lm, 1e-4) & (np.abs(gd - cfg.goal_tol) > 1e-4)
        _assert_step({k: got[k][s] for k in got}, want, ok, F32_TOL, f"N={N} B={B} t={s}")
        checked += int(ok.sum())
        fin = ref.t >= cfg.episode_length
        ends += int(fin.sum())
        ref.redraw(fin)
        # continue from the kernel's own state (exact fp32 values) where the env did not restart
        keep = ~fin
        ref.ag[keep, :, 2:] = got["obs"][s][keep][..., 0:2]
        ref.ag[keep, :, :2] = got["obs"][s][keep][..., 2:4]
    assert checked > 0.5 * T * B * N and ends >= B * (T - 1) // 25
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
