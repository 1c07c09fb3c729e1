"""Float64 numpy restatement of SPEC.md §1-8 for every scenario: Philox4x32-10 and the spawn draw (§8), the
contact force and integration (§2-4), the assignment (§5, scipy), the graph (§6), reward, cost and done (§7).

It shares no code with the kernels or with the C oracle; tests/test_nav_autoreset_reference.py and
tests/test_team_autoreset_reference.py pin it to the oracle on the CPU and compare the kernels with it on the GPU.
Pair arrays ([n, N, E]) are built for at most `chunk_elems` (env, agent, entity) triples at a time, so that
navigation-96 x 4096 envs fits in host memory.
"""
import numpy as np
from scipy.optimize import linear_sum_assignment

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
    precision of the state the kernel holds: a re-drawn position is rounded to it, as the kernel stores it.
    Row b is global env `genv[b]` (default env_offset + b), so a reference may follow a sample of a batch."""
    scenarios = ("navigation",)

    def __init__(self, cfg, agent_state, landmark_pos, t, episode, seed, env_offset=0, genv=None,
                 chunk_elems=1 << 22):
        assert cfg.scenario in self.scenarios, cfg.scenario
        self.cfg, self.seed = cfg, int(seed)
        self.real = np.float32 if cfg.dtype == "f32" else np.float64
        self.ag = np.array(agent_state, np.float64)            # [B, N, 4]: x, y, vx, vy
        self.lm = np.array(landmark_pos, np.float64)            # [B, L, 2]
        self.t = np.array(t, np.int64)
        self.ep = np.array(episode, np.int64)
        self.genv = (np.arange(self.B, dtype=np.int64) + int(env_offset) if genv is None
                     else np.asarray(genv, np.int64))
        c = cfg
        self.size = np.asarray(c.size, np.float64)
        self.collide = np.asarray(c.collide, bool)
        self.type = np.asarray(c.type, np.int64)
        self.u = np.asarray(c.discrete_u, np.float64)
        self.chunk = max(1, int(chunk_elems) // (c.n_agents * c.n_entities))

    @property
    def B(self):
        return self.ag.shape[0]

    def _chunks(self):
        for lo in range(0, self.B, self.chunk):
            yield slice(lo, min(lo + self.chunk, self.B))

    def redraw(self, mask):
        """SPEC §8 for the envs in `mask` [B]: spawn draw of (env, ep), v = 0, t = 0, then ep += 1."""
        idx = np.flatnonzero(mask)
        if idx.size == 0:
            return
        N = self.cfg.n_agents
        p = spawn_draw(self.cfg, self.genv[idx], self.ep[idx], self.seed).astype(self.real).astype(np.float64)
        self.ag[idx, :, :2] = p[:, :N]
        self.ag[idx, :, 2:] = 0.0
        self.lm[idx] = p[:, N:]
        self.t[idx] = 0
        self.ep[idx] += 1

    def _geometry(self, sl):
        N = self.cfg.n_agents
        pos = np.concatenate([self.ag[sl, :, :2], self.lm[sl]], 1)                # [b, E, 2]
        d = pos[:, None, :, :] - pos[:, :N, None, :]                              # [b, N, E, 2]: p_e - p_i
        dist = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1])
        return pos, d, dist

    def advance(self, actions):
        """SPEC §2-4 and t += 1, no outputs."""
        c, N = self.cfg, self.cfg.n_agents
        a = np.asarray(actions)
        if c.action_mode == "discrete":
            ok = (a >= 0) & (a < len(self.u))
            ctrl = np.where(ok[..., None], self.u[np.clip(a, 0, len(self.u) - 1)], 0.0)
        else:
            ctrl = a.astype(np.float64)
        F = np.asarray(c.accel, np.float64)[None, :, None] * ctrl                    # [B, N, 2]
        pair = self.collide[:N, None] & self.collide[None, :]
        pair[np.arange(N), np.arange(N)] = False
        dmin = (self.size[:N, None] + self.size[None, :])[None]
        for sl in self._chunks():                                                   # forces on the pre-step state
            _, d, dist = self._geometry(sl)
            x = -(dist - dmin) / c.contact_margin
            pen = np.logaddexp(0.0, x) * c.contact_margin
            with np.errstate(invalid="ignore", divide="ignore"):
                f = np.where(pair[None, ..., None], c.contact_force * (-d) / dist[..., None] * pen[..., None], 0.0)
            F[sl] = F[sl] + f.sum(2)
        v = self.ag[..., 2:] * (1.0 - c.damping) + (F / np.asarray(c.mass, np.float64)[None, :, None]) * c.dt
        ms = np.asarray(c.max_speed, np.float64)[None, :]
        sp = np.sqrt(v[..., 0] * v[..., 0] + v[..., 1] * v[..., 1])
        clamp = (ms > 0) & (sp > ms)
        v = np.where(clamp[..., None], v / np.where(clamp, sp, 1.0)[..., None] * ms[..., None], v)
        self.ag[..., 2:] = v
        self.ag[..., :2] = self.ag[..., :2] + v * c.dt
        self.t += 1

    def step(self, actions, assign=None):
        """SPEC §2-4, then the outputs of the new state (§5-7)."""
        self.advance(actions)
        return self.observe(assign)

    def targets(self, assign=None):
        """SPEC §5: (assign [B, N], target positions [B, N, 2]).  Navigation: goal i = landmark i."""
        assert assign is None, "navigation has no assignment to impose"
        N = self.cfg.n_agents
        return np.broadcast_to(np.arange(N, dtype=np.int32)[None], (self.B, N)), self.lm[:, :N]

    def observe(self, assign=None):
        c, N, K, E = self.cfg, self.cfg.n_agents, self.cfg.max_nbrs, self.cfg.n_entities
        B, W = self.B, (E + 31) // 32
        ar = np.arange(N)
        out = {"nbr_idx": np.full((B, N, K), -1, np.int32), "nbr_feat": np.zeros((B, N, K, 6)),
               "nbr_cnt": np.zeros((B, N), np.int32), "adj": np.zeros((B, N, W), np.uint32),
               "cost": np.zeros((B, N))}
        counted = (self.type == 0) | ((self.type == 2) & bool(c.cost_obstacles))
        counted = np.broadcast_to(counted[None, :], (N, E)).copy()
        counted[ar, ar] = False
        dmin = (self.size[:N, None] + self.size[None, :])[None]
        typ = self.type.astype(np.float64)
        bits = np.uint64(1) << np.arange(32, dtype=np.uint64)
        for sl in self._chunks():
            pos, d, dist = self._geometry(sl)
            b = dist.shape[0]
            vel = np.concatenate([self.ag[sl, :, 2:], np.zeros_like(self.lm[sl])], 1)   # [b, E, 2]
            nb = dist < c.sensing_radius
            if c.own_goal_always and c.scenario == "navigation":
                nb[:, ar, N + ar] = True
            nb[:, ar, ar] = False
            rank = np.cumsum(nb, 2) - 1
            keep = nb & (rank < K)
            bi, ii, ee = np.nonzero(keep)
            kk = rank[bi, ii, ee]
            out["nbr_idx"][sl][bi, ii, kk] = ee
            dv = vel[:, None, :, :] - vel[:, :N, None, :]
            out["nbr_feat"][sl][bi, ii, kk] = np.stack(
                [d[bi, ii, ee, 0], d[bi, ii, ee, 1], dv[bi, ii, ee, 0], dv[bi, ii, ee, 1], dist[bi, ii, ee], typ[ee]], -1)
            out["nbr_cnt"][sl] = np.minimum(nb.sum(2), K)
            nbw = np.zeros((b, N, W * 32), bool)
            nbw[..., :E] = nb
            out["adj"][sl] = (nbw.reshape(b, N, W, 32).astype(np.uint64) * bits).sum(-1).astype(np.uint32)
            out["cost"][sl] = ((dist < dmin) & counted[None]).sum(2)
        asg, tgt = self.targets(assign)
        g = tgt - self.ag[..., :2]
        gd = np.sqrt(g[..., 0] * g[..., 0] + g[..., 1] * g[..., 1])
        out["obs"] = np.concatenate([self.ag[..., 2:], self.ag[..., :2], g], -1)
        r = (0.0 - c.w_dist * gd) + np.where(gd < c.goal_tol, c.w_goal, 0.0)
        if c.share_reward:
            s = r[:, 0].copy()
            for i in range(1, N):
                s = s + r[:, i]
            r = np.repeat((s / N)[:, None], N, 1)
        out["reward"] = r
        out["done"] = np.repeat((self.t >= c.episode_length)[:, None], N, 1)
        out["assign"] = np.array(asg, np.int32)
        return out


class RefTeam(RefNav):
    """Polygon / line (SPEC §1, §5): slots from the marker(s) and cfg.slot_table, the cost matrix, and the
    assignment of scipy.optimize.linear_sum_assignment (the solver SPEC §5 pins).  Everything else is RefNav's."""
    scenarios = ("polygon", "line")

    def slots(self):
        """SPEC §1: slot positions [B, N, 2] of the current markers, component-wise as written there."""
        c, m = self.cfg, self.lm
        tab = np.asarray(c.slot_table, np.float64)
        if c.scenario == "polygon":
            return m[:, :1, :] + c.polygon_radius * tab[None]
        f = tab[:, 0][None, :, None]
        return m[:, :1, :] + f * (m[:, 1:2, :] - m[:, :1, :])

    def cost_matrix(self, agent_pos):
        """SPEC §5: C [B, N, N], C[b, i, k] = |s_k - p_i| of agent positions [B, N, 2]."""
        s = self.slots()
        dx = s[:, None, :, 0] - np.asarray(agent_pos, np.float64)[:, :, None, 0]
        dy = s[:, None, :, 1] - np.asarray(agent_pos, np.float64)[:, :, None, 1]
        return np.sqrt(dx * dx + dy * dy)

    @staticmethod
    def solve(C):
        """col4row [B, N] of each problem, scipy's solver (rows come back in order for a square matrix)."""
        out = np.empty(C.shape[:2], np.int32)
        for b in range(C.shape[0]):
            out[b] = linear_sum_assignment(C[b])[1]
        return out

    def targets(self, assign=None):
        if assign is None:
            assign = self.solve(self.cost_matrix(self.ag[..., :2]))
        assign = np.asarray(assign, np.int32)
        return assign, np.take_along_axis(self.slots(), assign[..., None].astype(np.int64), 1)


def make_ref(cfg, *args, **kw):
    return (RefNav if cfg.scenario == "navigation" else RefTeam)(cfg, *args, **kw)


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


# fp32 production bar (SPEC §9): 1e-4 relative; atol 2e-5 covers values that cross zero (positions, deltas)
# with ~2 ulp of the unit-scale state
F32_TOL = dict(rtol=1e-4, atol=2e-5)
INT_KEYS = ("nbr_idx", "nbr_cnt", "adj", "done", "assign", "cost")
REAL_KEYS = ("obs", "nbr_feat", "reward")


def assert_step(got, want, ok, tol, ctx, ok_reward=None):
    """Integer outputs (and the cost count) exact on the rows `ok` [B, N], reals within `tol` there; the reward
    on `ok_reward` (default `ok`)."""
    for k in INT_KEYS:
        g, w = np.asarray(got[k])[ok], np.asarray(want[k])[ok].astype(np.asarray(got[k]).dtype)
        bad = np.argwhere(g != w)
        assert bad.size == 0, f"{ctx} {k}: {len(bad)} rows differ"
    for k in REAL_KEYS:
        m = ok if k != "reward" or ok_reward is None else ok_reward
        np.testing.assert_allclose(got[k][m], want[k][m], **tol, err_msg=f"{ctx} {k}")


def check_fused_f32(ref, got, acts, ctx, assign_of=None):
    """An fp32 fused auto-reset rollout `got` ([T, B, ...] numpy outputs of the envs `ref` follows), slot by slot:
    fp32 and fp64 trajectories part at the stiff contacts, so each slot is ONE reference step from the kernel's own
    state of the slot before (the agent state is exactly obs[..., :4] of that slot; the landmarks change only in a
    re-draw, which the reference makes itself: fp64 draw rounded to fp32, as the kernel stores it).  Integer
    outputs and the cost must match except on rows with a pair distance within 1e-4 of the sensing radius or the
    contact distance (SPEC §9) or a goal distance within 1e-4 of goal_tol (the reward's step; with share_reward
    that excludes the env's reward); reals within F32_TOL.  `assign_of(s, ref)`: the assignment to score slot s
    with (team scenarios), None: the reference's own.  Returns (rows checked, rows, [T] envs re-drawn after
    each slot)."""
    from tests._util import near_threshold_rows
    cfg = ref.cfg
    checked = rows = 0
    ends = []
    for s in range(len(acts)):
        ref.advance(acts[s])
        want = ref.observe(None if assign_of is None else assign_of(s, ref))
        gd = np.hypot(want["obs"][..., 4], want["obs"][..., 5])
        goal_ok = np.abs(gd - cfg.goal_tol) > 1e-4
        ok = ~near_threshold_rows(cfg, ref.ag, ref.lm, 1e-4) & goal_ok
        ok_rew = ok & goal_ok.all(1, keepdims=True) if cfg.share_reward else None
        assert_step({k: got[k][s] for k in got}, want, ok, F32_TOL, f"{ctx} t={s}", ok_rew)
        checked += int(ok.sum())
        rows += ok.size
        fin = ref.t >= cfg.episode_length
        ends.append(int(fin.sum()))
        ref.redraw(fin)
        keep = ~fin                      # continue from the kernel's own state where the env did not restart
        ref.ag[keep, :, 2:] = got["obs"][s][keep][..., 0:2]
        ref.ag[keep, :, :2] = got["obs"][s][keep][..., 2:4]
    return checked, rows, np.asarray(ends)


def env_sample(B, n, t0, last_cta, seed=0):
    """Sorted env indices the reference follows: all of them if n == 0 or n >= B, else n of them that always
    include the last CTA's envs (`last_cta` of them) and the first two envs of every step-counter value in t0
    (so envs finish in every slot), filled up with a seeded uniform draw."""
    if n == 0 or n >= B:
        return np.arange(B)
    t0 = np.asarray(t0)
    must = [np.arange(max(0, B - last_cta), B)] + [np.flatnonzero(t0 == v)[:2] for v in np.unique(t0)]
    must = np.unique(np.concatenate(must))
    rest = np.setdiff1d(np.arange(B), must)
    fill = np.random.default_rng(seed).choice(rest, max(0, n - must.size), replace=False)
    return np.sort(np.concatenate([must, fill]))


def squeezed_start(cfg, B, seed, t0, scale=0.45):
    """A SPEC §8 draw pulled towards the origin (contacts from the first step on), at step counters t0."""
    p = spawn_draw(cfg, np.arange(B), np.zeros(B, np.int64), seed) * scale
    p = p.astype(np.float32 if cfg.dtype == "f32" else np.float64).astype(np.float64)
    N = cfg.n_agents
    ag = np.concatenate([p[:, :N], np.zeros_like(p[:, :N])], -1)
    return ag, p[:, N:], np.asarray(t0, np.int64)


def tie_heavy_start(cfg, ag, lm, envs_halfway, envs_reversed):
    """Agents placed where only scipy's scan order decides the assignment (test_team_kernel_group_lsa_f64):
    `envs_halfway` halfway between consecutive slots (two equally good shifts), `envs_reversed` exactly on the
    slots in reversed order; at rest.  Modifies `ag` in place."""
    N = cfg.n_agents
    tab = np.asarray(cfg.slot_table, np.float64)
    def slots_of(m):
        if cfg.scenario == "polygon":
            return m[:, :1, :] + cfg.polygon_radius * tab[None]
        return m[:, :1, :] + tab[:, 0][None, :, None] * (m[:, 1:2, :] - m[:, :1, :])
    h, r = np.asarray(envs_halfway), np.asarray(envs_reversed)
    if cfg.scenario == "polygon":
        ang = (2 * np.arange(N) + 1) * np.pi / N
        ag[h, :, :2] = lm[h, :1, :] + cfg.polygon_radius * np.stack([np.cos(ang), np.sin(ang)], -1)[None]
    else:
        sl = slots_of(lm[h])
        mid = 0.5 * (sl + np.roll(sl, -1, axis=1))
        mid[:, -1] = sl[:, -1] + 0.5 * (sl[:, -1] - sl[:, -2])
        ag[h, :, :2] = mid
    ag[r, :, :2] = slots_of(lm[r])[:, ::-1, :]
    ag[h, :, 2:] = 0
    ag[r, :, 2:] = 0
    if cfg.dtype == "f32":
        ag[...] = ag.astype(np.float32).astype(np.float64)
    return ag
