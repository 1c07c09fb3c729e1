"""Float64 restatement of SPEC.md §13 (episode statistics), the reference of tests/test_episode_stats.py.

Explicit loops: slots t ascending (vectorised over rows), agents j ascending for the team values.  The
per-episode values are formed by the same fp64 operations in the same order as the kernel, so they must
match it exactly; the totals are summed with math.fsum (correctly rounded) and match within a relative
tolerance, because the kernel adds the episodes in its own fixed tree order."""
import math

import numpy as np

FIELDS = 16


class Reference:
    """Carry, last_* and team last_* of n_envs x N rows across calls; `call` returns the call's totals and
    `episodes`.  last_* start as NaN / 0, like EpisodeTracker's tensors, and stay untouched until a row
    (an env) completes an episode."""

    def __init__(self, n_envs, N, agent_cost_limit=0.0, team_cost_limit=0.0):
        rows = n_envs * N
        self.n_envs, self.N = n_envs, N
        self.agent_limit, self.team_limit = float(agent_cost_limit), float(team_cost_limit)
        self.carry_return = np.zeros(rows)
        self.carry_cost = np.zeros(rows)
        self.carry_length = np.zeros(rows, np.int64)
        self.last_return = np.full(rows, np.nan)
        self.last_cost = np.full(rows, np.nan)
        self.last_length = np.zeros(rows, np.int64)
        self.team_last_return = np.full(n_envs, np.nan)
        self.team_last_cost = np.full(n_envs, np.nan)
        self.agent_lengths = [[] for _ in range(rows)] if rows <= 1 << 16 else None   # for hand-written cases

    def call(self, reward, cost, done):
        """reward, cost: [T, rows] (any real dtype; widened to fp64 exactly), done: [T, rows]."""
        reward = np.asarray(reward).reshape(len(reward), -1)
        cost = np.asarray(cost).reshape(len(cost), -1)
        done = np.asarray(done).reshape(len(done), -1) != 0
        T, N = reward.shape[0], self.N
        R, C, n = self.carry_return, self.carry_cost, self.carry_length
        ag = {"ret": [], "cost": [], "len": []}
        tm = {"ret": [], "cost": [], "len": []}
        episodes = np.zeros(self.n_envs, np.int64)
        for t in range(T):
            R = R + reward[t].astype(np.float64)
            C = C + cost[t].astype(np.float64)
            n = n + 1
            d0 = done[t, ::N]                           # an env's episode ends with its agent 0's done
            if d0.any():
                Rm, Cm = R.reshape(-1, N), C.reshape(-1, N)
                tr, tc = np.zeros(self.n_envs), np.zeros(self.n_envs)
                for j in range(N):
                    tr = tr + Rm[:, j]
                    tc = tc + Cm[:, j]
                tr = tr / N
                e = np.nonzero(d0)[0]
                tm["ret"].append(tr[e]); tm["cost"].append(tc[e]); tm["len"].append(n[::N][e])
                self.team_last_return[e] = tr[e]
                self.team_last_cost[e] = tc[e]
                episodes[e] += 1
            d = done[t]
            if d.any():
                r = np.nonzero(d)[0]
                ag["ret"].append(R[r]); ag["cost"].append(C[r]); ag["len"].append(n[r])
                self.last_return[r], self.last_cost[r], self.last_length[r] = R[r], C[r], n[r]
                if self.agent_lengths is not None:
                    for i in r:
                        self.agent_lengths[i].append(int(n[i]))
                R, C, n = np.where(d, 0.0, R), np.where(d, 0.0, C), np.where(d, 0, n)
        self.carry_return, self.carry_cost, self.carry_length = R, C, n
        totals = np.concatenate([_totals(ag, self.agent_limit), _totals(tm, self.team_limit)])
        return totals, episodes


def _totals(eps, limit):
    cat = {k: (np.concatenate(v) if v else np.zeros(0)) for k, v in eps.items()}
    ret, cost, ln = cat["ret"], cat["cost"], cat["len"].astype(np.int64)
    return np.array([len(ret), math.fsum(ret), math.fsum(ret * ret), math.fsum(cost), math.fsum(cost * cost),
                     int(ln.sum()), int((cost == 0).sum()), int((cost > limit).sum())], np.float64)


COUNT_FIELDS = (0, 5, 6, 7, 8, 13, 14, 15)     # counts and length sums: exact
SUM_FIELDS = (1, 2, 3, 4, 9, 10, 11, 12)


def assert_totals(got, want, rtol=1e-12, ctx=""):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    for f in COUNT_FIELDS:
        assert got[f] == want[f], f"{ctx} totals[{f}]: {got[f]} != {want[f]}"
    for f in SUM_FIELDS:
        assert abs(got[f] - want[f]) <= rtol * abs(want[f]), f"{ctx} totals[{f}]: {got[f]!r} vs {want[f]!r}"
