"""UNVERIFIED constant sets used by this repo's own tests and bench.

None of these values comes from GS-MARL: its `config.py`, `core.py` and scenario files
are withheld (reference readme.md:1).  They are the *lineage hypotheses* recorded in
SURVEY.md Appendix A (upstream-MPE-style `dt`, `damping`, `contact_force`,
`contact_margin`), chosen only so that every branch of the kernels — contact force,
speed clamp, sensing-radius cut, goal bonus, obstacle cost — is exercised by random
rollouts.  The library itself has no defaults; these live outside it on purpose and must
be replaced by the real constants once the reference sources are mounted.
"""
from __future__ import annotations

import math

UNVERIFIED_WORLD = dict(
    dt=0.1,
    damping=0.25,
    contact_force=1e2,
    contact_margin=1e-3,
)

UNVERIFIED_DISCRETE_U = (   # index -> control; 0 = no-op
    (0.0, 0.0), (1.0, 0.0), (-1.0, 0.0), (0.0, 1.0), (0.0, -1.0),
)

UNVERIFIED_AGENT = dict(size=0.10, mass=1.0, accel=5.0, max_speed=1.3)
UNVERIFIED_GOAL_SIZE = 0.05
UNVERIFIED_OBSTACLE_SIZE = 0.16     # demo GIF pixel ratio obstacle:agent ~ 1.65 (SURVEY App. C)
UNVERIFIED_MARKER_SIZE = 0.16

UNVERIFIED_REWARD = dict(w_dist=1.0, w_goal=1.0, goal_tol=0.1)


def unverified_sensing_radius(n_agents: int) -> float:
    return 1.0


def unverified_spawn_extent(n_agents: int) -> float:
    """World half-extent grows with sqrt(N/3) (demo GIFs zoom out with N; SURVEY App. C)."""
    return math.sqrt(max(n_agents, 3) / 3.0)

# PPO-Lagrangian hyper-parameters typical of the MAPPO / MAPPO-L lineage (the reference's learner and
# its config are withheld); `learner.LagrangianPPO` takes every one as a required keyword.
UNVERIFIED_PPO_LAG = dict(
    clip=0.2,
    value_clip=0.2,
    value_coef=1.0,
    entropy_coef=0.01,
    lr=5e-4,
    betas=(0.9, 0.999),
    eps=1e-5,
    max_grad_norm=10.0,
    ppo_epoch=5,
    num_mini_batch=1,
    lagrangian_lr=1e-2,
    cost_limit=0.0,
)
