"""Episode statistics (SPEC.md §13): `gsm_episode_stats` / `EpisodeTracker` against the float64 restatement
in tests/_episode_oracle.py — hand-written sequences, synthetic slots, real rollouts, determinism, the C
ABI's argument checks and guard bands around every output."""
import ctypes as C
import math
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from gs_marl_b200 import abi
from gs_marl_b200.episodes import EpisodeTracker, _check_update_inputs
from tests._episode_oracle import Reference, assert_totals
from tests._util import make_cfg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


# ---- the reference on hand-written sequences (CPU) ------------------------------------------------
def test_reference_episode_spanning_three_calls():
    ref = Reference(1, 1)
    tot, eps = ref.call([[1.0], [2.0]], [[0.0], [1.0]], [[0], [0]])
    assert tot[0] == 0 and tot[8] == 0 and eps[0] == 0
    assert (ref.carry_return[0], ref.carry_cost[0], ref.carry_length[0]) == (3.0, 1.0, 2)
    assert math.isnan(ref.last_return[0])
    ref.call([[3.0], [4.0], [5.0]], [[0.0]] * 3, [[0]] * 3)
    assert (ref.carry_return[0], ref.carry_length[0]) == (15.0, 5)
    tot, eps = ref.call([[6.0], [7.0]], [[0.0], [2.0]], [[0], [1]])
    assert (ref.last_return[0], ref.last_cost[0], ref.last_length[0]) == (28.0, 3.0, 7)
    assert (ref.carry_return[0], ref.carry_cost[0], ref.carry_length[0]) == (0.0, 0.0, 0)
    assert list(tot[:8]) == [1, 28.0, 784.0, 3.0, 9.0, 7, 0, 1]
    assert list(tot[8:]) == [1, 28.0, 784.0, 3.0, 9.0, 7, 0, 1] and eps[0] == 1


def test_reference_two_episodes_in_one_call_and_team_values():
    ref = Reference(1, 2, agent_cost_limit=1.0, team_cost_limit=1.0)
    r = [[1.0, 3.0], [1.0, 3.0], [2.0, 2.0], [2.0, 2.0], [2.0, 2.0], [5.0, 5.0]]
    c = [[0.0, 1.0], [0.0, 0.0], [0.0, 0.0], [0.0, 0.0], [0.0, 0.0], [0.0, 0.0]]
    d = [[0, 0], [1, 1], [0, 0], [0, 0], [1, 1], [0, 0]]
    tot, eps = ref.call(r, c, d)
    assert eps[0] == 2
    assert ref.agent_lengths == [[2, 3], [2, 3]]
    assert list(ref.last_return) == [6.0, 6.0] and list(ref.last_length) == [3, 3]
    assert list(ref.carry_return) == [5.0, 5.0] and list(ref.carry_length) == [1, 1]
    # team episodes: (2 + 6) / 2 = 4 with cost 1, then (6 + 6) / 2 = 6 with cost 0
    assert ref.team_last_return[0] == 6.0 and ref.team_last_cost[0] == 0.0
    assert list(tot[8:]) == [2, 10.0, 52.0, 1.0, 1.0, 5, 1, 0]
    # agent episodes: returns 2, 6, 6, 6; costs 0, 1, 0, 0; 3 safe, none over the limit 1 (1 is not > 1)
    assert list(tot[:8]) == [4, 20.0, 112.0, 1.0, 1.0, 10, 3, 0]


def test_reference_length_one_episodes():
    ref = Reference(2, 1)
    T = 5
    tot, eps = ref.call(np.arange(2 * T, dtype=np.float64).reshape(T, 2), np.zeros((T, 2)), np.ones((T, 2)))
    assert ref.agent_lengths == [[1] * T, [1] * T]
    assert list(eps) == [T, T] and tot[0] == 2 * T and tot[5] == 2 * T and tot[6] == 2 * T
    assert list(ref.last_return) == [8.0, 9.0] and list(ref.carry_length) == [0, 0]


def test_reference_cost_at_the_limit_is_not_over_it():
    ref = Reference(3, 1, agent_cost_limit=2.0, team_cost_limit=2.0)
    tot, _ = ref.call(np.zeros((2, 3)), [[1.0, 1.0, 2.0], [1.0, 1.5, 0.0]], np.ones((2, 3), np.uint8) * [[0], [1]])
    # episode costs 2.0 (at the limit), 2.5 (over), 2.0 (at the limit)
    assert list(ref.last_cost) == [2.0, 2.5, 2.0]
    assert tot[7] == 1 and tot[15] == 1 and tot[6] == 0


# ---- argument checks and the ABI (CPU) --------------------------------------------------------------
def test_update_inputs_are_checked_before_any_launch():
    dev = torch.device("cuda", 0)
    r = torch.zeros((4, 5, 3), dtype=torch.float32)
    d = torch.zeros((4, 5, 3), dtype=torch.uint8)
    with pytest.raises(abi.GsmError, match="CUDA tensors"):
        _check_update_inputs(r, r, d, 5, 3, torch.float32, dev)
    with pytest.raises(TypeError):
        _check_update_inputs(r.double(), r.double(), d, 5, 3, torch.float32, dev)
    with pytest.raises(TypeError):
        _check_update_inputs(r, r, d.bool(), 5, 3, torch.float32, dev)
    for shape in ((4, 5, 2), (4, 15), (0, 5, 3), (4, 6, 3)):
        x = torch.zeros(shape)
        with pytest.raises(ValueError):
            _check_update_inputs(x, x, x.to(torch.uint8), 5, 3, torch.float32, dev)
    with pytest.raises(ValueError):
        _check_update_inputs(r, r[:2].repeat(2, 1, 1)[:, :4], d, 5, 3, torch.float32, dev)


def test_episode_io_mirror_matches_the_header_as_compiled_by_gcc(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    fields = [f for f, _ in abi.GsmEpisodeIO._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "gsmarl_b200.h"', 'int main(void) {',
             '  printf("sizeof %zu\\n", sizeof(gsm_episode_io));',
             '  printf("fields %d\\n", GSM_EPISODE_STAT_FIELDS);']
    lines += [f'  printf("{f} %zu\\n", offsetof(gsm_episode_io, {f}));' for f in fields]
    lines += ['  return 0;', '}']
    src = tmp_path / "episode_layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "episode_layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o",
                    str(exe)], check=True)
    got = dict(ln.split() for ln in subprocess.run([str(exe)], capture_output=True, text=True,
                                                   check=True).stdout.splitlines())
    assert int(got["sizeof"]) == C.sizeof(abi.GsmEpisodeIO)
    assert int(got["fields"]) == abi.GSM_EPISODE_STAT_FIELDS
    for f in fields:
        assert int(got[f]) == getattr(abi.GsmEpisodeIO, f).offset, f


def _host_io(n_envs=4, N=3, T=2):
    """A valid io over HOST arrays: every argument check returns before a pointer is dereferenced."""
    rows = n_envs * N
    a = {"reward": np.zeros((T, rows), np.float32), "cost": np.zeros((T, rows), np.float32),
         "done": np.zeros((T, rows), np.uint8), "carry_return": np.full(rows, 7.0), "carry_cost": np.full(rows, 7.0),
         "carry_length": np.full(rows, 7, np.int32), "totals": np.full(16, 7.0), "episodes": np.full(n_envs, 7, np.int32),
         "last_return": np.full(rows, 7.0), "last_cost": np.full(rows, 7.0), "last_length": np.full(rows, 7, np.int32),
         "team_last_return": np.full(n_envs, 7.0), "team_last_cost": np.full(n_envs, 7.0)}
    io = abi.GsmEpisodeIO()
    io.struct_size, io.dtype = C.sizeof(abi.GsmEpisodeIO), abi.GSM_F32
    for k, v in a.items():
        setattr(io, k, v.ctypes.data)
    io.n_rows = io.slot_rows = rows
    io.n_steps, io.agents_per_env = T, N
    return io, a


def test_invalid_arguments_return_their_status():
    lib = abi.load_library()
    ws = np.zeros(1 << 16, np.uint8)
    need = lib.gsm_episode_stats_workspace(12, 3)
    assert 0 < need <= ws.nbytes
    for args in ((-3, 3), (12, 0), (12, 1025), (13, 3)):
        assert lib.gsm_episode_stats_workspace(*args) == -1, args

    def status(mutate, n_bytes=ws.nbytes, workspace=ws.ctypes.data):
        io, keep = _host_io()
        mutate(io)
        return lib.gsm_episode_stats(C.byref(io), C.c_void_p(workspace), n_bytes, 0, None)
    assert status(lambda io: setattr(io, "struct_size", 8)) == -3
    for k in ("reward", "cost", "done", "carry_return", "carry_cost", "carry_length", "totals", "episodes"):
        assert status(lambda io: setattr(io, k, None)) == -1, k
    for k, v in (("n_steps", 0), ("agents_per_env", 0), ("agents_per_env", 1025), ("n_rows", 13),
                 ("n_rows", -3), ("slot_rows", 11), ("dtype", 2)):
        assert status(lambda io: setattr(io, k, v)) == -1, (k, v)
    assert status(lambda io: None, n_bytes=need - 1) == -1
    assert status(lambda io: None, workspace=None) == -1
    assert lib.gsm_episode_stats(None, None, 0, 0, None) == -1


def test_zero_rows_is_a_no_op():
    lib = abi.load_library()
    io, a = _host_io()
    io.n_rows = 0
    before = {k: v.copy() for k, v in a.items()}
    assert lib.gsm_episode_stats(C.byref(io), None, 0, 0, None) == 0
    for k, v in a.items():
        assert np.array_equal(v, before[k]), k


# ---- GPU ----------------------------------------------------------------------------------------------
def _synthetic(rng, n_envs, N, T_total, dtype, max_len):
    """reward, cost, done [T_total, n_envs * N]: done uniform per env at random episode lengths 1..max_len,
    integer-valued costs with many zeros."""
    done = np.zeros((T_total, n_envs), np.uint8)
    t = rng.integers(0, max_len, n_envs)                 # the first end: anywhere up to max_len - 1
    while True:
        live = t < T_total
        if not live.any():
            break
        done[t[live], np.nonzero(live)[0]] = 1
        t = t + rng.integers(1, max_len + 1, n_envs)
    done = np.repeat(done, N, axis=1)
    reward = rng.uniform(-1.0, 0.25, (T_total, n_envs * N)).astype(dtype)
    cost = ((rng.random((T_total, n_envs * N)) < 0.08) * rng.integers(1, 3, (T_total, n_envs * N))).astype(dtype)
    return reward, cost, done


class _FakeEnv:
    def __init__(self, n_envs, N, dtype):
        class W:
            pass
        self.world = W()
        self.world.n_agents, self.world.dtype = N, dtype
        self.n_envs, self.device = n_envs, torch.device("cuda", 0)


def _dev(x, n_envs, N):
    return torch.as_tensor(np.ascontiguousarray(x)).reshape(len(x), n_envs, N).cuda()


def _assert_state(tr, ref, ctx=""):
    def eq(name, got, want):
        g = got.cpu().numpy().reshape(-1)
        assert np.array_equal(g, np.asarray(want).astype(g.dtype), equal_nan=True), \
            f"{ctx} {name}: {int((g != want).sum())} rows differ"
    for k in ("carry_return", "carry_cost", "carry_length", "last_return", "last_cost", "last_length",
              "team_last_return", "team_last_cost"):
        eq(k, getattr(tr, k), getattr(ref, k))


# (N, n_envs): every block partial (n_envs not a multiple of the envs per block); N = 1 at 303404 envs has
# more row tiles than the grid has blocks, so blocks walk several tiles
SYNTH = [(1, 805), (3, 347), (12, 109), (96, 7), (1023, 3), (1, 1184 * 256 + 300)]


@gpu
@pytest.mark.parametrize("dtype", ["f32", "f64"])
@pytest.mark.parametrize("N,n_envs", SYNTH)
def test_synthetic_calls_match_the_reference(N, n_envs, dtype):
    rng = np.random.default_rng(N * 7919 + n_envs)
    Ts = (1, 3, 7, 25)
    reward, cost, done = _synthetic(rng, n_envs, N, sum(Ts), np.float32 if dtype == "f32" else np.float64, 32)
    tr = EpisodeTracker(_FakeEnv(n_envs, N, dtype), agent_cost_limit=1.0, team_cost_limit=2.0 * N)
    ref = Reference(n_envs, N, 1.0, 2.0 * N)
    t0, seen = 0, set()
    for T in Ts:
        sl = slice(t0, t0 + T)
        got = tr.update(_dev(reward[sl], n_envs, N), _dev(cost[sl], n_envs, N), _dev(done[sl], n_envs, N))
        want, eps = ref.call(reward[sl], cost[sl], done[sl])
        _assert_state(tr, ref, f"T={T}")
        assert np.array_equal(tr.episodes.cpu().numpy(), eps), f"T={T} episodes"
        assert_totals(got.cpu().numpy(), want, ctx=f"T={T}")
        seen |= set(np.unique(eps).tolist())
        t0 += T
    if n_envs >= 100:                                  # envs with none, one and several completions per call
        assert {0, 1} <= seen and max(seen) >= 2


@gpu
def test_chunked_calls_equal_one_call():
    N, n_envs = 3, 2000
    reward, cost, done = _synthetic(np.random.default_rng(5), n_envs, N, 60, np.float32, 40)
    one = EpisodeTracker(_FakeEnv(n_envs, N, "f32"), 1.0, 3.0)
    many = EpisodeTracker(_FakeEnv(n_envs, N, "f32"), 1.0, 3.0)
    t_one = one.update(_dev(reward, n_envs, N), _dev(cost, n_envs, N), _dev(done, n_envs, N))
    t_many, t0 = torch.zeros_like(t_one), 0
    for T in (10, 17, 33):
        sl = slice(t0, t0 + T)
        t_many += many.update(_dev(reward[sl], n_envs, N), _dev(cost[sl], n_envs, N), _dev(done[sl], n_envs, N))
        t0 += T
    for k in ("carry_return", "carry_cost", "carry_length", "last_return", "last_cost", "last_length",
              "team_last_return", "team_last_cost"):
        assert torch.equal(getattr(one, k).nan_to_num(-1), getattr(many, k).nan_to_num(-1)), k
    assert_totals(t_many.cpu().numpy(), t_one.cpu().numpy())


def _nav3_rollouts(env, B, T=10, rollouts=6):
    from gs_marl_b200.policy import GraphAttentionActor
    from gs_marl_b200.rollout import GraphRolloutBuffer, collect_fused
    actor = GraphAttentionActor(5, seed=4)
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    t0 = np.random.default_rng(11).integers(0, 25, B).astype(np.int32)
    env.set_state(step_count=t0)                           # staggered episode ends
    tr = EpisodeTracker(env, agent_cost_limit=1.0, team_cost_limit=2.0)
    tr.reset()
    slots = {k: [] for k in ("reward", "cost", "done")}
    window = torch.zeros(abi.GSM_EPISODE_STAT_FIELDS, dtype=torch.float64, device="cuda")
    for k in range(rollouts):
        collect_fused(env, actor, buf, seed=3, first_step=k * T)
        window += tr.update(buf["reward"], buf["cost"], buf["done"])
        for key in slots:
            slots[key].append(buf[key].cpu().numpy().reshape(T, -1))
        buf.after_update()
    return tr, window, {k: np.concatenate(v) for k, v in slots.items()}, t0


@gpu
@pytest.mark.parametrize("sharded", [False, True])
def test_staggered_rollouts_straddle_calls(sharded):
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv, StreamShardedEnv
    B, N = 16384, 3
    cfg = make_cfg("navigation", N, "f32", episode_length=25)
    env = (StreamShardedEnv(cfg, B, n_streams=4, auto_reset=True, seed=9) if sharded
           else MultiAgentGraphConstrainEnv(cfg, B, auto_reset=True, seed=9))
    tr, window, s, t0 = _nav3_rollouts(env, B)
    ref = Reference(B, N, 1.0, 2.0)
    want, _ = ref.call(s["reward"], s["cost"], s["done"])
    _assert_state(tr, ref)
    assert_totals(window.cpu().numpy(), want)
    # each env's first episode has 25 - t0 steps, every later one 25
    d = s["done"].reshape(60, B, N)
    assert (d == d[:, :, :1]).all()
    first = np.argmax(d[:, :, 0], axis=0)
    assert np.array_equal(first + 1, 25 - t0)
    ends = [np.nonzero(d[:, g, 0])[0] for g in range(0, B, 97)]
    assert all((np.diff(e) == 25).all() for e in ends)
    assert (tr.last_length.cpu().numpy() == 25).all()     # every env has completed a second episode by slot 49
    env.close()


@gpu
def test_aligned_rollout_gives_the_buffer_sum():
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
    from gs_marl_b200.policy import GraphAttentionActor
    from gs_marl_b200.rollout import GraphRolloutBuffer, collect_fused
    B, N, T = 4096, 3, 25
    env = MultiAgentGraphConstrainEnv(make_cfg("navigation", N, "f32", episode_length=T), B, auto_reset=True, seed=2)
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    tr = EpisodeTracker(env)
    tr.reset()
    collect_fused(env, GraphAttentionActor(5, seed=1), buf, seed=5)
    tr.update(buf["reward"], buf["cost"], buf["done"])
    want = torch.zeros((B, N), dtype=torch.float64, device="cuda")
    for t in range(T):
        want += buf["reward"][t].double()
    assert torch.equal(tr.last_return, want)
    assert (tr.episodes == 1).all() and (tr.last_length == T).all()
    env.close()


@gpu
def test_fp64_team_kernel_rollout():
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
    from tests._util import random_actions
    B, N = 1001, 6
    cfg = make_cfg("polygon", N, "f64", episode_length=7)
    env = MultiAgentGraphConstrainEnv(cfg, B, seed=4)
    env.reset()
    tr = EpisodeTracker(env, agent_cost_limit=0.5, team_cost_limit=1.5)
    ref = Reference(B, N, 0.5, 1.5)
    rng = np.random.default_rng(8)
    for T in (9, 11):
        out = env.rollout(torch.as_tensor(random_actions(cfg, rng, (T, B))).cuda(), auto_reset=True)
        got = tr.update(out["reward"], out["cost"], out["done"])
        want, eps = ref.call(*(out[k].cpu().numpy().reshape(T, -1) for k in ("reward", "cost", "done")))
        _assert_state(tr, ref, f"T={T}")
        assert np.array_equal(tr.episodes.cpu().numpy(), eps)
        assert_totals(got.cpu().numpy(), want)
    assert ref.last_length.min() >= 1                       # every agent row has completed an episode
    env.close()


@gpu
def test_deterministic_across_streams_and_graph_replay():
    N, n_envs = 3, 120000                                   # 1412 row tiles: blocks walk several
    reward, cost, done = _synthetic(np.random.default_rng(1), n_envs, N, 25, np.float32, 30)
    r, c, d = _dev(reward, n_envs, N), _dev(cost, n_envs, N), _dev(done, n_envs, N)
    tr = EpisodeTracker(_FakeEnv(n_envs, N, "f32"), 1.0, 3.0)
    tr.update(r, c, d)                                      # a carry to start from
    state = ("carry_return", "carry_cost", "carry_length", "last_return", "last_cost", "last_length",
             "team_last_return", "team_last_cost", "episodes")
    s0 = {k: getattr(tr, k).clone() for k in state}

    def restore():
        for k in state:
            getattr(tr, k).copy_(s0[k])
    outs = []
    for st in (torch.cuda.Stream(), torch.cuda.Stream()):
        restore()
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            t = tr.update(r, c, d)
        torch.cuda.current_stream().wait_stream(st)
        outs.append((t.clone(), {k: getattr(tr, k).clone() for k in state}))
    assert torch.equal(outs[0][0], outs[1][0])
    restore()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        t_graph = tr.update(r, c, d)
    restore()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(t_graph, outs[0][0])
    for k in state:
        assert torch.equal(getattr(tr, k).nan_to_num(-1), outs[0][1][k].nan_to_num(-1)), k


@gpu
@pytest.mark.parametrize("N,n_envs,dtype", [(3, 347, "f32"), (1023, 3, "f64"), (12, 109, "f32")])
def test_no_writes_outside_the_buffers(N, n_envs, dtype):
    """Every output, carry and the workspace sit between 4 KB guard bands that must stay untouched."""
    lib = abi.load_library()
    G, rows, T = 4096, n_envs * N, 13
    reward, cost, done = _synthetic(np.random.default_rng(3), n_envs, N, T, np.float32 if dtype == "f32"
                                    else np.float64, 6)
    r, c, d = (torch.as_tensor(x).cuda() for x in (reward, cost, done))
    n_ws = lib.gsm_episode_stats_workspace(rows, N)
    sizes = {"carry_return": (rows, torch.float64), "carry_cost": (rows, torch.float64),
             "carry_length": (rows, torch.int32), "totals": (16, torch.float64), "episodes": (n_envs, torch.int32),
             "last_return": (rows, torch.float64), "last_cost": (rows, torch.float64),
             "last_length": (rows, torch.int32), "team_last_return": (n_envs, torch.float64),
             "team_last_cost": (n_envs, torch.float64), "workspace": (n_ws, torch.uint8)}
    raw, view = {}, {}
    for k, (n, dt) in sizes.items():
        nb = n * torch.empty((), dtype=dt).element_size()
        raw[k] = torch.full((nb + 2 * G,), 0xA5, dtype=torch.uint8, device="cuda")
        view[k] = raw[k][G:G + nb].view(dt)
        view[k].zero_()
    io = abi.GsmEpisodeIO()
    io.struct_size, io.dtype = C.sizeof(abi.GsmEpisodeIO), abi.GSM_F32 if dtype == "f32" else abi.GSM_F64
    io.reward, io.cost, io.done = r.data_ptr(), c.data_ptr(), d.data_ptr()
    for k in sizes:
        if k != "workspace":
            setattr(io, k, view[k].data_ptr())
    io.n_rows = io.slot_rows = rows
    io.n_steps, io.agents_per_env = T, N
    io.agent_cost_limit, io.team_cost_limit = 1.0, 2.0
    for _ in range(2):
        assert lib.gsm_episode_stats(C.byref(io), C.c_void_p(view["workspace"].data_ptr()), n_ws, 0,
                                     C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
    torch.cuda.synchronize()
    for k, b in raw.items():
        assert bool((b[:G] == 0xA5).all()) and bool((b[-G:] == 0xA5).all()), f"{k}: guard band overwritten"
    assert int(view["totals"][0]) > 0 and int(view["episodes"].sum()) > 0


@gpu
def test_summary_and_masked_reset():
    N, n_envs = 2, 3
    tr = EpisodeTracker(_FakeEnv(n_envs, N, "f64"), agent_cost_limit=0.5, team_cost_limit=0.5)
    assert math.isnan(EpisodeTracker.summary(torch.zeros(16, dtype=torch.float64))["team_return_mean"])
    r = torch.ones((2, n_envs, N), dtype=torch.float64, device="cuda")
    c = torch.zeros_like(r)
    c[0, 0, 1] = 1.0
    d = torch.zeros((2, n_envs, N), dtype=torch.uint8, device="cuda")
    d[1] = 1
    s = EpisodeTracker.summary(tr.update(r, c, d))
    assert s["episodes"] == 6 and s["team_episodes"] == 3
    assert s["return_mean"] == 2.0 and s["return_std"] == 0.0 and s["length_mean"] == 2.0
    assert abs(s["cost_mean"] - 1 / 6) < 1e-15 and abs(s["safe_rate"] - 5 / 6) < 1e-15
    assert abs(s["over_limit_rate"] - 1 / 6) < 1e-15 and abs(s["team_over_limit_rate"] - 1 / 3) < 1e-15
    d.zero_()
    tr.update(r, c, d)
    tr.reset(torch.tensor([True, False, True]))
    assert tr.carry_length.cpu().tolist() == [[0, 0], [2, 2], [0, 0]]
    with pytest.raises(abi.GsmError):
        tr.update(r.cpu(), c.cpu(), d.cpu())
