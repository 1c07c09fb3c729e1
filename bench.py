#!/usr/bin/env python
"""bench.py — agent-steps/s of the batched GS-MARL env hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (this repo's arm)
    python bench.py --impl reference --gpus N --steps K --warmup W   (CPU arm)

A "step" is one env step of the whole batch: BASELINE.json configs[1] — cooperative
navigation, 3 agents, 16384 envs per GPU, random discrete actions — in the production
precision (fp32).  `value` is device-resident throughput over exactly K timed steps (actions
already in HBM, outputs written to a rotating 25-slot rollout buffer larger than L2, 25 steps
per fused launch).  `e2e` is the same metric through the numpy-facing drop-in (`GraphVecEnv.step`):
host actions in, host outputs out, both copies inside the timed region.

`--dump-outputs DIR` writes what the last timed step computed (the nine outputs of rank 0's envs)
as DIR/<name>.npy.  The inputs are seeded and the warm-up and timed steps run from the reset state,
so two builds run with the same arguments can be compared output for output.

IMPORTANT LABEL: the GS-MARL env sources are withheld (reference readme.md:1), so the
model is the declared one of SPEC.md with the UNVERIFIED constants of
gs_marl_b200/presets.py, and the CPU arm is this repo's reference-STYLE numpy port
(oracle/py_env.py: one Python env object per world, subprocess workers), not GS-MARL's
own code.  Every JSON line says so in `config.spec_status`.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_AGENTS = 3
ENVS_PER_GPU = 16384
ROLLOUT_T = 25      # steps fused per launch (rollout-buffer slots)
EPISODE_LEN = 25    # envs are re-drawn in-kernel every EPISODE_LEN steps
SPEC_STATUS = ("declared model (SPEC.md) with UNVERIFIED constants; GS-MARL env sources withheld, "
               "parity with the reference unpinned")
METRIC = "agent-steps/sec (graph obs+reward+cost) at 1/2/4/8 B200; % HBM roofline"   # BASELINE.json
UNIT = "agent-steps/s"


def workload_config(n_gpus, envs_per_gpu=ENVS_PER_GPU):
    """The `config` object of BOTH arms (this repo's and `--impl reference`): identical keys and
    values for the same command line, so that the driver can prove both ran the same workload.
    How each arm runs it lives elsewhere (`method` here, `cpu_baseline.sample` there)."""
    return {"workload": f"cooperative navigation, {N_AGENTS} agents, {envs_per_gpu} envs per GPU, "
                        "random discrete actions, fp32 production mode",
            "n_agents": N_AGENTS, "envs_per_gpu": envs_per_gpu, "global_envs": envs_per_gpu * n_gpus,
            "episode_length": EPISODE_LEN,
            "parallelism": f"env-sharded x{n_gpus}, no collective on the step path",
            "spec_status": SPEC_STATUS}


# ---------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0=None, t1=None):
        """Median SM clock of the samples that arrived inside [t0, t1] (the timed region); if the
        region was shorter than the sampling period, of all samples taken under load."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def parse(rows):
            sm, mx, reasons = [], [], set()
            for _, ln in rows:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for nm, v in zip(names, f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            return sm, mx, reasons
        inside = [r for r in self.lines if t0 is not None and t0 <= r[0] <= t1]
        window = "timed region"
        if not inside:
            inside, window = self.lines, "warm-up + timed region (region shorter than the 50 ms sampling period)"
        sm, mx, reasons = parse(inside)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


def pin_to_gpu_numa(gpu_index):
    """Bind this rank to the CPUs NVML reports as local to its GPU, before any pinned host memory
    is allocated, so that the e2e arena and the copy threads sit on the GPU's own socket."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {w * 64 + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cpus local to gpu {gpu_index}"
    except Exception as e:        # topology unknown: leave the affinity alone
        return f"unpinned ({type(e).__name__})"
    return "unpinned"


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(outputs, out_dir, limit=DUMP_LIMIT_BYTES):
    """Write each output (leading dimension: envs) as out_dir/<name>.npy: real outputs in their own
    precision, integer ones as float64 (exact; adj as its unsigned bit masks).  If all of them would
    take more than `limit` bytes, every file holds the same fixed, seeded sample of env rows, and
    env_index.npy says which."""
    import numpy as np
    arrays = {}
    for k, v in outputs.items():
        a = v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)
        if k == "adj":
            a = a.view(np.uint32)
        arrays[k] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    n_envs = len(next(iter(arrays.values())))
    per_env = sum(a.nbytes for a in arrays.values()) // n_envs
    if per_env * n_envs > limit:
        keep = (limit - 4096 * (len(arrays) + 1)) // (per_env + 8)      # room for the .npy headers and the index
        idx = np.sort(np.random.default_rng(0).choice(n_envs, keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def ncu_traffic():
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


# ---------------------------------------------------------------------------------------
# CPU arm: reference-STYLE numpy port in subprocess workers (SubprocVecEnv lineage)
def _cpu_worker(conn, n_envs, seed):
    import numpy as np
    from oracle import gsm_oracle as O, py_env, worlds
    cfg = worlds.make_world("navigation", N_AGENTS, dtype="f64")      # the oracle's own table of the workload
    init = O.OracleEnv(cfg, n_envs, env_offset=seed * 100003)
    init.reset(1)
    envs = [py_env.PyEnv(cfg) for _ in range(n_envs)]
    for b, e in enumerate(envs):
        e.set_state(init.agent_state[b], init.landmark_pos[b])
    rng = np.random.default_rng(seed)
    conn.send("ready")
    while True:
        cmd = conn.recv()
        if cmd == "close":
            break
        acts = rng.integers(0, 5, (n_envs, N_AGENTS))
        outs = [e.step(acts[b]) for b, e in enumerate(envs)]
        # stack like the vec-env wrapper does (obs, graph, reward, cost, done per env)
        stacked = {k: np.stack([o[k] for o in outs]) for k in outs[0]}
        conn.send(float(stacked["reward"].sum()))
    conn.close()


class CpuVecEnv:
    def __init__(self, n_envs, cores):
        import multiprocessing as mp
        ctx = mp.get_context("spawn")
        self.cores = max(1, min(cores, n_envs))
        per = [n_envs // self.cores + (1 if r < n_envs % self.cores else 0) for r in range(self.cores)]
        self.n_envs = n_envs
        self.conns, self.procs = [], []
        for r, m in enumerate(per):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker, args=(b, m, r), daemon=True)
            p.start()
            self.conns.append(a); self.procs.append(p)
        for c in self.conns:
            assert c.recv() == "ready"

    def step(self):
        for c in self.conns:
            c.send("step")
        return sum(c.recv() for c in self.conns)

    def close(self):
        for c in self.conns:
            c.send("close")
        for p in self.procs:
            p.join(5)


def cpu_sample_envs(total_budget_s, n_steps):
    """Env count of the bounded CPU sample used by the GPU arm's `cpu_baseline` leg only (the
    reference ARM never shrinks its workload): sized so n_steps steps take about total_budget_s."""
    cores = os.cpu_count() or 1
    probe = CpuVecEnv(cores * 2, cores)
    probe.step()
    t0 = time.perf_counter()
    for _ in range(3):
        probe.step()
    per_env_step = (time.perf_counter() - t0) / 3 / 2          # seconds per env-step per core
    probe.close()
    # at least 8 envs per worker so that pipe round-trips do not dominate what is measured
    envs = int(max(cores * 8, min(ENVS_PER_GPU, total_budget_s / max(n_steps, 1) / per_env_step * cores)))
    return cores, envs


def cpu_c_oracle_rate(seconds=3.0):
    """The C restatement of the same model on all cores (a much stronger CPU baseline than the
    reference's Python style) — reported for context."""
    import numpy as np
    from oracle import gsm_oracle as O, worlds
    cores = os.cpu_count() or 1
    O.set_threads(cores)
    cfg = worlds.make_world("navigation", N_AGENTS, dtype="f32")
    env = O.OracleEnv(cfg, ENVS_PER_GPU)
    env.reset(1)
    bufs = env.alloc_io()
    a = np.random.default_rng(0).integers(0, 5, (ENVS_PER_GPU, N_AGENTS)).astype(np.int32)
    env.step(a, bufs)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        env.step(a, bufs); n += 1
    dt = time.perf_counter() - t0
    O.set_threads(1)
    return {"value": n * ENVS_PER_GPU * N_AGENTS / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"C oracle (oracle/gsm_oracle.c, fp32), {ENVS_PER_GPU} envs x {n} steps, pthreads"}


def run_reference(args):
    """The CPU arm: the reference-STYLE numpy port in subprocess workers on all host cores, on EXACTLY
    the GPU arm's workload — `--envs` (default 16384) envs per step, never a smaller sample: one
    step is ~0.1 s on 16 cores, so the driver's --steps/--warmup finish in seconds.  Same `config`
    as the GPU arm for the same command line."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    cores, envs = os.cpu_count() or 1, args.envs
    vec = CpuVecEnv(envs, cores)
    if vec.n_envs != envs:
        raise SystemExit("reference arm could not build the full workload")
    for _ in range(warm):
        vec.step()
    t0 = time.perf_counter()
    for _ in range(steps):
        vec.step()
    dt = time.perf_counter() - t0
    vec.close()
    value = envs * N_AGENTS * steps / dt
    sample = (f"reference-STYLE numpy port (oracle/py_env.py; GS-MARL's own env is withheld), fp64, "
              f"the full workload: {envs} envs per step in {vec.cores} subprocess workers, {steps} steps")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.gpus, envs),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": vec.cores, "kind": "port", "sample": sample,
                             "sample_envs_per_step": envs},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------
def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from gs_marl_b200 import scenarios
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
    from gs_marl_b200.env_wrappers import GraphVecEnv, ShardedStats

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = pin_to_gpu_numa(local)
    if world > 1:
        # NCCL prints its version banner to stdout when the first communicator is built; stdout
        # must carry exactly one JSON line, so fd 1 points at stderr until NCCL is up.
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    K, W, T = args.steps, args.warmup, args.rollout_t
    sampler = ClockSampler(local); sampler.start()
    spec_p = os.environ.get("GSM_SPEC_P", "4 (default)")
    cfg = scenarios.load("navigation").make_world(N_AGENTS, dtype="f32", episode_length=EPISODE_LEN)
    env = MultiAgentGraphConstrainEnv(cfg, args.envs, device=local, env_offset=rank * args.envs, seed=1)
    env.reset()
    gen = torch.Generator(device=dev); gen.manual_seed(rank)
    acts = torch.randint(0, 5, (T, args.envs, N_AGENTS), generator=gen, device=dev, dtype=torch.int32)
    ring = {k: env._alloc(k, (T,)) for k in env.OUTPUTS}       # rollout buffer, T slots
    ring_bytes = sum(v.numel() * v.element_size() for v in ring.values())

    import ctypes as C
    from bench_util import GRAPH_CHUNK_STEPS, RolloutRegion, time_rollouts
    from gs_marl_b200.environment import StreamShardedEnv
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    # The timed region drives S contiguous sub-shards of this GPU's envs, each its own handle on
    # its own stream, all filling the SAME rollout buffer (gsm_set_slot_envs): the tail of one
    # shard's launch overlaps the body of the next (StreamShardedEnv docstring; --streams 1 = one handle).
    S = max(1, args.streams)
    sh_env = StreamShardedEnv(cfg, args.envs, n_streams=S, device=local, env_offset=rank * args.envs, seed=1)
    sh_env.reset()
    start_state, start_episode = sh_env.get_state(), sh_env.get_episode()

    # ---- THE timed region: exactly K env steps = fused T-step launches on the S shard streams,
    # captured in a CUDA graph (fork / join inside); envs are re-drawn in-kernel every EPISODE_LEN
    # steps (state and episode counters persist across replays); all nine outputs are written.
    region = RolloutRegion(sh_env, acts, ring, K, T, auto_reset=True, pack=False)
    # untimed pre-run: loads the modules and brings the clocks up.  The clock sampler was started
    # first thing in this function; on a busy host (8 ranks, 8 nvidia-smi processes) its first sample
    # can take seconds: keep the GPU under load until it reports (bounded)
    for _ in range(max(1, GRAPH_CHUNK_STEPS // K)):
        region.replay_unit()
    torch.cuda.synchronize()
    t_wait = time.time()
    while not sampler.lines and time.time() - t_wait < 15.0:
        region.replay_unit()
        torch.cuda.synchronize()
    # the pre-run ran for a time-dependent number of steps: start again from the reset state, so that
    # every run computes the same steps (--dump-outputs compares builds output for output)
    sh_env.set_state(*start_state)
    sh_env.set_episode(start_episode)
    barrier()
    wall0 = time.time()
    # warm-up: ceil(max(W, 256) / K) replays of the K-step region, enqueued right before the timed one so
    # that the GPU is still busy with them when the first event is recorded (no launch gap inside the events)
    for _ in range(-(-max(W, 256) // K)):
        region.replay_unit()
    ms, repeats = region.run(1)
    barrier()
    wall1 = time.time()
    clocks = sampler.stop(wall0, wall1)
    if args.dump_outputs and rank == 0:
        dump_outputs({k: ring[k][region.last_slot] for k in sh_env.OUTPUTS}, args.dump_outputs)
    launches = repeats * region.launches_per_region
    bytes_region = region.bytes_per_region(cfg)

    # ---- the same kernel in other arrangements (explains the headline; same graph method, shorter) ----
    side_ms = min(args.region_ms, 60.0)
    plain = time_rollouts(sh_env, cfg, acts, ring, K, T, False, side_ms)       # MODE 0: no auto-reset
    one_auto = time_rollouts(env, cfg, acts, ring, K, T, True, side_ms)        # ONE launch per T steps
    one_plain = time_rollouts(env, cfg, acts, ring, K, T, False, side_ms)
    env._check(env.lib.gsm_set_auto_reset(env._h, 0))

    # ---- un-fused API: one gsm_step launch per env step (what a policy-in-the-loop caller uses) ----
    io_slots = [env._make_io({k: v[sidx] for k, v in ring.items()}, acts[sidx]) for sidx in range(T)]
    env._check(env.lib.gsm_set_auto_reset(env._h, 0))
    n_single = max(T, min(2000, K))
    for sidx in range(T):
        env._check(env.lib.gsm_step(env._h, C.byref(io_slots[sidx]), stream))
    torch.cuda.synchronize()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for q in range(n_single):
        env._check(env.lib.gsm_step(env._h, C.byref(io_slots[q % T]), stream))
    s1.record()
    torch.cuda.synchronize()
    single_us = s0.elapsed_time(s1) * 1e3 / n_single

    # ---- same kernel at a batch that saturates the GPU (explains the small-batch fraction) -------
    large = None
    if world == 1 and args.large_envs > 0:
        nl = args.large_envs
        big = MultiAgentGraphConstrainEnv(cfg, nl, device=local, seed=2)
        big.reset()
        Tl = 8
        bacts = torch.randint(0, 5, (Tl, nl, N_AGENTS), generator=gen, device=dev, dtype=torch.int32)
        bring = {k: big._alloc(k, (Tl,)) for k in big.OUTPUTS}
        r = time_rollouts(big, cfg, bacts, bring, Tl, Tl, True, side_ms)
        pk, _ = measured_peak()
        large = {"envs": nl, "step_us": r["step_us"], "achieved": r["achieved"], "unit": "GB/s",
                 "frac": r["achieved"] / pk, "agent_steps_per_s": nl * N_AGENTS / (r["step_us"] * 1e-6),
                 "steps_per_launch": Tl,
                 "buffer_mb": sum(v.numel() * v.element_size() for v in bring.values()) / 1e6}
        big.close()
        del bring, bacts

    # ---- BASELINE configs[2], [3], [4] in the same run, under the same clock record --------------
    other = None
    if args.configs:
        other = other_configs(args, local, rank, world, dev)

    # ---- closed loop: a random-init graph policy (plain PyTorch, library kernels) picks the actions
    # from obs + neighbour rows every step; one gsm_step launch per env step (BASELINE configs[4]
    # flavour: the env feeding a policy on the same GPU, nothing leaves the device)
    closed = None
    if args.closed_loop_steps > 0:
        closed = closed_loop(env, cfg, args.closed_loop_steps, dev)
        closed["fused_actor"] = closed_loop_fused(cfg, args.envs, args.closed_loop_steps, local, rank,
                                                  args.collect_streams)

    # ---- e2e through the numpy-facing drop-in ------------------------------------------------
    vec = GraphVecEnv(cfg, args.envs, device=local, env_offset=rank * args.envs, seed=1)
    vec.reset()
    host_acts = np.random.default_rng(rank).integers(0, 5, (8, args.envs, N_AGENTS)).astype(np.int32)
    stats = ShardedStats()
    Ke = max(10, min(args.e2e_steps, K))
    for s in range(5):
        vec.step(host_acts[s % 8])
    barrier()
    t0 = time.perf_counter()
    for s in range(Ke):
        obs, graph, rew, cost, done, infos = vec.step(host_acts[s % 8])
        if s % EPISODE_LEN == EPISODE_LEN - 1:
            vec.reset()
    e2e_s = time.perf_counter() - t0
    stats.add(args.envs * Ke, N_AGENTS, float(rew.sum()), float(cost.sum()), float(done.sum()))
    h2d = host_acts[0].nbytes
    d2h_dense = sum(v.nbytes for k, v in vec.buf.items() if k != "actions")
    # bytes that actually cross PCIe per step in the default (sparse) mode: the dense small outputs plus the
    # nbr_cnt valid rows of nbr_feat / nbr_idx (counted on the last step's nbr_cnt)
    row_b = vec.buf["nbr_feat"].itemsize * vec.buf["nbr_feat"].shape[-1]
    d2h = d2h_dense - vec.buf["nbr_feat"].nbytes + int(graph["nbr_cnt"].sum()) * row_b

    def e2e_variant(n, **kw):
        vec.set_host_outputs(**kw)
        for s_ in range(3):
            vec.step(host_acts[s_ % 8])
        t1 = time.perf_counter()
        for s_ in range(n):
            vec.step(host_acts[s_ % 8])
        return args.envs * N_AGENTS * n / (time.perf_counter() - t1)
    e2e_dense = e2e_variant(max(10, Ke // 4), outputs=None, sparse=False)
    lean = [k for k in vec.buf if k not in ("actions", "nbr_idx", "assign")]
    e2e_lean = e2e_variant(max(10, Ke // 4), outputs=lean, sparse=True)
    vec.close()
    # the ceiling of that path on this box: one pinned D2H copy of the same size, nothing else
    dsrc = torch.empty(d2h_dense, dtype=torch.uint8, device=dev)
    hdst = torch.empty(d2h_dense, dtype=torch.uint8, pin_memory=True)
    for _ in range(3):
        hdst.copy_(dsrc, non_blocking=True)
    torch.cuda.synchronize()
    tp0 = time.perf_counter()
    for _ in range(20):
        hdst.copy_(dsrc, non_blocking=True)
        torch.cuda.synchronize()
    pcie_d2h_gbs = d2h_dense * 20 / (time.perf_counter() - tp0) / 1e9
    del dsrc, hdst

    cl_ms = [closed["ms"], closed["fused_actor"]["ms"]] if closed is not None else [0.0, 0.0]
    tms = torch.tensor([ms, e2e_s * 1e3] + cl_ms, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    totals = stats.all_reduce(device=dev)        # the only collective: final stats gather
    ms, e2e_ms, cl_torch_ms, cl_fused_ms = tms.tolist()

    if rank == 0:
        agents = args.envs * N_AGENTS
        value = agents * K * repeats * world / (ms * 1e-3)
        step_us = ms * 1e3 / (repeats * K)
        peak, peak_src = measured_peak()
        achieved = bytes_region * repeats / (ms * 1e-3) / 1e9
        per_step_bytes = cfg.bytes_per_agent_step() * agents     # state r/w charged every step (r1 accounting)
        region_desc = ("one CUDA graph" if K <= GRAPH_CHUNK_STEPS else
                       f"CUDA graphs of {GRAPH_CHUNK_STEPS}-step chunks")

        def variant(r):
            return {"step_us": r["step_us"], "achieved": r["achieved"], "frac": r["achieved"] / peak}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "repeats": repeats, "ms_per_step": ms / (repeats * K), "timed_region_ms": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(world, args.envs),
            "method": {
                "l2_policy": f"outputs rotate through a {T}-slot rollout buffer of {ring_bytes / 1e6:.0f} MB "
                             "(> 126 MB L2); no explicit flush",
                "episode": f"episode_length {EPISODE_LEN}: every env is re-drawn in-kernel every {EPISODE_LEN} steps "
                           "(gsm_set_auto_reset; state persists across launches and graph replays)",
                "launch": f"fused launches of min({T}, remaining) steps (gsm_rollout); {S} contiguous env sub-shards of "
                          f"{args.envs // S} envs, one handle + one CUDA stream each, all writing the same rollout "
                          f"buffer (gsm_set_slot_envs)",
                "timed_region": f"exactly K = {K} steps, captured in {region_desc} (shard streams fork and join inside "
                                f"the graph) and replayed once between two CUDA events, right behind the warm-up "
                                f"(ceil(max(W, 256) / K) replays from the reset state): {ms:.3f} ms; ms_per_step = "
                                "region time / K; no host launch inside the events",
                "streams": S},
            "env_steps_per_s": value / N_AGENTS,
            "clocks": clocks,
            "e2e": {"value": agents * Ke * world / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "d2h_bytes_per_step_dense": d2h_dense,
                    "d2h_bytes_note": "d2h_bytes_per_step = the small outputs in full + the nbr_cnt valid rows of nbr_feat "
                                      "(last step's counts): an UPPER bound, the slowly changing small outputs cross as "
                                      "changed 16-byte pieces only; d2h_bytes_per_step_dense = the nine host arrays",
                    "steps": Ke,
                    "api": "GraphVecEnv.step -> gsm_step_host (mapped pinned arena; 1 H2D copy + the step kernel + one "
                           "export kernel that writes the outputs into the host arrays over PCIe: the nbr_cnt valid rows "
                           "of nbr_feat, obs / reward in full, the 16-byte pieces of the other outputs that changed; all "
                           "nine host arrays bit-identical to the device tensors)",
                    "host_affinity": numa,
                    "bound": "PCIe D2H of the step's outputs",
                    "d2h_gbs_achieved": d2h * Ke / e2e_s / 1e9,
                    "d2h_gbs_ceiling": pcie_d2h_gbs,
                    "ceiling_note": "one pinned cudaMemcpy D2H of the DENSE outputs + sync, measured in this run "
                                    "on rank 0 (the e2e step adds the H2D of the actions, the kernels and the "
                                    "Python wrapper)",
                    "dense_copy_variant": {"value": e2e_dense * world, "note": "rank 0 x world; gsm_set_host_outputs("
                                           "sparse = 0): one dense D2H copy per step (the round-1 path)"},
                    "lean_variant": {"value": e2e_lean * world, "note": "rank 0 x world; sparse, nbr_idx (redundant "
                                     "with adj) and assign (the identity in navigation) switched off"}},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(),
                         "kernel": "gsm::env_wide_kernel<float, N=3, L=6, MODE=2 (auto-reset), K=8>" if not os.environ.get("GSM_NO_WIDE")
                                   else f"gsm::env_steps_kernel<float, NAVIGATION, 3, 6, P={spec_p}, MODE=2 (auto-reset)>",
                         "how": "THE timed region itself (same events as `value`): algorithmic bytes of every fused "
                                "launch in it (WorldConfig.bytes_fused: action + all outputs per step; agent state, "
                                "landmarks and step counter once per launch) / region time, max over ranks",
                         "step_us": step_us,
                         "algorithmic_bytes_per_region": bytes_region,
                         "algorithmic_bytes_per_agent_step": bytes_region / (agents * K),
                         "frac_per_step_accounting": per_step_bytes / (step_us * 1e-6) / 1e9 / peak,
                         "per_step_accounting_note": f"round-1 figure: {cfg.bytes_per_agent_step()} B per agent-step, i.e. "
                                                     "state read+write, landmarks and counter charged on EVERY step "
                                                     "although a fused launch moves them once",
                         "plain_variant": variant(plain),
                         "one_stream": {"note": "the same envs as ONE launch per fused rollout on one stream (what a single "
                                                "ncu launch corresponds to)",
                                        "auto_reset": variant(one_auto), "plain": variant(one_plain)},
                         "peak_source": peak_src,
                         "note": "layout is the declared one of SPEC.md §6 (reference layout unknown)"},
            "single_step_api": {"value": agents * world / (single_us * 1e-6), "unit": UNIT,
                                "us_per_step": single_us, "steps": n_single,
                                "note": "gsm_step, one kernel launch per env step from Python, outputs to rotating slots"},
            "final_stats": totals,
        }
        if world == 1 and not args.no_cpu:
            cores, envs = cpu_sample_envs(args.cpu_budget, 10)
            cvec = CpuVecEnv(envs, cores)
            cvec.step()
            t0 = time.perf_counter()
            for _ in range(10):
                cvec.step()
            dt = time.perf_counter() - t0
            cvec.close()
            line["cpu_baseline"] = {
                "value": envs * N_AGENTS * 10 / dt, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"reference-STYLE numpy port (oracle/py_env.py; GS-MARL's own env is withheld), "
                          f"fp64, {envs} envs x 10 steps in {cores} subprocess workers"}
            line["cpu_baseline_c_port"] = cpu_c_oracle_rate()
        if world == 1 and args.large_envs > 0:
            line["roofline_large_batch"] = large
        if other is not None:
            line["configs"] = other
        if closed is not None:
            # every rank runs the same closed loop on its own shard: whole-job value from the MAX time
            closed["value"] = agents * closed["steps"] * world / (cl_torch_ms * 1e-3)
            f = closed["fused_actor"]
            f["value"] = agents * f["steps"] * world / (cl_fused_ms * 1e-3)
            line["closed_loop"] = closed

        print(json.dumps(line), flush=True)
    env.close()
    sh_env.close()
    if world > 1:
        dist.destroy_process_group()


OTHER_CONFIGS = [   # BASELINE.json configs[2] and [3]: (label, scenario, N, envs per GPU, make_world kwargs)
    ("configs[2] navigation 24 agents x 4096 envs", "navigation", 24, 4096, {"max_nbrs": 32}),
    ("configs[2] navigation 48 agents x 4096 envs", "navigation", 48, 4096, {"max_nbrs": 32}),
    ("configs[2] navigation 96 agents x 4096 envs", "navigation", 96, 4096, {"max_nbrs": 32}),
    ("configs[3] polygon 6 agents x 16384 envs", "polygon", 6, 16384, {}),
    ("configs[3] polygon 12 agents x 16384 envs", "polygon", 12, 16384, {}),
    ("configs[3] line 6 agents x 16384 envs", "line", 6, 16384, {}),
    ("configs[3] line 12 agents x 16384 envs", "line", 12, 16384, {}),
]


def other_configs(args, local, rank, world, dev):
    """Device-resident step time of BASELINE.json configs[2] (navigation 24/48/96 agents x 4096 envs),
    configs[3] (polygon / line, 6 and 12 agents, per-step batched assignment) and configs[4] (navigation
    12 agents, 65536 envs over the job's GPUs, closed loop with a random-init graph actor), measured in
    THIS run under the same clock record as the headline: fused rollouts with in-kernel auto-reset,
    CUDA-graph replay for >= --config-ms, every rank runs its own copy (weak scaling, like the headline)
    except configs[4], which shards a fixed 65536 envs (strong)."""
    import torch
    import torch.distributed as dist
    from bench_util import time_rollouts
    from gs_marl_b200 import scenarios
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv, StreamShardedEnv
    peak, _ = measured_peak()
    rows, times = [], []
    for label, scn, N, n_envs, kw in OTHER_CONFIGS:
        cfg = scenarios.load(scn).make_world(N, dtype="f32", **kw)     # episode length: the scenario's own (25 / 100)
        per_step = cfg.bytes_fused(n_envs, 1)
        T = 25 if per_step * 25 < 6e9 else 8                 # rollout-buffer slots; always > L2
        S = max(1, args.streams)
        env = (StreamShardedEnv(cfg, n_envs, n_streams=S, device=local, env_offset=rank * n_envs, seed=5)
               if S > 1 else MultiAgentGraphConstrainEnv(cfg, n_envs, device=local, env_offset=rank * n_envs, seed=5))
        env.reset()
        acts = torch.randint(0, 5, (T, n_envs, N), device=dev, dtype=torch.int32)
        ring = {k: env._alloc(k, (T,)) for k in env.OUTPUTS}
        r = time_rollouts(env, cfg, acts, ring, T, T, True, args.config_ms)
        env.close()
        rows.append({"config": label, "envs_per_gpu": n_envs, "n_agents": N, "steps_per_launch": T, "streams": S,
                     "max_nbrs": cfg.max_nbrs, "episode_length": cfg.episode_length, "bytes_per_agent_step": cfg.bytes_fused(n_envs, T) / (n_envs * N * T),
                     "buffer_mb": sum(v.numel() * v.element_size() for v in ring.values()) / 1e6,
                     "regions": r["regions"], "region_ms": r["ms"], "_bytes": cfg.bytes_fused(n_envs, T)})
        times.append(r["ms"])
        del ring, acts
        torch.cuda.empty_cache()
    # configs[4]: closed loop, 65536 envs in total
    n5 = 65536 // world
    cfg5 = scenarios.load("navigation").make_world(12, dtype="f32", episode_length=EPISODE_LEN)
    c5 = closed_loop_fused(cfg5, n5, max(EPISODE_LEN, args.config5_steps), local, rank, args.collect_streams,
                           actor_alone=False)
    times.append(c5["ms"])
    t = torch.tensor(times, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t = t.tolist()
    for row, ms in zip(rows, t):
        steps = row["regions"] * row["steps_per_launch"]
        row["step_us"] = ms * 1e3 / steps
        row["agent_steps_per_s"] = row["envs_per_gpu"] * row["n_agents"] * steps * world / (ms * 1e-3)
        row["achieved"] = row.pop("_bytes") * row["regions"] / (ms * 1e-3) / 1e9
        row["frac"] = row["achieved"] / peak
        row["region_ms"] = ms
    ms5 = t[-1]
    rows.append({"config": f"configs[4] navigation 12 agents, 65536 envs over {world} GPU(s) ({n5} per GPU), closed loop: "
                           "graph_actor_kernel + env step per step (gsm_collect, CUDA graph), reset per rollout",
                 "envs_per_gpu": n5, "n_agents": 12, "scaling": "strong", "steps": c5["steps"],
                 "step_us": ms5 * 1e3 / c5["steps"], "region_ms": ms5,
                 "agent_steps_per_s": n5 * 12 * c5["steps"] * world / (ms5 * 1e-3),
                 "bound": "actor kernel: fp32 issue (not HBM); env step: HBM write stream"})
    return rows


def closed_loop_fused(cfg, n_envs, n_steps, local, rank, n_streams=1, actor_alone=True):
    """Closed loop with THIS library's actor kernel (SURVEY.md §8 f3) and C-level collect loop (f1):
    gsm_collect = per env step one graph_actor_kernel launch (forward + Gumbel-max sampling +
    log-prob, weights in the kernel parameter space) and one env-step launch, written straight into
    a [T+1]/[T] rollout buffer (f2); the 2T launches are replayed from a CUDA graph; the env is
    reset between rollouts.  Same declared actor architecture as the torch policy above."""
    import torch
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv, StreamShardedEnv
    from gs_marl_b200.policy import GraphAttentionActor
    from gs_marl_b200.rollout import GraphRolloutBuffer, collect_fused
    dev = torch.device("cuda", local)
    env = (MultiAgentGraphConstrainEnv(cfg, n_envs, device=local, env_offset=rank * n_envs, seed=3)
           if n_streams <= 1 else
           StreamShardedEnv(cfg, n_envs, n_streams=n_streams, device=local, env_offset=rank * n_envs, seed=3))
    actor = GraphAttentionActor(len(cfg.discrete_u), seed=0)
    T = EPISODE_LEN
    buf = GraphRolloutBuffer(env, T)
    buf.reset_env()
    g = collect_fused(env, actor, buf, seed=1, first_step=0, graph=True, with_values=False)
    for _ in range(2):
        g.replay(); buf.reset_env()
    torch.cuda.synchronize()
    reps = max(1, n_steps // T)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
        buf.reset_env()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if not actor_alone:
        env.close()
        return {"ms": ms, "steps": reps * T}
    # the actor kernel alone on one slot of the buffer
    obs, graph = buf["obs"][1], buf.graph(1)
    out = (buf["actions"][0], buf["logp"][0])
    for _ in range(3):
        actor.act(obs, graph, seed=1, step=0, out=out)
    torch.cuda.synchronize()
    ga = torch.cuda.CUDAGraph()            # 50 launches per replay: device time, not Python time
    with torch.cuda.graph(ga):
        for q in range(50):
            actor.act(obs, graph, seed=1, step=q, out=out)
    ga.replay()
    torch.cuda.synchronize()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    for q in range(4):
        ga.replay()
    k1.record()
    torch.cuda.synchronize()
    actor_us = k0.elapsed_time(k1) * 1e3 / 200
    cnt = graph["nbr_cnt"].float()
    rows = float(cnt.sum().item())
    n_agents = cnt.numel()
    H, A = 64, len(cfg.discrete_u)
    flops = 2.0 * (n_agents * H * (6 + A) + rows * H * (6 + 1 + A))
    env.close()
    return {"value": n_envs * cfg.n_agents * reps * T / (ms * 1e-3), "unit": UNIT, "steps": reps * T,
            "ms": ms, "ms_per_step": ms / (reps * T),
            "policy": "graph_actor_kernel<5,0> (this library, fp32, weights as kernel parameters) via gsm_collect; "
                      f"CUDA graph of {2 * T} launches per {T}-step rollout per sub-shard ({max(1, n_streams)} "
                      "sub-shard(s), each its own actor -> env chain on its own stream) + reset per rollout",
            "actor_kernel_us": actor_us, "mean_valid_rows_per_agent": rows / n_agents,
            "actor_tflops": flops / (actor_us * 1e-6) / 1e12,
            "actor_bound": "fp32 issue / FMA pipe (packed FFMA2 with broadcast uniform-register weights); measured "
                           "FFMA peak on this GPU 72 TFLOP/s (profiles/fma_peak.cu; nominal 148 SM x 128 FMA/clk x 2 x "
                           "1.965 GHz = 74.5)"}


def closed_loop(env, cfg, n_steps, dev):
    """agent-steps/s with a random-init GS-MARL-style policy in the loop (not part of the hot
    path: SURVEY.md §8 f3 'next' row; here only as the consumer of the env outputs)."""
    import torch
    torch.manual_seed(0)
    H, K, n_act = 64, cfg.max_nbrs, len(cfg.discrete_u)
    ego = torch.nn.Sequential(torch.nn.Linear(6, H), torch.nn.ReLU()).to(dev)
    nbr = torch.nn.Sequential(torch.nn.Linear(6, H), torch.nn.ReLU()).to(dev)
    att = torch.nn.Linear(H, 1).to(dev)
    head = torch.nn.Linear(2 * H, n_act).to(dev)
    ar = torch.arange(K, device=dev)

    @torch.no_grad()
    def act(obs, graph):
        h = ego(obs)                                              # [B, N, H]
        m = nbr(graph["nbr_feat"])                                # [B, N, K, H]
        valid = ar[None, None, :] < graph["nbr_cnt"][..., None]   # padded rows masked out
        w = att(m).squeeze(-1).masked_fill(~valid, -1e9).softmax(-1)
        agg = (w[..., None] * m).sum(2) * valid.any(-1, keepdim=True)
        logits = head(torch.cat([h, agg], -1))
        g = -torch.log(-torch.log(torch.rand_like(logits).clamp_min(1e-9)))
        return (logits + g).argmax(-1).to(torch.int32)            # Gumbel-max sample

    obs, graph = env.reset()
    for _ in range(10):
        obs, graph, *_ = env.step(act(obs, graph))
    torch.cuda.synchronize()
    # one closed-loop iteration (policy forward + sampling + gsm_step) captured in a CUDA graph:
    # env.step reads/writes fixed buffers, so replaying the graph advances the rollout
    mode = "CUDA graph of one policy+env iteration"
    try:
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(3):
                env.step(act(obs, graph))
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            env.step(act(obs, graph))
        step = g.replay
    except Exception as e:                                # capture unsupported: eager fallback
        mode = f"eager ({type(e).__name__})"

        def step():
            env.step(act(obs, graph))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(n_steps):
        step()
        if (s + 1) % EPISODE_LEN == 0:
            env.reset()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return {"value": env.n_envs * cfg.n_agents * n_steps / (ms * 1e-3), "unit": UNIT, "steps": n_steps,
            "ms": ms, "ms_per_step": ms / n_steps,
            "policy": f"random-init graph-attention policy, hidden {H}, plain PyTorch (library kernels); {mode}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100000, help="env steps in the timed region")
    ap.add_argument("--warmup", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (rank 0's envs) as DIR/<name>.npy")
    ap.add_argument("--large-envs", type=int, default=1048576,
                    help="extra roofline line at a GPU-saturating env count (0 = skip)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="envs per GPU")
    ap.add_argument("--e2e-steps", type=int, default=200)
    ap.add_argument("--rollout-t", type=int, default=ROLLOUT_T, help="steps fused per launch")
    ap.add_argument("--streams", type=int, default=4,
                    help="env sub-shards per GPU, each on its own CUDA stream (1 = one handle, one stream)")
    ap.add_argument("--closed-loop-steps", type=int, default=1000)
    ap.add_argument("--collect-streams", type=int, default=1,
                    help="env sub-shards (streams) of the fused closed loop: one shard's actor overlaps another's env step")
    ap.add_argument("--region-ms", type=float, default=300.0,
                    help="minimum length of the side measurements (variants of the headline, large batch; "
                         "capped at 60 ms): their K-step regions are replayed until they last this long")
    ap.add_argument("--configs", type=int, default=1, help="1: add the BASELINE configs[2..4] block to the line")
    ap.add_argument("--config-ms", type=float, default=60.0, help="timed length per entry of the configs block")
    ap.add_argument("--config5-steps", type=int, default=100)
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--ref-budget", type=float, default=90.0, help="(ignored: the reference arm always runs the full workload)")
    ap.add_argument("--no-cpu", action="store_true")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the GPU arm's timed path")
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
