"""bench.py's output contract: the CPU reference arm runs here end to end; the GPU arm's line
is checked on the B200 box."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
             "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def _run(args, timeout):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True,
                         text=True, timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines                      # exactly one JSON line on stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "2", "--warmup", "1", "--envs", "256"], 300)
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    assert d["unit"] == "agent-steps/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert "withheld" in d["cpu_baseline"]["sample"]   # never presented as GS-MARL's own env
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0 and "unpinned" in d["config"]["spec_status"]
    # the reference arm never shrinks its workload: exactly the envs it was asked for, and the same
    # `config` object the GPU arm prints for the same command line
    assert d["config"]["envs_per_gpu"] == 256 and d["cpu_baseline"]["sample_envs_per_step"] == 256
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config(1, 256)


@pytest.mark.gpu
def test_gpu_arm_line():
    d = _run(["--steps", "60", "--warmup", "5", "--e2e-steps", "10", "--closed-loop-steps", "25",
              "--large-envs", "65536", "--cpu-budget", "2", "--region-ms", "100", "--config-ms", "20",
              "--config5-steps", "25"], 900)
    assert BASE_KEYS | {"clocks", "roofline", "repeats", "configs", "method"} <= set(d)
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config(1)       # same object as the reference arm's
    # the timed region: exactly --steps env steps (one K-step region replayed from a CUDA graph: per
    # shard stream, fused launches of 25 + 25 + 10 steps), and value / ms_per_step / roofline all
    # derived from that one region
    assert d["steps"] == 60 and d["repeats"] == 1 and d["timed_region_ms"] > 0
    assert d["gpu_launches"] == d["method"]["streams"] * 3
    assert abs(d["ms_per_step"] - d["timed_region_ms"] / (d["repeats"] * d["steps"])) < 1e-9
    assert abs(d["value"] - 16384 * 3 / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-6
    r = d["roofline"]
    assert abs(r["step_us"] - d["ms_per_step"] * 1e3) < 1e-6
    assert abs(r["achieved"] - r["algorithmic_bytes_per_agent_step"] * d["value"] / 1e9) / r["achieved"] < 1e-6
    assert r["frac"] < r["frac_per_step_accounting"]      # state / landmarks / counter charged once per launch
    # (a cold nvidia-smi can deliver its first sample after a 100 ms region: the sampler then reports the
    # warm-up + region window and says so)
    assert d["clocks"]["window"].endswith("timed region") or "timed region" in d["clocks"]["window"]
    assert d["clocks"]["samples"] >= 1
    labels = [c["config"] for c in d["configs"]]
    assert sum(l.startswith("configs[2]") for l in labels) == 3 and sum(l.startswith("configs[3]") for l in labels) == 4
    assert sum(l.startswith("configs[4]") for l in labels) == 1
    for c in d["configs"]:
        assert c["step_us"] > 0 and c["agent_steps_per_s"] > 0
        if not c["config"].startswith("configs[4]"):
            assert 0.02 < c["frac"] < 1.2 and c["bytes_per_agent_step"] > 0
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert 0.05 < r["frac"] < 1.2 and r["traffic"] is None or r["traffic"] > 0
    assert d["gpu_launches"] > 0 and d["e2e"]["d2h_bytes_per_step_dense"] == 13221888 and 0 < d["e2e"]["d2h_bytes_per_step"] < 13221888
    assert d["e2e"]["value"] < d["value"]              # the host path cannot beat the device path
    assert d["cpu_baseline"]["kind"] == "port" and d["dtype"] == "f32" and d["scaling"] == "weak"
    assert d["config"]["workload"].startswith("cooperative navigation, 3 agents, 16384 envs")
    e = d["e2e"]
    assert 0 < e["d2h_gbs_achieved"] < e["d2h_gbs_ceiling"] * 1.25      # about or below the measured pinned-copy rate (10 steps: noisy)
    f = d["closed_loop"]["fused_actor"]
    assert f["value"] > d["closed_loop"]["value"] and f["actor_kernel_us"] > 0


def test_dump_outputs_format_and_seeded_sample(tmp_path):
    """bench.dump_outputs: one .npy per output, float32 / float64 only, integer outputs exact (adj as
    unsigned bit masks); above the byte limit every file holds the same seeded sample of env rows."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(1)
    n = 1000
    outs = {"obs": rng.standard_normal((n, 3, 6)).astype(np.float32),
            "nbr_idx": rng.integers(-1, 9, (n, 3, 8)).astype(np.int32),
            "adj": rng.integers(0, 2 ** 32, (n, 3, 1), dtype=np.uint32).view(np.int32),
            "reward": rng.standard_normal((n, 3)),
            "done": rng.integers(0, 2, (n, 3)).astype(np.uint8)}

    def load(d):
        return {p.stem: np.load(p) for p in sorted(d.iterdir())}
    bench.dump_outputs(outs, str(tmp_path / "full"))
    full = load(tmp_path / "full")
    assert set(full) == set(outs)
    assert full["obs"].dtype == np.float32 and full["reward"].dtype == np.float64
    for k in ("nbr_idx", "adj", "done"):
        assert full[k].dtype == np.float64
    assert (full["adj"] == outs["adj"].view(np.uint32)).all() and full["adj"].max() >= 2 ** 31
    for k in ("obs", "nbr_idx", "reward", "done"):
        assert (full[k] == outs[k]).all(), k

    limit = 100_000
    for d in ("a", "b"):
        bench.dump_outputs(outs, str(tmp_path / d), limit=limit)
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    assert set(a) == set(outs) | {"env_index"}
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= limit
    idx = a["env_index"].astype(np.int64)
    assert 0 < len(idx) < n and (np.diff(idx) > 0).all()
    for k in a:
        assert np.array_equal(a[k], b[k]), k                       # fixed seed: the same sample
        if k != "env_index":
            assert np.array_equal(a[k], full[k][idx]), k


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--dump-outputs of a run with K = 30 timed steps after W = 270 warm-up steps equals step 300 from the
    reset state recomputed on one env handle (the bench drives 4 sub-shard handles): the pre-run before the
    warm-up does not leak into the timed steps, and --steps sets how many there are."""
    import numpy as np
    import torch
    d = _run(["--steps", "30", "--warmup", "270", "--envs", "2048", "--no-cpu", "--configs", "0",
              "--closed-loop-steps", "0", "--large-envs", "0", "--e2e-steps", "10", "--region-ms", "5",
              "--dump-outputs", str(tmp_path / "dump")], 600)
    assert d["steps"] == 30 and d["repeats"] == 1 and d["gpu_launches"] == 2 * d["method"]["streams"]
    sys.path.insert(0, ROOT)
    import bench
    from gs_marl_b200 import scenarios
    from gs_marl_b200.environment import MultiAgentGraphConstrainEnv
    got = {p.stem: np.load(p) for p in (tmp_path / "dump").iterdir()}
    assert set(got) == set(MultiAgentGraphConstrainEnv.OUTPUTS)
    cfg = scenarios.load("navigation").make_world(3, dtype="f32", episode_length=bench.EPISODE_LEN)
    env = MultiAgentGraphConstrainEnv(cfg, 2048, seed=1)
    env.reset()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(0)
    acts = torch.randint(0, 5, (25, 2048, 3), generator=gen, device="cuda", dtype=torch.int32)
    for _ in range(10):                          # 9 warm-up + 1 timed replay: launches of 25 + 5 steps
        env.rollout(acts[:25], auto_reset=True)
        out = env.rollout(acts[:5], auto_reset=True)
    want = {k: v[4].cpu().numpy() for k, v in out.items() if k != "actions"}
    want["adj"] = want["adj"].view(np.uint32)
    env.close()
    assert want["done"].all()                    # step 300: the 12th episode end
    for k, w in want.items():
        assert got[k].dtype == (np.float32 if w.dtype == np.float32 else np.float64), k
        assert np.array_equal(got[k], w), k
