"""bench.py's reference arm runs on the host alone, so its JSON contract can be checked without a GPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["unit"] == "env-steps/s" and d["value"] > 0 and d["steps"] == 2 and d["warmup"] == 1
    assert d["metric"].startswith("env-steps/sec (CartPole-v1")
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["vs_baseline"] is None and "workload" in d["config"]


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--gpus", "2"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def _bench_module():
    sys.path.insert(0, ROOT)
    import importlib

    return importlib.import_module("bench")


def test_both_arms_emit_the_same_config_object():
    """The driver compares the two arms' `config`; it must not depend on which arm builds it."""
    b = _bench_module()
    for world in (1, 2, 8):
        cfg = b.bench_config(b.NUM_ENVS_PER_GPU, world)
        assert cfg["workload"].startswith("CartPole-v1, 16777216 envs per GPU") and cfg["mode"] == "step"
        assert cfg["parallelism"].startswith(f"dp{world} ")
        assert "model" not in cfg  # no ML vocabulary in the workload description
    assert b.STEP_CONTRACT == [42, 22, 25, 37, 66] and b.ROLLOUT_CONTRACT == [22, 14, 17, 21, 30]  # SURVEY 8(d)
    assert sum(b.MIXED_PER_GPU) == 1 << 24  # configs[4]: 2^24 envs per GPU, 2^27 on 8


def test_clock_records_are_cut_from_one_sampler_by_wall_clock_window():
    b = _bench_module()
    s = b.ClockSampler(0)
    s.proc = object()  # pretend nvidia-smi is running; only the parsed lines matter here
    row = "0, {sm}, 1965, {w}, 0x0000000000000004, Not Active, Not Active, Not Active, {cap}"
    s.lines = [(100.00, row.format(sm=1965, w=300.0, cap="Not Active")),
               (100.05, row.format(sm=1800, w=990.0, cap="Active")),
               (100.10, row.format(sm=1700, w=995.0, cap="Active")),
               (100.60, row.format(sm=1965, w=200.0, cap="Not Active"))]
    rec = s.window(100.04, 100.11)
    assert rec["samples"] == 2 and rec["sm_mhz"] == 1750.0 and rec["reasons"] == ["sw_power_cap"]
    assert rec["sm_max_mhz"] == 1965.0 and rec["power_w_max"] == 995.0
    quiet = s.window(100.55, 100.65)
    assert quiet["samples"] == 1 and quiet["reasons"] == []
    short = s.window(100.30, 100.301)  # shorter than the sampling period: the nearest sample, and it says so
    assert short["samples"] == 1 and "nearest" in short["note"]


def test_dump_outputs_writes_a_fixed_sample_of_the_last_step(tmp_path):
    """--dump-outputs: what env.step returned, as float32/float64 .npy files under 64 MB, the same sample every run."""
    import numpy as np

    torch = __import__("pytest").importorskip("torch")
    from modurl_gym_b200.vec_env import StepInfo

    b = _bench_module()
    n, base = 3 * b.DUMP_MAX_ENVS + 5, 7 << 24
    gen = torch.Generator().manual_seed(1)
    obs, reward = torch.rand((4, n), generator=gen), torch.rand(n, generator=gen)
    flags = torch.randint(0, 4, (n,), dtype=torch.uint8, generator=gen)
    for d in ("a", "b"):
        b.dump_step_outputs(torch, StepInfo(obs, reward, flags), n, base, str(tmp_path / d))
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["env_index.npy", "obs.npy", "reward.npy", "terminated.npy", "truncated.npy"]
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        assert np.array_equal(got[f[:-4]], np.load(tmp_path / "b" / f))
        assert got[f[:-4]].dtype in (np.float32, np.float64)
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    idx = got["env_index"].astype(np.int64) - base
    assert len(idx) == b.DUMP_MAX_ENVS and np.all(np.diff(idx) > 0) and idx[-1] < n
    assert np.array_equal(got["obs"], obs.numpy()[:, idx]) and np.array_equal(got["reward"], reward.numpy()[idx])
    assert np.array_equal(got["terminated"], (flags.numpy()[idx] & 1).astype(np.float32))
    assert np.array_equal(got["truncated"], (flags.numpy()[idx] >> 1 & 1).astype(np.float32))
    small = tmp_path / "small"
    b.dump_step_outputs(torch, StepInfo(obs[:, :10], reward[:10], flags[:10]), 10, 0, str(small))
    assert np.array_equal(np.load(small / "env_index.npy"), np.arange(10.0))


def test_statistics_comparison_tolerates_only_the_float_sum():
    torch = __import__("pytest").importorskip("torch")
    b = _bench_module()
    want = torch.tensor([[10.0, 4.0, 6.0, 220.0, -453532899750.8663], [3.0, 3.0, 0.0, 60.0, 60.0]], dtype=torch.float64)
    got = want.clone()
    got[0, 4] = -453532899750.8662  # a different summation order inside NCCL
    assert b.same_statistics(torch, got, want)
    got[1, 0] = 4.0  # a count must match exactly
    assert not b.same_statistics(torch, got, want)
    got = want.clone()
    got[0, 4] *= 1.0 + 1e-9
    assert not b.same_statistics(torch, got, want)
