#!/usr/bin/env python
"""bench.py -- env-steps/sec of the classic-control hot path on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline (`value`, `roofline`, `e2e`): a "step" is ONE mgym_step launch over 2^24 CartPole-v1 envs per GPU with
device-side auto-reset (BASELINE.json configs[1]).  Envs shard over ranks as independent contiguous slices (no
data-path collective; "scaling": "weak").

`configs` (same JSON line): the other BASELINE.json configurations, each timed on the device with its own
nvidia-smi clock record -- CartPole / MountainCar / MountainCarContinuous fused rollouts at 2^24 envs
(configs[2]: 1000 steps as 32-step chunks over one reused trajectory ring), Pendulum and Acrobot per-call steps
and rollouts at 2^22 envs (configs[3]), and the mixed suite with its statistics all-reduce (configs[4]: 2^24
envs per GPU = 2^27 on 8 GPUs).  Fractions are quoted against the SURVEY 8(d) contract bytes.

At N > 1 the statistics all-reduce also runs through the C ABI's own NCCL entry point (mgym_stats_allreduce on a
raw ncclComm_t) and is checked against torch.distributed's result ("native_nccl_allreduce").

--impl reference times the CPU restatement of the reference's step loop (oracle/, a C port: the Rust crate
cannot be built in this image) on the host cores; one "step" there is the same 2^24 env-steps.
"""
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

METRIC = "env-steps/sec (CartPole-v1, 2^24 envs)"
UNIT = "env-steps/s"
KIND_NAME = "CartPole-v1"
NUM_ENVS_PER_GPU = 1 << 24
# Algorithmic bytes per env-step of the per-call step kernel (DESIGN.md section 4, SURVEY 8(d)):
# state read 16 + state/obs write 16 + action u8 1 + reward f32 4 + flags u8 1 + u16 counter 2+2
BYTES_PER_ENV_STEP = 42
BYTES_SEPARATE_OBS = 58  # the same step when the caller asks for a separate observation buffer (BASELINE.md 3)

NAMES = ["CartPole-v1", "MountainCar-v0", "MountainCarContinuous-v0", "Pendulum-v1", "Acrobot-v1"]
OBS_DIM = [4, 2, 2, 3, 6]
OBS_BYTES = [16, 8, 8, 12, 24]
ACT_BYTES = [1, 1, 4, 4, 1]
# SURVEY 8(d) / BASELINE.md 3 contract bytes per env-step, per-call step (obs aliases the state rows where the
# observation IS the state).  MountainCarContinuous has no row there: 8 + 8 state, f32 action, reward, flags.
STEP_CONTRACT = [42, 22, 25, 37, 66]
# fused rollout: observation + reward + flags written, action read (state/counters amortised over K)
ROLLOUT_CONTRACT = [OBS_BYTES[k] + 4 + 1 + ACT_BYTES[k] for k in range(5)]  # 22, 14, 17, 21, 30
ROLLOUT_CHUNK = 32  # steps per fused launch = depth of the reused trajectory ring

# name, kind, envs per GPU, mode, steps per pass, BASELINE.json configs[] index
SUBCONFIGS = [
    ("cartpole_step_separate_obs", 0, 1 << 24, "step_obs", 1, 1),
    ("cartpole_rollout", 0, 1 << 24, "rollout", ROLLOUT_CHUNK, 1),
    ("mountain_car_step", 1, 1 << 24, "step", 1, 2),
    ("mountain_car_rollout_1000", 1, 1 << 24, "rollout", 1000, 2),
    ("mountain_car_continuous_step", 2, 1 << 24, "step", 1, 2),
    ("mountain_car_continuous_rollout_1000", 2, 1 << 24, "rollout", 1000, 2),
    ("pendulum_step", 3, 1 << 22, "step", 1, 3),
    ("pendulum_rollout", 3, 1 << 22, "rollout", 200, 3),
    ("acrobot_step", 4, 1 << 22, "step", 1, 3),
    ("acrobot_rollout", 4, 1 << 22, "rollout", 128, 3),
]
MIXED_PER_GPU = [1 << 22, 1 << 22, 1 << 22, 1 << 21, 1 << 21]  # 2^24 envs per GPU in total


def workload_name(n):
    return (f"{KIND_NAME}, {n} envs per GPU, per-call step kernel with device-side auto-reset "
            "(BASELINE.json configs[1])")


def bench_config(n, world):
    """The `config` object of the JSON line -- the SAME for both arms (the driver compares them)."""
    return {
        "workload": workload_name(n),
        "num_envs_per_gpu": n, "mode": "step",
        "obs": "zero-copy (obs aliases the resident state rows)",
        "actions": "uniform random {0,1}, pre-generated (rotating pool of 16 uint8[N] buffers on the GPU arm)",
        "l2": f"working set {BYTES_PER_ENV_STEP * n / 1e6:.0f} MB per step > 126 MB L2 (inputs larger than L2)",
        "parallelism": f"dp{world} (independent env slices, no data-path collective)",
    }


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", choices=["native", "reference"], default="native")
    ap.add_argument("--num-envs", type=int, default=NUM_ENVS_PER_GPU, help="envs per GPU")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-configs", action="store_true", help="skip the configs[2..4] legs (headline only)")
    ap.add_argument("--only-configs", default="", help="comma-separated sub-config names (default: all)")
    ap.add_argument("--config-seconds", type=float, default=0.2, help="one timed window of a sub-config (3 are taken)")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink every sub-config (smoke runs on small GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (rank 0's envs, a fixed "
                         "sample of at most 2^20 of them) as DIR/<name>.npy, so that two builds can be compared")
    args = ap.parse_args()
    if args.dump_outputs is not None and args.impl != "native":
        ap.error("--dump-outputs needs --impl native: the reference arm returns no arrays")
    return args


# -------------------------------------------------------------------------------------------------
# clocks: nvidia-smi sampled DURING the timed regions (B200_PROFILING.md recipe).  ONE sampler process per
# run; every timed region reads the samples that fall inside its own wall-clock window.
# -------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index):
        self.gpu_index, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", os.environ.get("MGYM_SMI_MS", "50")], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def wait_first_sample(self, timeout=3.0):
        t_end = time.time() + timeout
        while self.proc is not None and not self.lines and time.time() < t_end:
            time.sleep(0.02)

    def window(self, t0, t1):
        """Clock record of the wall-clock window [t0, t1] (a little slack either side: nvidia-smi stamps late)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        inside = [l for (ts, l) in list(self.lines) if t0 - 0.03 <= ts <= t1 + 0.12]
        nearest = False
        if not inside and self.lines:  # a region shorter than the sampling period: the sample nearest to it
            mid = 0.5 * (t0 + t1)
            inside = [min(list(self.lines), key=lambda x: abs(x[0] - mid))[1]]
            nearest = True
        sm, sm_max, reasons, power = [], [], set(), []
        for l in inside:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                sm_max.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(self.NAMES, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        rec = {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(sm_max) if sm_max else None,
               "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}
        if nearest:
            rec["note"] = "region shorter than the sampling period: nearest sample"
        return rec

    def stop(self):
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()


def ncu_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu captures (profiles/traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)[key]
        return t["dram_bytes_read"] + t["dram_bytes_write"], t["source"]
    except Exception:
        return None, None


def bind_to_gpu_numa_node(gpu_index):
    """Pin this rank to the CPUs next to its GPU (NVML's ideal affinity) so that the pinned host buffers of the
    end-to-end leg are allocated on the local NUMA node; matters when 8 ranks stream over PCIe at once."""
    try:
        import pynvml

        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1]
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"{len(allowed)} cpus ({allowed[0]}-{allowed[-1]})"
    except Exception as e:  # affinity is an optimisation only
        return f"unbound ({type(e).__name__})"
    return "unbound"


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# -------------------------------------------------------------------------------------------------
# CPU arm: the oracle's scalar step loop, one env loop per thread
# -------------------------------------------------------------------------------------------------
def cpu_step_loop(seconds, threads):
    """Runs the reference's caller loop (cartpole.rs:460-471, restated in oracle/mgym_oracle.c) for
    about `seconds` on `threads` host threads; returns (env_steps_per_sec, total_steps, wall)."""
    from oracle import oracle as o

    total, wall, _ = o.baseline_loop(o.CARTPOLE, 1_000_000, threads, seed=0x5EED)  # calibrate
    rate = total / max(wall, 1e-9)
    per_thread = max(1_000_000, int(rate * seconds / threads))
    total, wall, _ = o.baseline_loop(o.CARTPOLE, per_thread, threads, seed=0x5EED)
    return total / wall, total, wall


def run_reference(args, rank):
    """--impl reference: one 'step' is the same 2^24 env-steps as a step of the GPU arm, executed by the reference's
    own loop shape -- each host thread advances its own CartPole env with random actions and reset-on-done
    (cartpole.rs:460-471), threads x (num_envs / threads) env-steps per step."""
    if rank != 0:
        return
    from oracle import oracle as o

    threads = os.cpu_count() or 1
    # one 'step' = the env-steps of one step of the GPU arm at this N (num_envs per GPU x GPUs), unless K of those
    # would not end within about three minutes on these cores: then each step is a bounded sample of it
    want = args.num_envs * max(args.gpus, 1)
    total, wall, _ = o.baseline_loop(o.CARTPOLE, 1 << 18, threads, seed=0x5EED)  # calibrate (~10 ms)
    rate = total / max(wall, 1e-9)
    budget = int(rate * 180.0 / max(args.steps + args.warmup, 1))
    per_step = max(threads, min(want, budget))
    per_thread = max(1, per_step // threads)
    for _ in range(args.warmup):
        o.baseline_loop(o.CARTPOLE, per_thread, threads, seed=0x5EED)
    t0 = time.perf_counter()
    total = 0
    for _ in range(args.steps):
        n, _, _ = o.baseline_loop(o.CARTPOLE, per_thread, threads, seed=0x5EED)
        total += n
    wall = time.perf_counter() - t0
    value = total / wall
    sample = (f"each step = {threads} threads x {per_thread} CartPole-v1 env-steps = {threads * per_thread} env-steps "
              f"({'the same as' if threads * per_thread >= want - threads else 'a bounded sample of'} one {want}-env-step "
              f"step of the GPU arm; one env loop per thread, random actions, reset on done): the oracle C port of cartpole.rs:251-348, "
              f"an upper bound on the Rust crate, which cannot be built here (no cargo/rustc) and also allocates 3 "
              f"tensors per step")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args.num_envs, max(args.gpus, 1)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------------------
# native arm helpers
# -------------------------------------------------------------------------------------------------
class Ctx:
    """Per-process bench context: device, ranks, the clock sampler, barrier and max-over-ranks timing."""

    def __init__(self, torch, dist, device, rank, local_rank, world, sampler):
        self.torch, self.dist, self.device = torch, dist, device
        self.rank, self.local_rank, self.world, self.sampler = rank, local_rank, world, sampler

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        from modurl_gym_b200.distributed import max_over_ranks

        return max_over_ranks(v, self.device)

    def timed(self, fn, reps):
        """reps calls of fn between a barrier + synchronize on both sides, timed with CUDA events on the launching
        stream; returns (seconds, max over ranks; clock record of the region on rank 0)."""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        self.barrier()
        w1 = time.time()
        sec = self.max_over_ranks(e0.elapsed_time(e1) * 1e-3)
        clocks = self.sampler.window(w0, w1) if (self.rank == 0 and self.sampler) else None
        return sec, clocks

    def calibrated(self, fn, seconds, windows=3, idle=0.25, min_reps=2, max_reps=100000, counter=None):
        """warm-up (>= 3 calls), then `windows` timed regions of about `seconds` each with `idle` seconds of rest
        before each (the chip's power governor clocks a hot kernel down within milliseconds, and how far depends on
        what ran just before: every window starts from the same rested state).  Returns the BEST window (time, reps,
        its own clock record) and the per-window times -- the same best-of-N convention as MEASURED_PEAKS.json."""
        torch = self.torch
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        one = self.max_over_ranks(max(e0.elapsed_time(e1) * 1e-3, 1e-6))
        reps = int(min(max_reps, max(min_reps, round(seconds / one))))
        best, all_sec = None, []
        self.timed_launches = 0  # kernel launches inside the timed windows (`counter[0]` counts the caller's launches)
        for _ in range(windows):
            time.sleep(idle)
            fn()  # one untimed call: the first launch after an idle gap pays the clock ramp
            before = counter[0] if counter else 0
            sec, clocks = self.timed(fn, reps)
            self.timed_launches += (counter[0] - before) if counter else 0
            all_sec.append(sec)
            if best is None or sec < best[0]:
                best = (sec, clocks)
        return best[0], reps, best[1], all_sec


def same_statistics(torch, got, want):
    """Two all-reduces of the statistics agree: the four counts exactly; the return sum -- a float64 sum that two
    NCCL calls of different sizes may reduce in different orders (ring vs tree) -- to 1e-12 relative."""
    got, want = got.reshape(-1, 5), want.reshape(-1, 5)
    if not bool(torch.equal(got[:, :4], want[:, :4])):
        return False
    scale = torch.clamp(want[:, 4].abs(), min=1.0)
    return bool(((got[:, 4] - want[:, 4]).abs() <= 1e-12 * scale).all())


def make_actions(torch, env, kind, shape, device, gen):
    if env.continuous:
        lim = 1.0 if kind == 2 else 2.0
        return (torch.rand(shape, device=device, generator=gen) * 2 - 1) * lim
    return torch.randint(0, env.action_space().n, shape, dtype=torch.uint8, device=device, generator=gen)


def run_subconfig(ctx, m, spec, args, peak):
    """One of the BASELINE configs[1..3] legs: env-steps/s with everything resident, against its contract bytes."""
    torch = ctx.torch
    name, kind, n, mode, steps_per_pass, cfg_index = spec
    n = max(1024, int(n * args.scale) // 1024 * 1024)
    dev = ctx.device
    env = m.GpuVecEnv(kind, n, device=ctx.local_rank, seed=0x5EED, env_index_base=ctx.rank * n)
    env.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(100 + kind + 17 * ctx.rank)
    od = OBS_DIM[kind]
    zero_copy = env.obs_is_state and mode != "step_obs"
    launches = [0]
    if mode in ("step", "step_obs"):
        pool = make_actions(torch, env, kind, (16, n), dev, gen)
        reward = torch.empty(n, device=dev)
        flags = torch.empty(n, dtype=torch.uint8, device=dev)
        obs = None if zero_copy else torch.empty((od, n), device=dev)
        i = [0]

        def one_pass():
            env.step_raw(pool[i[0] & 15], obs, reward, flags)
            i[0] += 1
            launches[0] += 1

        contract = BYTES_SEPARATE_OBS if mode == "step_obs" else STEP_CONTRACT[kind]
        what = "per-call step" + (" writing a separate observation buffer" if mode == "step_obs" else "")
    else:
        K = ROLLOUT_CHUNK
        acts = make_actions(torch, env, kind, (K, n), dev, gen)  # one ring of actions, reused by every chunk
        obs = torch.empty((K, od, n), device=dev)
        reward = torch.empty((K, n), device=dev)
        flags = torch.empty((K, n), dtype=torch.uint8, device=dev)

        def one_pass():
            done = 0
            while done < steps_per_pass:
                k = min(K, steps_per_pass - done)
                env.rollout(k, acts[:k], obs=obs[:k], reward=reward[:k], flags=flags[:k], count_done=False)
                done += k
                launches[0] += 1

        contract = ROLLOUT_CONTRACT[kind]
        what = (f"fused rollout, {steps_per_pass} steps per pass as {K}-step launches over one reused "
                f"[{K}][..][N] trajectory ring, actions read from a [{K}][N] ring")
    sec, reps, clocks, windows = ctx.calibrated(one_pass, args.config_seconds, counter=launches)
    env_steps = float(n) * ctx.world * steps_per_pass * reps
    rate = env_steps / sec
    per_gpu_gbs = contract * (rate / ctx.world) / 1e9
    stats = env.stats()
    out = {
        "baseline_config": cfg_index, "kind": NAMES[kind], "num_envs_per_gpu": n, "mode": what,
        "steps_per_pass": steps_per_pass, "passes": reps, "ms_per_pass": 1e3 * sec / reps,
        "ms_per_env_step_batch": 1e3 * sec / (reps * steps_per_pass),
        "env_steps_per_s": rate, "bytes_per_env_step_contract": contract,
        "achieved_GBps_per_gpu": per_gpu_gbs, "peak_GBps": peak, "frac": per_gpu_gbs / peak,
        "mean_episode_length": stats.length_sum / max(stats.episodes, 1), "clocks": clocks,
        "window_ms_per_pass": [1e3 * w / reps for w in windows], "timing": "best of the windows listed",
    }
    env.close()
    del env
    torch.cuda.empty_cache()
    return out, ctx.timed_launches


def run_mixed_suite(ctx, m, args, native_comm):
    """BASELINE configs[4]: every GPU hosts an equal slice of every kind (2^24 envs per GPU, 2^27 on 8 GPUs), steps them
    with fused rollouts and the device-side random policy; the per-kind episode statistics are summed over ranks
    with ONE all-reduce of a 5 x 5 double matrix (torch.distributed/NCCL) and, per kind, through the C ABI's own
    NCCL entry point mgym_stats_allreduce on a raw ncclComm_t; both must agree."""
    torch, dist = ctx.torch, ctx.dist
    dev = ctx.device
    K = 16
    envs, bufs = [], []
    for kind, n in enumerate(MIXED_PER_GPU):
        n = max(1024, int(n * args.scale) // 1024 * 1024)
        env = m.GpuVecEnv(kind, n, device=ctx.local_rank, seed=0x5EED, env_index_base=ctx.rank * n, track_returns=True)
        env.reset()
        envs.append(env)
        bufs.append((torch.empty((K, env.obs_dim, n), device=dev), torch.empty((K, n), device=dev),
                     torch.empty((K, n), dtype=torch.uint8, device=dev)))
    count = [0]

    def sweep():
        for env, (o, r, f) in zip(envs, bufs):
            env.rollout(K, None, obs=o, reward=r, flags=f, count_done=False)
            count[0] += 1

    sec, reps, clocks, windows = ctx.calibrated(sweep, args.config_seconds, counter=count)
    launches = ctx.timed_launches
    steps = K * reps
    # the collective (off the per-step path): one all-reduce of the 5 x 5 statistics matrix
    mat = torch.stack([env.stats_tensor() for env in envs])
    local = mat.clone()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    e0.record()
    if ctx.world > 1:
        dist.all_reduce(mat, op=dist.ReduceOp.SUM)
    e1.record()
    torch.cuda.synchronize()
    allreduce_ms = e0.elapsed_time(e1)
    native = "not run (single rank: no communicator)"
    if native_comm is not None:
        got = torch.stack([env.all_reduce_stats_native(native_comm) for env in envs])
        torch.cuda.synchronize()
        native = "ok" if same_statistics(torch, got, mat) else f"MISMATCH: native {got.tolist()} vs torch {mat.tolist()}"
    rows = {}
    total_envs = 0
    for kind, env in enumerate(envs):
        ep, term, trunc, length, ret = mat[kind].tolist()
        total_envs += env.num_envs * ctx.world
        rows[NAMES[kind]] = {"envs_total": env.num_envs * ctx.world, "episodes": int(ep), "terminated": int(term),
                             "truncated": int(trunc), "mean_length": length / max(ep, 1), "mean_return": ret / max(ep, 1),
                             "episodes_this_rank": int(local[kind][0].item())}
    out = {
        "baseline_config": 4, "mode": "fused rollouts (16-step launches), device-side random policy (Space::sample)",
        "n_gpus": ctx.world, "envs_total": total_envs, "envs_per_gpu": total_envs // ctx.world,
        "steps_per_env": steps, "suite_env_steps_per_s": total_envs * steps / sec, "ms_per_sweep": 1e3 * sec / reps,
        "per_kind": rows,
        "collective": "one all-reduce (sum) of a 5x5 float64 statistics matrix after the timed region",
        "allreduce_ms": allreduce_ms, "native_nccl_allreduce": native, "clocks": clocks,
        "window_ms_per_sweep": [1e3 * w / reps for w in windows], "timing": "best of the windows listed",
    }
    for env in envs:
        env.close()
    del envs, bufs
    torch.cuda.empty_cache()
    return out, launches


DUMP_MAX_ENVS = 1 << 20  # 16 + 4 + 4 + 4 + 8 bytes per sampled env: 36 MB at most
DUMP_SAMPLE_SEED = 0x5EED


def dump_step_outputs(torch, info, n, env_index_base, out_dir):
    """The StepInfo a caller of env.step received from the last timed step -- observation, reward, terminated,
    truncated -- for a fixed, seeded sample of the envs (every env when n <= DUMP_MAX_ENVS), as float32 .npy files,
    plus the global index of each sampled env (float64, exact below 2^53)."""
    import numpy as np

    if n <= DUMP_MAX_ENVS:
        idx = np.arange(n, dtype=np.int64)
    else:
        idx = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(n, DUMP_MAX_ENVS, replace=False))
    sel = torch.from_numpy(idx).to(info.reward.device)
    obs, reward, done, truncated = info
    arrays = {
        "obs": obs.index_select(1, sel).cpu().numpy(),
        "reward": reward.index_select(0, sel).cpu().numpy(),
        "terminated": done.index_select(0, sel).to(torch.float32).cpu().numpy(),
        "truncated": truncated.index_select(0, sel).to(torch.float32).cpu().numpy(),
        "env_index": (idx + env_index_base).astype(np.float64),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def measure_host_link(ctx, nbytes=256 << 20, reps=4):
    """Pinned-memory copy ceilings of THIS box, all ranks copying at once: D2H alone, H2D alone, and both directions
    concurrently on two streams.  GB/s per GPU (max-over-ranks time) and aggregated over the ranks."""
    torch = ctx.torch
    dev = ctx.device
    d_a = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_b = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    h_in = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def run(d2h, h2d):
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        s1.wait_event(e0)
        s2.wait_event(e0)
        for _ in range(reps):
            if d2h:
                with torch.cuda.stream(s1):
                    h_out.copy_(d_a, non_blocking=True)
            if h2d:
                with torch.cuda.stream(s2):
                    d_b.copy_(h_in, non_blocking=True)
        torch.cuda.current_stream().wait_stream(s1)
        torch.cuda.current_stream().wait_stream(s2)
        e1.record()
        ctx.barrier()
        return ctx.max_over_ranks(e0.elapsed_time(e1) * 1e-3)

    run(True, True)  # warm-up
    t_d2h = min(run(True, False) for _ in range(3))
    t_h2d = min(run(False, True) for _ in range(3))
    t_both = min(run(True, True) for _ in range(3))
    gb = nbytes * reps / 1e9
    out = {"d2h_GBps_per_gpu": gb / t_d2h, "h2d_GBps_per_gpu": gb / t_h2d,
           "duplex_d2h_GBps_per_gpu": gb / t_both, "duplex_total_GBps_per_gpu": 2 * gb / t_both,
           "aggregate_d2h_GBps": ctx.world * gb / t_d2h, "ranks_copying_at_once": ctx.world,
           "how": f"{reps} x {nbytes >> 20} MiB cudaMemcpyAsync per direction between pinned host memory and HBM, "
                  f"all ranks at once, CUDA events, max over ranks, best of 3"}
    del d_a, d_b, h_in, h_out
    return out


# -------------------------------------------------------------------------------------------------
# native arm
# -------------------------------------------------------------------------------------------------
def run_native(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    import modurl_gym_b200 as m

    assert torch.cuda.is_available(), "bench.py needs a CUDA device; there is no CPU fallback"
    m.load_library()
    numa = bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1 and not dist.is_initialized():
        # NCCL prints its version banner (and, with NCCL_DEBUG=INFO, its topology log) on stdout when the
        # communicator comes up; stdout is reserved for the ONE JSON line, so fd 1 points at stderr meanwhile.
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()  # eager communicator creation
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    from modurl_gym_b200.distributed import NativeNcclComm, shard_range

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        sampler.wait_first_sample()
    ctx = Ctx(torch, dist, device, rank, local_rank, world, sampler)

    n = args.num_envs  # weak scaling: a fixed slice per GPU
    begin, end = shard_range(n * world, rank, world)
    assert end - begin == n
    env = m.GpuVecEnv(KIND_NAME, n, device=local_rank, seed=0x5EED, env_index_base=begin)
    env.reset()
    # rotating pool of pre-generated random actions keeps RNG out of the timed kernel (SURVEY 8(d))
    gen = torch.Generator(device=device)
    gen.manual_seed(1234 + rank)
    pool = [torch.randint(0, 2, (n,), dtype=torch.uint8, device=device, generator=gen) for _ in range(16)]
    step_i = [0]
    last = [None]

    def one_step():
        # the public call: Gym::step.  For CartPole the returned observation is a view of the resident state rows
        # (obs_out = NULL in the C call), reward and flags go to the env's own buffers.
        last[0] = env.step(pool[step_i[0] & 15])
        step_i[0] += 1

    warmup = max(args.warmup, 3)
    for _ in range(warmup):
        one_step()
    env.reset_stats()
    ms_max, clocks = ctx.timed(one_step, args.steps)
    ms_max *= 1e3
    gpu_launches = args.steps
    if args.dump_outputs is not None and rank == 0:
        # before anything else runs on this env: the returned tensors are views of buffers the next step overwrites
        dump_step_outputs(torch, last[0], n, begin, args.dump_outputs)

    # the statistics collective: torch.distributed (NCCL) and, at N > 1, the C ABI's own NCCL entry point
    native_comm, native = None, "not run (single rank: no communicator)"
    stats = env.all_reduce_stats()
    if world > 1:
        try:
            native_comm = NativeNcclComm(rank, world, device)
            got = env.all_reduce_stats_native(native_comm)
            torch.cuda.synchronize()
            want = torch.tensor([float(x) for x in stats], dtype=torch.float64, device=device)
            native = ("ok" if same_statistics(torch, got, want)
                      else f"MISMATCH: native {got.tolist()} vs torch {want.tolist()}")
        except Exception as e:  # reported, never hidden: the key says what happened
            native = f"FAILED: {type(e).__name__}: {e}"
            native_comm = None

    # ---- end to end through the host-buffer entry point: H2D actions, step, D2H obs/reward/flags ----
    h_act = torch.randint(0, 2, (n,), dtype=torch.uint8).pin_memory()
    h_obs = torch.empty((4, n), dtype=torch.float32).pin_memory()
    h_rew = torch.empty(n, dtype=torch.float32).pin_memory()
    h_flg = torch.empty(n, dtype=torch.uint8).pin_memory()

    def host_step():
        env.step_host(h_act, h_obs, h_rew, h_flg)

    for _ in range(3):
        host_step()
    # best of three windows of e2e_steps each (the host side of a PCIe-bound call is noisy: other processes, page
    # migration of the pinned buffers' first touch); the link ceiling below is taken the same way
    e2e_windows = [ctx.timed(host_step, args.e2e_steps) for _ in range(3)]
    e2e_s, e2e_clocks = min(e2e_windows, key=lambda w: w[0])
    h2d = h_act.numel() * h_act.element_size()
    d2h = sum(x.numel() * x.element_size() for x in (h_obs, h_rew, h_flg))
    link = measure_host_link(ctx)
    env.close()
    del env, pool, h_act, h_obs, h_rew, h_flg
    torch.cuda.empty_cache()

    peak, peak_src = measured_peak_gbs()
    configs = {}
    if not args.no_configs:
        only = [s for s in args.only_configs.split(",") if s]
        # a leg that fails (out of memory on a smaller GPU, say) is reported in its own entry; the headline line
        # still prints.  Every rank runs the same code on the same sizes, so a failure is the same on all of them.
        for spec in SUBCONFIGS:
            if only and spec[0] not in only:
                continue
            try:
                configs[spec[0]], k = run_subconfig(ctx, m, spec, args, peak)
                gpu_launches += k
            except Exception as e:
                configs[spec[0]] = {"error": f"{type(e).__name__}: {e}"}
                torch.cuda.empty_cache()
        if not only or "mixed_suite" in only:
            try:
                configs["mixed_suite"], k = run_mixed_suite(ctx, m, args, native_comm)
                gpu_launches += k
            except Exception as e:
                configs["mixed_suite"] = {"error": f"{type(e).__name__}: {e}"}
                torch.cuda.empty_cache()
    if native_comm is not None:
        native_comm.close()

    if rank == 0:
        total_env_steps = float(n) * world * args.steps
        value = total_env_steps / (ms_max * 1e-3)
        launch_s = ms_max * 1e-3 / args.steps
        achieved = BYTES_PER_ENV_STEP * n / launch_s / 1e9
        traffic, traffic_src = ncu_traffic(f"{KIND_NAME}/{n}/step")
        d2h_rate = d2h * args.e2e_steps / e2e_s / 1e9  # per GPU
        kernel_share = (ms_max / args.steps) / (1e3 * e2e_s / args.e2e_steps)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(n, world),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": BYTES_PER_ENV_STEP * n,
                         "kernel": "step_kernel_tma<CartPole-v1>" if n % 1024 == 0 else "step_kernel_tma + step_kernel tail",
                         "bytes_per_env_step": BYTES_PER_ENV_STEP, "peak_source": peak_src},
            "e2e": {"value": float(n) * world * args.e2e_steps / e2e_s, "unit": UNIT,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": args.e2e_steps,
                    "window_ms_per_step": [1e3 * w[0] / args.e2e_steps for w in e2e_windows],
                    "timing": "best of the windows listed",
                    "path": "mgym_step_host: pinned host actions -> device, step, obs/reward/flags -> pinned host",
                    "pcie_GBps_per_gpu": (h2d + d2h) * args.e2e_steps / e2e_s / 1e9,
                    "roofline": {"bound": "pcie", "achieved": d2h_rate, "peak": link["d2h_GBps_per_gpu"],
                                 "unit": "GB/s", "frac": d2h_rate / link["d2h_GBps_per_gpu"],
                                 "what": "device->host bytes of the step (95 % of what crosses the link) per second per "
                                         "GPU, against this box's pinned-memory D2H copy rate per GPU measured in the "
                                         "same run with all ranks copying at once (host_link)"},
                    "host_link": link,
                    "kernel_share_of_call": kernel_share,
                    "host_affinity_rank0": numa, "clocks": e2e_clocks},
            "gpu_launches": gpu_launches,
            "clocks": clocks,
            "native_nccl_allreduce": native,
            "episode_stats": {"episodes": stats.episodes, "mean_length": stats.length_sum / max(stats.episodes, 1),
                              "mean_return": stats.return_sum / max(stats.episodes, 1)},
            "configs": configs,
        }
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            rate, total, wall = cpu_step_loop(args.cpu_seconds, threads)
            line["cpu_baseline"] = {
                "value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                "sample": f"{total} CartPole-v1 env-steps in {wall:.1f} s: oracle C port of cartpole.rs:251-348, one env "
                          f"loop per thread, random actions, reset on done; an upper bound on the Rust reference, "
                          f"which also allocates 3 tensors per step"}
        print(json.dumps(line), flush=True)
    if sampler:
        sampler.stop()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True  # the benchmark may run from a read-only checkout: it writes nothing into the tree
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # `python bench.py --gpus N` without a launcher: start one rank per GPU ourselves
        port = os.environ.get("MASTER_PORT", "29541")
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", port, os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.gpus != world:
        sys.exit(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; launch one rank per GPU "
                 f"(python -m torch.distributed.run --nproc-per-node {args.gpus} ... bench.py --gpus {args.gpus})")
    run_native(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
