#!/usr/bin/env python
"""Per-env physics parameters: the per-call step and a 32-step rollout of each kind with and without parameters.

Both arms live in the same process and are timed alternately (warm-up, a rest before every window, best of three
windows, CUDA events), at the BASELINE sizes (2^24 envs; Pendulum 2^22).  The parameter arm draws every env's
parameters from +-20 % of the defaults.  Contract bytes per env-step are bench.py's plus the parameter rows:
4 P for the step, 4 P / K for the rollout.  Prints one JSON line with the card's name and power limit.

    python tools/bench_params.py [--kinds 0,1,2,3] [--window 0.4] [--out profiles/bench_params_rNN.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import modurl_gym_b200 as m  # noqa: E402

import bench  # noqa: E402  (one table of contract bytes for every tool)

SIZES = [1 << 24, 1 << 24, 1 << 24, 1 << 22]
NUM_PARAMS = [6, 2, 2, 3]
K = bench.ROLLOUT_CHUNK
PEAK_GBS = 6451.5  # the measured HBM peak every fraction in DESIGN.md is quoted against (MEASURED_PEAKS.json)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, sm = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": sm}
    except Exception as exc:  # the numbers are still worth having; say that the card was not read
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"not read ({exc})"}


def window(fn, seconds, reps_hint):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = reps_hint
    while True:
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        sec = e0.elapsed_time(e1) * 1e-3
        if sec >= seconds or reps >= 100000:
            return sec / reps, reps
        reps = max(reps * 2, int(reps * seconds / max(sec, 1e-6)) + 1)


def measure(arms, seconds, idle, windows=3):
    """arms: name -> fn.  Alternating windows; per arm the best seconds per call."""
    for fn in arms.values():  # warm-up: module load, occupancy queries, first-touch
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    reps = {k: window(fn, 0.05, 2)[1] for k, fn in arms.items()}
    best = {k: [] for k in arms}
    for _ in range(windows):
        for k, fn in arms.items():
            time.sleep(idle)
            sec, reps[k] = window(fn, seconds, reps[k])
            best[k].append(sec)
    return {k: (min(v), v) for k, v in best.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kinds", default="0,1,2,3")
    ap.add_argument("--window", type=float, default=0.4, help="seconds per timed window")
    ap.add_argument("--idle", type=float, default=0.25, help="rest before every window")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(0)
    result = {"card": card(), "peak_gbs": PEAK_GBS, "rollout_k": K, "kinds": []}
    for kind in [int(k) for k in args.kinds.split(",")]:
        n = SIZES[kind]
        plain = m.GpuVecEnv(kind, n, seed=1)
        param = m.GpuVecEnv(kind, n, seed=1)
        d = m.GpuVecEnv.param_defaults(kind)
        param.sample_params([0.8 * x for x in d], [1.2 * x for x in d], key=1)
        for e in (plain, param):
            e.reset()
        acts = bench.make_actions(torch, plain, kind, (n,), dev, gen)
        acts_k = bench.make_actions(torch, plain, kind, (K, n), dev, gen)
        obs = torch.empty((K, plain.obs_dim, n), dtype=torch.float32, device=dev)
        rew = torch.empty((K, n), dtype=torch.float32, device=dev)
        flg = torch.empty((K, n), dtype=torch.uint8, device=dev)
        arms = {}
        for name, e in (("plain", plain), ("params", param)):
            arms[f"step_{name}"] = lambda e=e: e.step(acts)
            arms[f"rollout_{name}"] = lambda e=e: e.rollout(K, acts_k, obs=obs, reward=rew, flags=flg, count_done=False)
        got = measure(arms, args.window, args.idle)
        P = NUM_PARAMS[kind]
        row = {"kind": bench.NAMES[kind], "num_envs": n}
        for mode in ("step", "rollout"):
            for name in ("plain", "params"):
                sec, windows = got[f"{mode}_{name}"]
                steps = n * (1 if mode == "step" else K)
                extra = (4 * P if mode == "step" else 4 * P / K) if name == "params" else 0
                contract = (bench.STEP_CONTRACT[kind] if mode == "step" else bench.ROLLOUT_CONTRACT[kind]) + extra
                rate = steps / sec
                row[f"{mode}_{name}"] = {
                    "env_steps_per_s": rate, "contract_bytes_per_env_step": contract,
                    "gbs": rate * contract / 1e9, "fraction_of_peak": rate * contract / 1e9 / PEAK_GBS,
                    "ms_per_call": sec * 1e3, "window_ms_per_call": [w * 1e3 for w in windows]}
        result["kinds"].append(row)
        print(json.dumps(row), flush=True)
        plain.close(), param.close()
        del obs, rew, flg, acts, acts_k
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
