#!/usr/bin/env python
"""Per-episode parameter redraws: the per-call step and a 32-step rollout of each kind with parameter rows, without
and with redraw ranges.

Both arms live in the same process and are timed alternately, like tools/bench_params.py (warm-up, a rest before
every window, best of three windows, CUDA events), at the BASELINE sizes (2^24 envs; Pendulum 2^22).  Both handles
start from the same rows, drawn from +-20 % of the defaults; the redraw arm also redraws every env's parameters from
+-20 % at each of its resets.  Contract bytes per env-step are those of bench_params.py's parameter arm for both arms:
redraw adds none, its extra traffic is 4 P bytes per RESET (reported as `resets_per_env_step`).  Prints one JSON line
with the card's name and power limit.

    python tools/bench_param_redraw.py [--kinds 0,1,2,3] [--window 0.4] [--out profiles/bench_param_redraw_rNN.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

import modurl_gym_b200 as m  # noqa: E402

import bench  # noqa: E402  (one table of contract bytes for every tool)
from bench_params import NUM_PARAMS, PEAK_GBS, SIZES, card, measure  # noqa: E402

K = bench.ROLLOUT_CHUNK


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kinds", default="0,1,2,3")
    ap.add_argument("--window", type=float, default=0.4, help="seconds per timed window")
    ap.add_argument("--idle", type=float, default=0.25, help="rest before every window")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(0)
    result = {"card": card(), "peak_gbs": PEAK_GBS, "rollout_k": K, "spread": 0.2, "kinds": []}
    for kind in [int(k) for k in args.kinds.split(",")]:
        n = SIZES[kind]
        d = m.GpuVecEnv.param_defaults(kind)
        low, high = [0.8 * x for x in d], [1.2 * x for x in d]
        rows = m.GpuVecEnv(kind, n, seed=1)
        redraw = m.GpuVecEnv(kind, n, seed=1)
        for e in (rows, redraw):
            e.sample_params(low, high, key=1)
            e.reset()
        redraw.set_param_redraw(low, high)
        acts = bench.make_actions(torch, rows, kind, (n,), dev, gen)
        acts_k = bench.make_actions(torch, rows, kind, (K, n), dev, gen)
        obs = torch.empty((K, rows.obs_dim, n), dtype=torch.float32, device=dev)
        rew = torch.empty((K, n), dtype=torch.float32, device=dev)
        flg = torch.empty((K, n), dtype=torch.uint8, device=dev)
        arms = {}
        for name, e in (("rows", rows), ("redraw", redraw)):
            arms[f"step_{name}"] = lambda e=e: e.step(acts)
            arms[f"rollout_{name}"] = lambda e=e: e.rollout(K, acts_k, obs=obs, reward=rew, flags=flg, count_done=False)
        got = measure(arms, args.window, args.idle)
        P = NUM_PARAMS[kind]
        row = {"kind": bench.NAMES[kind], "num_envs": n, "num_params": P,
               "resets_per_env_step": redraw.stats().episodes / max(1, redraw.step_index * n)}
        for mode in ("step", "rollout"):
            for name in ("rows", "redraw"):
                sec, windows = got[f"{mode}_{name}"]
                steps = n * (1 if mode == "step" else K)
                contract = (bench.STEP_CONTRACT[kind] + 4 * P if mode == "step"
                            else bench.ROLLOUT_CONTRACT[kind] + 4 * P / K)
                rate = steps / sec
                row[f"{mode}_{name}"] = {
                    "env_steps_per_s": rate, "contract_bytes_per_env_step": contract,
                    "gbs": rate * contract / 1e9, "fraction_of_peak": rate * contract / 1e9 / PEAK_GBS,
                    "ms_per_call": sec * 1e3, "window_ms_per_call": [w * 1e3 for w in windows]}
            r, p = row[f"{mode}_redraw"], row[f"{mode}_rows"]
            row[f"{mode}_redraw_vs_rows"] = r["env_steps_per_s"] / p["env_steps_per_s"]
        result["kinds"].append(row)
        print(json.dumps(row), flush=True)
        rows.close(), redraw.close()
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
