#!/usr/bin/env python
"""Final observations in fused rollouts: mgym_rollout against mgym_rollout_final, 32-step launches with the device
policy.

Both arms live in the same process and are timed alternately, like tools/bench_param_redraw.py (warm-up, a rest
before every window, best of three windows, CUDA events), at the BASELINE sizes (2^24 envs; Pendulum and Acrobot
2^22).  The two handles of a row have the same seed and configuration, so they finish the same envs.  Rows: every
kind without parameters, and CartPole with parameter rows (+-20 % of the defaults) and with redraw ranges (+-20 %),
the PARAMS and REDRAW kernel forms.  The final arm's extra traffic is OD scattered 4-byte stores per FINISHED env
(reported as `resets_per_env_step` and `final_bytes_per_env_step`, the bytes stored, not the sectors they dirty);
`spread` is (slowest - fastest) / fastest of each arm's three windows.  Prints one JSON line with the card's name and
power limit.

    python tools/bench_rollout_final.py [--rows cartpole,...] [--window 0.4] [--out profiles/bench_rollout_final_rNN.json]
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

import bench  # noqa: E402  (one table of names and dimensions for every tool)
from bench_params import card, measure  # noqa: E402

K = bench.ROLLOUT_CHUNK
SIZES = [1 << 24, 1 << 24, 1 << 24, 1 << 22, 1 << 22]
# row name -> (kind, parameter mode)
ROWS = {"cartpole": (0, None), "mountain_car": (1, None), "mountain_car_continuous": (2, None),
        "pendulum": (3, None), "acrobot": (4, None), "cartpole_params": (0, "rows"), "cartpole_redraw": (0, "redraw")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default=",".join(ROWS))
    ap.add_argument("--window", type=float, default=0.4, help="seconds per timed window")
    ap.add_argument("--idle", type=float, default=0.25, help="rest before every window")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rollout_final.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    result = {"card": card(), "rollout_k": K, "policy": "device", "rows": []}
    for name in args.rows.split(","):
        kind, mode = ROWS[name]
        n = SIZES[kind]
        plain, final_env = m.GpuVecEnv(kind, n, seed=1), m.GpuVecEnv(kind, n, seed=1)
        for e in (plain, final_env):
            if mode is not None:
                d = m.GpuVecEnv.param_defaults(kind)
                low, high = [0.8 * x for x in d], [1.2 * x for x in d]
                e.sample_params(low, high, key=1)
                if mode == "redraw":
                    e.set_param_redraw(low, high)
            e.reset()
        od = plain.obs_dim
        obs = torch.empty((K, od, n), dtype=torch.float32, device=dev)
        rew = torch.empty((K, n), dtype=torch.float32, device=dev)
        flg = torch.empty((K, n), dtype=torch.uint8, device=dev)
        fin = torch.empty((K, od, n), dtype=torch.float32, device=dev)
        arms = {
            "rollout": lambda: plain.rollout(K, obs=obs, reward=rew, flags=flg, count_done=False),
            "rollout_final": lambda: final_env.rollout(K, obs=obs, reward=rew, flags=flg, count_done=False,
                                                       final_obs=fin, want_final_obs=True),
        }
        got = measure(arms, args.window, args.idle)
        resets = final_env.stats().episodes / max(1, final_env.step_index * n)
        row = {"row": name, "kind": bench.NAMES[kind], "num_envs": n, "params": mode or "none",
               "resets_per_env_step": resets, "final_bytes_per_env_step": resets * 4 * od}
        for arm in arms:
            sec, windows = got[arm]
            row[arm] = {"env_steps_per_s": n * K / sec, "ms_per_call": sec * 1e3,
                        "window_ms_per_call": [w * 1e3 for w in windows],
                        "spread": (max(windows) - min(windows)) / min(windows)}
        row["final_vs_rollout"] = row["rollout_final"]["env_steps_per_s"] / row["rollout"]["env_steps_per_s"]
        result["rows"].append(row)
        print(json.dumps(row), flush=True)
        plain.close(), final_env.close()
        del obs, rew, flg, fin
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
