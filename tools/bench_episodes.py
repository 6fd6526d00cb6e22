#!/usr/bin/env python
"""Per-episode returns and lengths: mgym_step against mgym_step_episodes (caller uniform-random actions), and 32-step
mgym_rollout against mgym_rollout_episodes (device policy).

Both arms live in the same process and are timed alternately, like tools/bench_rollout_final.py (warm-up, a rest
before every window, best of three windows, CUDA events), at the BASELINE sizes (2^24 envs; Pendulum and Acrobot
2^22).  The two handles of a row have the same seed and configuration, so they finish the same envs; MountainCarContinuous
and Pendulum keep running returns (track_returns) in both handles, which ep_return needs.  The step arms call the C
entry points with pre-marshalled pointers, so both carry the same host overhead.  Rows: every kind without parameters,
and CartPole with parameter rows (+-20 % of the defaults) and with redraw ranges (+-20 %), the PARAMS and REDRAW kernel
forms.  The episode arms ask for both outputs and no final observations: two scattered 4-byte stores per FINISHED env
(`resets_per_env_step`); `spread` is (slowest - fastest) / fastest of each arm's three windows.  Prints one JSON line
with the card's name and power limit.

    python tools/bench_episodes.py [--rows cartpole,...] [--window 0.4] [--out profiles/bench_episodes_rNN.json]
"""
import argparse
import ctypes as C
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


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default=",".join(ROWS))
    ap.add_argument("--window", type=float, default=0.4, help="seconds per timed window")
    ap.add_argument("--idle", type=float, default=0.25, help="rest before every window")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_episodes.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(0)
    result = {"card": card(), "rollout_k": K, "step_actions": "caller", "rollout_policy": "device", "rows": []}
    for name in args.rows.split(","):
        kind, mode = ROWS[name]
        n = SIZES[kind]
        plain, epis = (m.GpuVecEnv(kind, n, seed=1, track_returns=kind in (2, 3)) for _ in range(2))
        for e in (plain, epis):
            if mode is not None:
                d = m.GpuVecEnv.param_defaults(kind)
                low, high = [0.8 * x for x in d], [1.2 * x for x in d]
                e.sample_params(low, high, key=1)
                if mode == "redraw":
                    e.set_param_redraw(low, high)
            e.reset()
        od = plain.obs_dim
        acts = bench.make_actions(torch, plain, kind, (n,), dev, gen)
        s_obs = torch.empty((od, n), dtype=torch.float32, device=dev)
        s_rew = torch.empty(n, dtype=torch.float32, device=dev)
        s_flg = torch.empty(n, dtype=torch.uint8, device=dev)
        s_ret = torch.empty(n, dtype=torch.float32, device=dev)
        s_len = torch.empty(n, dtype=torch.int32, device=dev)
        obs = torch.empty((K, od, n), dtype=torch.float32, device=dev)
        rew = torch.empty((K, n), dtype=torch.float32, device=dev)
        flg = torch.empty((K, n), dtype=torch.uint8, device=dev)
        ret = torch.empty((K, n), dtype=torch.float32, device=dev)
        length = torch.empty((K, n), dtype=torch.int32, device=dev)
        lib = plain._lib
        sa, so, sr, sf, se, sl = (ptr(t) for t in (acts, s_obs, s_rew, s_flg, s_ret, s_len))
        stream = plain._stream()
        check = m._lib.check
        arms = {
            "step": lambda: check(lib.mgym_step(plain._h, sa, so, sr, sf, None, stream)),
            "step_episodes": lambda: check(lib.mgym_step_episodes(epis._h, sa, so, sr, sf, None, se, sl, stream)),
            "rollout": lambda: plain.rollout(K, obs=obs, reward=rew, flags=flg, count_done=False),
            "rollout_episodes": lambda: epis.rollout(K, obs=obs, reward=rew, flags=flg, count_done=False,
                                                     ep_return=ret, ep_length=length, want_episodes=True),
        }
        got = measure(arms, args.window, args.idle)
        resets = epis.stats().episodes / max(1, epis.step_index * n)
        row = {"row": name, "kind": bench.NAMES[kind], "num_envs": n, "params": mode or "none",
               "track_returns": kind in (2, 3), "resets_per_env_step": resets,
               "episode_bytes_per_env_step": resets * 8}
        for arm in arms:
            sec, windows = got[arm]
            steps = n * (1 if arm.startswith("step") else K)
            row[arm] = {"env_steps_per_s": steps / sec, "ms_per_call": sec * 1e3,
                        "window_ms_per_call": [w * 1e3 for w in windows],
                        "spread": (max(windows) - min(windows)) / min(windows)}
        row["step_episodes_vs_step"] = row["step_episodes"]["env_steps_per_s"] / row["step"]["env_steps_per_s"]
        row["rollout_episodes_vs_rollout"] = (row["rollout_episodes"]["env_steps_per_s"] /
                                              row["rollout"]["env_steps_per_s"])
        result["rows"].append(row)
        print(json.dumps(row), flush=True)
        plain.close(), epis.close()
        del obs, rew, flg, ret, length, s_obs, s_rew, s_flg, s_ret, s_len, acts
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
