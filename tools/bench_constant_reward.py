#!/usr/bin/env python
"""The handle-owned reward row: `mgym_step` into the handle's own reward row (what `GpuVecEnv.step` passes; a handle
whose rewards are all one value stores none) against `mgym_step` into an explicit reward buffer (written every step).

Both arms live in the same process and are timed alternately, like tools/bench_episodes.py (warm-up, a rest before
every window, best of three windows, CUDA events), with caller uniform-random actions from a pre-generated pool.  The two
handles of a row have the same seed and configuration and are called with pre-marshalled pointers, so both carry the
same host overhead.  CartPole-v1 and MountainCar-v0 (2^24 envs) are the constant-reward kinds and pass no observation
buffer (the observation is the state rows, as in `bench.py`'s headline); Pendulum-v1 (2^22, its BASELINE size) is the
control: its rewards are not constant, so both arms store them and also write the observation buffer.  `spread` is
(slowest - fastest) / fastest of each arm's three windows.  Prints one JSON line with the card's name and power limit.

    python tools/bench_constant_reward.py [--rows cartpole,...] [--window 0.4] [--out profiles/bench_constant_reward_rNN.json]
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

# row name -> (kind, envs, bytes per env-step moved by the explicit arm, by the row arm)
ROWS = {"cartpole": (0, 1 << 24, 40, 36), "mountain_car": (1, 1 << 24, 22, 18), "pendulum": (3, 1 << 22, 39, 39)}
POOL = 16


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
        raise SystemExit("bench_constant_reward.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(0)
    result = {"card": card(), "step_actions": "caller, uniform random, pool of 16", "rows": []}
    for name in args.rows.split(","):
        kind, n, bytes_explicit, bytes_row = ROWS[name]
        row_env, buf_env = (m.GpuVecEnv(kind, n, seed=1) for _ in range(2))
        for e in (row_env, buf_env):
            e.reset()
        pool = [bench.make_actions(torch, row_env, kind, (n,), dev, gen) for _ in range(POOL)]
        pa = [ptr(a) for a in pool]
        od = row_env.obs_dim
        obs = None if row_env.obs_is_state else torch.empty((od, n), dtype=torch.float32, device=dev)
        rew = torch.empty(n, dtype=torch.float32, device=dev)
        flg = torch.empty(n, dtype=torch.uint8, device=dev)
        po, pr, pf = ptr(obs), ptr(rew), ptr(flg)
        p_row = C.c_void_p(row_env._lib.mgym_reward_ptr(row_env._h))
        lib, check, stream = row_env._lib, m._lib.check, row_env._stream()
        i = {"row": 0, "explicit": 0}

        def step_row():
            check(lib.mgym_step(row_env._h, pa[i["row"] % POOL], po, p_row, pf, None, stream))
            i["row"] += 1

        def step_explicit():
            check(lib.mgym_step(buf_env._h, pa[i["explicit"] % POOL], po, pr, pf, None, stream))
            i["explicit"] += 1

        arms = {"row": step_row, "explicit": step_explicit}
        got = measure(arms, args.window, args.idle)
        out = {"name": name, "kind": bench.NAMES[kind], "num_envs": n, "reward_constant": row_env.reward_constant,
               "bytes_per_env_step": {"row": bytes_row, "explicit": bytes_explicit}}
        for arm in arms:
            sec, windows = got[arm]
            out[arm] = {"env_steps_per_s": n / sec, "ms_per_call": sec * 1e3,
                        "window_ms_per_call": [w * 1e3 for w in windows],
                        "spread": (max(windows) - min(windows)) / min(windows)}
        out["row_vs_explicit"] = out["row"]["env_steps_per_s"] / out["explicit"]["env_steps_per_s"]
        result["rows"].append(out)
        print(json.dumps(out), flush=True)
        row_env.close(), buf_env.close()
        del pool, obs, rew, flg
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
