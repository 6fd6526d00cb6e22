"""Per-env physics parameters in the CPU oracle (tests/params_oracle.c: oracle_vec_step_p / oracle_vec_rollout_p /
oracle_sample_params).

1. The kinds' constants passed as parameters, and no parameters, give the same bits as the oracle's own drivers.
2. Random per-env parameters (+-50 % of the defaults) against a float64 recomputation of one step, written here."""
import numpy as np
import pytest

from helpers import assert_bit_equal, random_actions, random_states

import params_oracle as po
from oracle import oracle

DEFAULTS = {
    0: [9.8, 1.0, 0.1, 0.5, 10.0, 0.02],
    1: [0.001, 0.0025],
    2: [0.0015, 0.0025],
    3: [10.0, 1.0, 1.0],
}
KINDS = sorted(DEFAULTS)


def default_rows(kind, n):
    return np.repeat(np.asarray(DEFAULTS[kind], dtype=np.float32)[:, None], n, axis=1)


def trio(kind, n, seed, **cfg):
    """The oracle's own drivers, the parameter drivers with the defaults, and the parameter drivers with NULL."""
    rng = np.random.default_rng(seed)
    a = oracle.VecState(kind, n, seed=seed, **cfg)
    b = po.VecState(kind, n, seed=seed, **cfg)
    c = po.VecState(kind, n, seed=seed, **cfg)
    st = random_states(rng, kind, n)
    steps = rng.integers(0, 150, n).astype(np.uint32)
    for e in (a, b, c):
        e.state[:] = st
        e.steps[:] = steps
    b.set_params(default_rows(kind, n))
    return rng, a, b, c


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("mode", ["auto", "manual", "non_euler"])
def test_default_parameters_step_bit_equal(kind, mode):
    if mode == "non_euler" and kind != 0:
        pytest.skip("is_euler is a CartPole option")
    cfg = {"auto_reset": int(mode != "manual")}
    if mode == "non_euler":
        cfg["is_euler"] = 0
    n = 512
    rng, a, b, c = trio(kind, n, 11, **cfg)
    for _ in range(40):
        act = random_actions(rng, kind, n)
        out_a = a.step(act, want_final_obs=True)
        for e in (b, c):
            for x, y, what in zip(out_a, e.step(act, want_final_obs=True), ("obs", "reward", "flags", "final_obs")):
                assert_bit_equal(y, x, what)
    for e in (b, c):
        assert_bit_equal(e.state, a.state, "state")
        assert_bit_equal(e.steps, a.steps, "steps")
        assert_bit_equal(e.sbt, a.sbt, "sbt")


@pytest.mark.parametrize("kind", KINDS)
def test_default_parameters_rollout_bit_equal(kind):
    """The rollout driver (defaults, and NULL) against K calls of the oracle's own step driver."""
    n, K = 384, 64
    rng, a, b, c = trio(kind, n, 12, auto_reset=1)
    acts = random_actions(rng, kind, (K, n))
    want = [a.step(acts[k]) for k in range(K)]
    for e in (b, c):
        obs, rew, flg, dc = e.rollout(K, acts)
        for k, (wo, wr, wf) in enumerate(want):
            assert_bit_equal(obs[k], wo, f"obs {k}")
            assert_bit_equal(rew[k], wr, f"reward {k}")
            assert_bit_equal(flg[k], wf, f"flags {k}")
        assert dc == sum(int((wf != 0).sum()) for _, _, wf in want)
        assert_bit_equal(e.state, a.state, "state")
        assert (e.stats.episodes, e.stats.length_sum) == (a.stats.episodes, a.stats.length_sum)
    for x, y in zip(b.rollout(32, None), c.rollout(32, None)):  # device policy
        assert_bit_equal(x, y, "rollout, sampled actions")


def random_params(rng, kind, n):
    d = np.asarray(DEFAULTS[kind], dtype=np.float64)[:, None]
    return (d * rng.uniform(0.5, 1.5, (len(DEFAULTS[kind]), n))).astype(np.float32)


def f64_step(kind, st, a, prm):
    """One step in float64 (Gymnasium / cartpole.rs equations, no reset): new state, reward, flags."""
    f32 = lambda x: float(np.float32(x))
    st = st.astype(np.float64)
    prm = prm.astype(np.float64)
    if kind == 0:
        g, mc, mp, l, fm, tau = prm
        x, xd, th, thd = st
        force = np.where(a == 0, -fm, fm)
        tm, pml = mp + mc, mp * l
        s, c = np.sin(th), np.cos(th)
        temp = (force + pml * thd * thd * s) / tm
        thacc = (g * s - c * temp) / (l * (4.0 / 3.0 - mp * c * c / tm))
        xacc = temp - pml * thacc * c / tm
        new = np.stack([x + tau * xd, xd + tau * xacc, th + tau * thd, thd + tau * thacc])
        thr = f32(f32(f32(12.0 * 2.0) * f32(np.pi)) / 360.0)
        term = (np.abs(new[0]) > f32(2.4)) | (np.abs(new[2]) > thr)
        return new, np.ones_like(x), term.astype(np.uint8)
    if kind in (1, 2):
        p, v = st
        lo, hi, vmax = f32(-1.2), f32(0.6), f32(0.07)
        if kind == 1:
            force, grav = prm
            v = v + (a.astype(np.float64) - 1.0) * force + np.cos(3 * p) * (-grav)
        else:
            power, grav = prm
            v = v + np.clip(a.astype(np.float64), -1, 1) * power - grav * np.cos(3 * p)
        v = np.clip(v, -vmax, vmax)
        p = np.clip(p + v, lo, hi)
        v = np.where((p == lo) & (v < 0), 0.0, v)
        goal = f32(0.5) if kind == 1 else f32(0.45)
        term = (p >= goal) & (v >= 0)
        rew = -np.ones_like(p) if kind == 1 else np.where(term, 100.0, 0.0) - 0.1 * a.astype(np.float64) ** 2
        return np.stack([p, v]), rew, term.astype(np.uint8)
    g, m, l = prm
    th, thd = st
    u = np.clip(a.astype(np.float64), -2, 2)
    an = np.mod(th + np.pi, 2 * np.pi) - np.pi
    cost = an ** 2 + 0.1 * thd ** 2 + 0.001 * u ** 2
    nthd = np.clip(thd + (3 * g / (2 * l) * np.sin(th) + 3.0 / (m * l * l) * u) * 0.05, -8, 8)
    return np.stack([th + nthd * 0.05, nthd]), -cost, np.zeros(th.shape, np.uint8)


@pytest.mark.parametrize("kind", KINDS)
def test_random_parameters_against_float64(kind):
    n = 4096
    rng = np.random.default_rng(20 + kind)
    v = po.VecState(kind, n, seed=3, auto_reset=0, max_episode_steps=0)
    st = random_states(rng, kind, n)
    if kind == 3:
        st[0] = rng.uniform(-3, 3, n)  # away from the +-pi seam of angle_normalize, where f32 and f64 may wrap apart
    v.state[:] = st
    v.sbt[:] = 0  # steps_beyond_terminated = None: a falling pole still earns 1 (cartpole.rs:319-329)
    prm = random_params(rng, kind, n)
    v.set_params(prm)
    act = random_actions(rng, kind, n)
    obs, rew, flags = v.step(act)
    want_st, want_rew, want_flags = f64_step(kind, st, act, prm)
    floor = 1e-3 if kind in (1, 2) else 1.0  # MountainCar velocities are ~1e-3
    err = np.abs(v.state.astype(np.float64) - want_st) / np.maximum(floor, np.abs(want_st))
    assert err.max() <= 1e-5, float(err.max())
    err_r = np.abs(rew.astype(np.float64) - want_rew) / np.maximum(1.0, np.abs(want_rew))
    assert err_r.max() <= 1e-5, float(err_r.max())
    assert np.array_equal(flags & 1, want_flags)


@pytest.mark.parametrize("kind", KINDS)
def test_sample_params_rule(kind):
    """oracle_sample_params: word c % 4 of the Philox block (g, key) with tag 3 + c // 4, U[low, high) in f64."""
    n = 64
    v = po.VecState(kind, n, seed=99, env_index_base=1000)
    d = np.asarray(DEFAULTS[kind], dtype=np.float32)
    low, high = d * np.float32(0.5), d * np.float32(1.5)
    mask = (np.arange(n) % 3 != 0).astype(np.uint8)
    rows = v.sample_params(low, high, mask=mask, key=77, defaults=d).copy()
    assert_bit_equal(rows[:, mask == 0], default_rows(kind, n)[:, mask == 0], "unmasked rows")
    for i in np.flatnonzero(mask)[:8]:
        for c in range(len(d)):
            w = oracle.philox([(1000 + i) & 0xFFFFFFFF, (1000 + i) >> 32, 77, (3 + c // 4) << 24], [99, 0])[c % 4]
            want = np.float32((float(w) * 2.0 ** -32) * (float(high[c]) - float(low[c])) + float(low[c]))
            assert_bit_equal(rows[c, i], want, f"param {c} of env {i}")
    assert ((rows >= low[:, None]) & (rows <= high[:, None])).all()
