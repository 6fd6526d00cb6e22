"""Per-episode parameter redraws in the CPU oracle (tests/redraw_oracle.c: oracle_vec_step_r / oracle_vec_rollout_r /
oracle_reset_r).

1. Without ranges the redraw drivers are the parameter drivers, bit for bit; degenerate ranges at the defaults are
   no ranges.
2. With random ranges, rows change exactly where an env finished (or was reset), to the Philox draw recomputed here.
3. K steps and one rollout of K leave the same rows and states."""
import numpy as np
import pytest

from helpers import assert_bit_equal, random_actions, random_states

import params_oracle as po
import redraw_oracle as ro
from oracle import oracle

DEFAULTS = {
    0: [9.8, 1.0, 0.1, 0.5, 10.0, 0.02],
    1: [0.001, 0.0025],
    2: [0.0015, 0.0025],
    3: [10.0, 1.0, 1.0],
}
KINDS = sorted(DEFAULTS)


def defaults(kind):
    return np.asarray(DEFAULTS[kind], dtype=np.float32)


def ranges(kind, spread=0.2):
    d = defaults(kind)
    return d * np.float32(1 - spread), d * np.float32(1 + spread)


def start(cls, kind, n, seed, st, **cfg):
    """A handle in state `st`, its episodes 0-149 steps old (Pendulum's 200-step limit is then near)."""
    e = cls(kind, n, seed=seed, **cfg)
    e.state[:] = st
    e.steps[:] = np.random.default_rng(n).integers(0, 150, n).astype(np.uint32)
    e.sbt[:] = 0
    return e


def draw(seed, g, k, tag0, low, high):
    """Parameter c: word c % 4 of philox(counter (g lo, g hi, k lo, k hi[23:0] | tag << 24), key = seed), mapped in
    f64 to U[low, high) and rounded to f32."""
    out = []
    for c in range(len(low)):
        ctr = [g & 0xFFFFFFFF, g >> 32, k & 0xFFFFFFFF, ((k >> 32) & 0xFFFFFF) | ((tag0 + c // 4) << 24)]
        w = oracle.philox(ctr, [seed & 0xFFFFFFFF, seed >> 32])[c % 4]
        out.append(np.float32((float(w) * 2.0 ** -32) * (float(high[c]) - float(low[c])) + float(low[c])))
    return np.asarray(out, dtype=np.float32)


@pytest.mark.parametrize("kind", KINDS)
def test_no_ranges_and_default_ranges_equal_the_parameter_drivers(kind):
    n, T = 512, 120
    rng = np.random.default_rng(kind)
    st = random_states(rng, kind, n)
    rows = np.repeat(defaults(kind)[:, None], n, axis=1)
    ref = start(po.VecState, kind, n, 3, st, auto_reset=1)
    ref.set_params(rows)
    plain = start(ro.VecState, kind, n, 3, st, auto_reset=1)  # rows, no ranges
    plain.set_params(rows)
    degen = start(ro.VecState, kind, n, 3, st, auto_reset=1)  # ranges [default, default]
    degen.set_param_redraw(defaults(kind), defaults(kind), defaults(kind))
    for t in range(T):
        a = random_actions(rng, kind, n)
        want = ref.step(a, want_final_obs=True)
        for e in (plain, degen):
            for x, y, what in zip(want, e.step(a, want_final_obs=True), ("obs", "reward", "flags", "final_obs")):
                assert_bit_equal(y, x, f"{what} {t}")
    assert ref.stats.episodes > 0
    acts = random_actions(rng, kind, (32, n))
    want = ref.rollout(32, acts)
    for e in (plain, degen):
        got = e.rollout(32, acts)
        for x, y, what in zip(want[:3], got[:3], ("obs", "reward", "flags")):
            assert_bit_equal(y, x, f"rollout {what}")
        assert got[3] == want[3]
        assert_bit_equal(e.state, ref.state, "state")
        assert_bit_equal(e.steps, ref.steps, "steps")
        assert_bit_equal(e.params, ref.params, "rows")
        assert (e.stats.episodes, e.stats.length_sum) == (ref.stats.episodes, ref.stats.length_sum)


@pytest.mark.parametrize("kind", KINDS)
def test_random_ranges_redraw_exactly_the_finished_envs(kind):
    n, T, seed, base = 256, 150, 0x1234_5678_9ABC, 1000
    rng = np.random.default_rng(10 + kind)
    low, high = ranges(kind)
    e = start(ro.VecState, kind, n, seed, random_states(rng, kind, n), auto_reset=1, env_index_base=base)
    e.set_param_redraw(low, high, defaults(kind))
    checked = 0
    for t in range(T):
        before_rows, before_steps = e.params.copy(), e.steps.copy()
        _, _, flags = e.step(random_actions(rng, kind, n))
        live = flags == 0
        assert_bit_equal(e.params[:, live], before_rows[:, live], f"rows of live envs, step {t}")
        for i in np.flatnonzero(~live)[:4]:
            k = t - int(before_steps[i])  # t + 1 - (length of the finished episode)
            assert_bit_equal(e.params[:, i], draw(seed, base + int(i), k, 5, low, high), f"env {i}, step {t}")
            checked += 1
    assert checked > 20
    assert ((e.params >= low[:, None]) & (e.params <= high[:, None])).all()


@pytest.mark.parametrize("kind", KINDS)
def test_explicit_resets_redraw_the_masked_envs(kind):
    n, seed = 300, 77
    rng = np.random.default_rng(30 + kind)
    low, high = ranges(kind, 0.5)
    e = ro.VecState(kind, n, seed=seed, auto_reset=0)
    e.set_param_redraw(low, high, defaults(kind))
    e.reset()  # reset call 0
    for i in (0, 17, n - 1):
        assert_bit_equal(e.params[:, i], draw(seed, i, 0, 7, low, high), f"env {i}")
    mask = (rng.random(n) < 0.3).astype(np.uint8)
    before = e.params.copy()
    plain = po.VecState(kind, n, seed=seed, auto_reset=0)
    plain.reset()
    plain.reset(mask)
    e.reset(mask)  # reset call 1
    assert_bit_equal(e.state, plain.state, "reset states are the oracle's")
    assert_bit_equal(e.params[:, mask == 0], before[:, mask == 0], "unmasked rows")
    for i in np.flatnonzero(mask)[:6]:
        assert_bit_equal(e.params[:, i], draw(seed, int(i), 1, 7, low, high), f"masked env {i}")
    # manual-mode steps never redraw
    rows = e.params.copy()
    for _ in range(60):
        e.step(random_actions(rng, kind, n))
    assert_bit_equal(e.params, rows, "rows after manual steps")


@pytest.mark.parametrize("kind", KINDS)
def test_k_steps_and_one_rollout_leave_the_same_rows(kind):
    n, K = 384, 96
    rng = np.random.default_rng(40 + kind)
    low, high = ranges(kind)
    st = random_states(rng, kind, n)
    a = start(ro.VecState, kind, n, 9, st, auto_reset=1)
    b = start(ro.VecState, kind, n, 9, st, auto_reset=1)
    for e in (a, b):
        e.set_param_redraw(low, high, defaults(kind))
    acts = random_actions(rng, kind, (K, n))
    for k in range(K):
        a.step(acts[k])
    b.rollout(K, acts)
    assert a.stats.episodes > 0
    assert_bit_equal(b.params, a.params, "rows")
    assert_bit_equal(b.state, a.state, "state")
    assert_bit_equal(b.steps, a.steps, "steps")
    assert (a.stats.episodes, a.stats.length_sum) == (b.stats.episodes, b.stats.length_sum)
    assert not np.array_equal(a.params, np.repeat(defaults(kind)[:, None], n, axis=1))
