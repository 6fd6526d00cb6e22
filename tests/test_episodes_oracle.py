"""Per-episode outputs in the CPU oracle (tests/episodes_oracle.c: oracle_vec_step_e / oracle_vec_rollout_e).

1. The episode outputs equal an independent accumulation over the oracle's own reward and flag trajectories: an f32
   running sum of the rewards in step order and a step count, from a fresh reset and from set_state ages that force
   truncations.  Entries of envs that did not finish keep a sentinel.
2. They add up to the statistics: sum of lengths = delta length_sum, written entries = delta episodes, sum of returns
   = delta return_sum (the analytic return of the counts for CartPole, MountainCar, Acrobot).
3. With NULL episode outputs the drivers are the redraw drivers, bit for bit; K steps equal one rollout of K."""
import numpy as np
import pytest

from helpers import assert_bit_equal, random_actions, random_states

import episodes_oracle as eo
import redraw_oracle as ro
from oracle import oracle

# (kind, config overrides); CartPole also with Sutton & Barto's rewards, MountainCar-v0 (no time limit by default)
# also with Gymnasium's 200 steps
CASES = [(0, {}), (0, {"sutton_barto_reward": 1}), (1, {}), (1, {"max_episode_steps": 200}), (2, {}), (3, {}), (4, {})]
IDS = ["CartPole-v1", "CartPole-v1-sutton-barto", "MountainCar-v0", "MountainCar-v0-200", "MountainCarContinuous-v0",
       "Pendulum-v1", "Acrobot-v1"]
ANALYTIC = (0, 1, 4)
T = 48


def time_limit(kind, cfg):
    """The step count at which an episode is truncated, or 0 for none."""
    return 500 if kind == 0 else int(cfg.max_episode_steps)


def start(kind, n, seed, aged, cls=eo.VecState, **cfg):
    """A handle in a random state; aged: its episodes already 1-T steps short of the time limit (set_state), so that
    truncations happen within T steps (without a limit: 1000 steps old, less up to T)."""
    rng = np.random.default_rng(seed)
    e = cls(kind, n, seed=seed, auto_reset=1, **cfg)
    e.state[:] = random_states(rng, kind, n)
    limit = time_limit(kind, e.cfg) or 1000
    e.steps[:] = (limit - rng.integers(1, T + 1, n)).astype(np.uint32) if aged else 0
    e.sbt[:] = 0
    e.ep_return[:] = 0.0  # set_state clears the running returns
    return e


def initial_return(kind, cfg, ages):
    """The f32 running return an episode of `ages` steps carries into the first step, from its constant rewards (the
    running return itself restarts at 0 on set_state for the kinds without constant rewards)."""
    if kind == 0:
        return np.zeros_like(ages, dtype=np.float32) if cfg.sutton_barto_reward else ages.astype(np.float32)
    if kind in (1, 4):
        return -ages.astype(np.float32)
    return np.zeros_like(ages, dtype=np.float32)


def expected(kind, cfg, ages, rew, flg):
    """Episode outputs [T, n] recomputed from the reward and flag trajectories [T, n]; unwritten entries = sentinel."""
    n = flg.shape[1]
    length = ages.astype(np.uint64).copy()
    ret = initial_return(kind, cfg, ages)
    want_len = np.full(flg.shape, eo.SENTINEL_LEN, dtype=np.uint32)
    want_ret = np.full(flg.shape, eo.SENTINEL_RET, dtype=np.float32)
    for k in range(flg.shape[0]):
        length += 1
        ret = (ret + rew[k]).astype(np.float32)  # f32 additions in step order
        fin = flg[k] != 0
        want_len[k, fin] = length[fin]
        want_ret[k, fin] = ret[fin]
        length[fin] = 0
        ret[fin] = 0.0
    assert n == len(ages)
    return want_ret, want_len


def stats_of(e):
    s = e.stats
    return s.episodes, s.terminated, s.truncated, s.length_sum, s.return_sum


def check_sums(kind, cfg, before, after, flg, ret, length):
    d_eps, d_term, d_trunc, d_len = (after[i] - before[i] for i in range(4))
    fin = flg != 0
    assert int(fin.sum()) == d_eps
    assert int(length[fin].astype(np.uint64).sum()) == d_len
    if kind in ANALYTIC:
        analytic = {0: (d_trunc - d_term) if cfg.sutton_barto_reward else d_len, 1: -d_len, 4: d_term - d_len}[kind]
        assert float(ret[fin].astype(np.float64).sum()) == float(analytic)
    else:
        s = before[4]
        for k in range(flg.shape[0]):  # in the oracle's own order: step by step, env by env
            for r in ret[k][fin[k]]:
                s += float(r)
        assert s == after[4]


@pytest.mark.parametrize("aged", [False, True], ids=["fresh", "aged"])
@pytest.mark.parametrize("kind,over", CASES, ids=IDS)
def test_rollout_episodes_match_an_independent_accumulation(kind, over, aged):
    n = 512
    e = start(kind, n, 7 + kind, aged, **over)
    ages = e.steps.copy()
    acts = random_actions(np.random.default_rng(kind), kind, (T, n))
    before = stats_of(e)
    obs, rew, flg, dones, ret, length = e.rollout_e(T, acts)
    want_ret, want_len = expected(kind, e.cfg, ages, rew, flg)
    assert_bit_equal(length, want_len, "ep_length")
    assert_bit_equal(ret, want_ret, "ep_return")
    assert dones == int((flg != 0).sum())
    assert dones > 0 or (kind == 3 and not aged), "Pendulum-v1 only truncates"
    if aged and time_limit(kind, e.cfg):
        assert (flg & oracle.FLAG_TRUNCATED).any(), "the ages force truncations"
    check_sums(kind, e.cfg, before, stats_of(e), flg, ret, length)


@pytest.mark.parametrize("kind,over", CASES, ids=IDS)
def test_steps_equal_a_rollout_and_null_outputs_are_the_redraw_drivers(kind, over):
    n = 256
    rng = np.random.default_rng(100 + kind)
    acts = random_actions(rng, kind, (T, n))
    stepped, rolled = start(kind, n, 3, True, **over), start(kind, n, 3, True, **over)
    plain_s, plain_r = (start(kind, n, 3, True, cls=ro.VecState, **over) for _ in range(2))  # the redraw drivers
    rets, lens = [], []
    for k in range(T):
        got = stepped.step_e(acts[k])
        want = plain_s.step(acts[k])
        for x, y, what in zip(want, got[:3], ("obs", "reward", "flags")):
            assert_bit_equal(y, x, f"step {what} {k}")
        rets.append(got[3])
        lens.append(got[4])
    out = rolled.rollout_e(T, acts)
    want = plain_r.rollout(T, acts)
    for x, y, what in zip(want[:3], out[:3], ("obs", "reward", "flags")):
        assert_bit_equal(y, x, f"rollout {what}")
    assert out[3] == want[3]
    assert_bit_equal(out[4], np.stack(rets), "rollout ep_return against K steps")
    assert_bit_equal(out[5], np.stack(lens), "rollout ep_length against K steps")
    for a, b in ((stepped, plain_s), (rolled, plain_r), (stepped, rolled)):
        assert_bit_equal(a.state, b.state, "state")
        assert_bit_equal(a.steps, b.steps, "steps")
        assert_bit_equal(a.ep_return, b.ep_return, "running returns")
        assert stats_of(a) == stats_of(b)
    # one output alone writes the same entries
    lone = start(kind, n, 3, True, **over)
    got = lone.rollout_e(T, acts, want_return=False)
    assert got[4] is None
    assert_bit_equal(got[5], out[5], "ep_length alone")


@pytest.mark.parametrize("kind", [0, 1, 2, 3])
def test_redraw_keeps_the_episode_outputs(kind):
    """With parameter rows and redraw ranges, the outputs still match the independent accumulation."""
    n = 256
    e = start(kind, n, 11, True)
    d = np.asarray({0: [9.8, 1.0, 0.1, 0.5, 10.0, 0.02], 1: [0.001, 0.0025], 2: [0.0015, 0.0025],
                    3: [10.0, 1.0, 1.0]}[kind], dtype=np.float32)
    e.set_param_redraw(d * np.float32(0.8), d * np.float32(1.2), d)
    ages = e.steps.copy()
    acts = random_actions(np.random.default_rng(kind), kind, (T, n))
    before = stats_of(e)
    obs, rew, flg, dones, ret, length = e.rollout_e(T, acts)
    want_ret, want_len = expected(kind, e.cfg, ages, rew, flg)
    assert_bit_equal(length, want_len, "ep_length")
    assert_bit_equal(ret, want_ret, "ep_return")
    check_sums(kind, e.cfg, before, stats_of(e), flg, ret, length)
