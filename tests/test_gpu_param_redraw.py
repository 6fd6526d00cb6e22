"""Per-episode parameter redraws on the device (mgym_set_param_redraw / mgym_get_param_redraw): every reset draws
the env's parameters, inside the step, the TMA step's reset warp, the rollout and the explicit resets."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import redraw_oracle as ro
from helpers import assert_bit_equal, random_actions, random_states

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

KINDS = [0, 1, 2, 3]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def gym():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import modurl_gym_b200 as m

    m.load_library()
    return m


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def same(x, y):
    if x is None or y is None:
        return x is y
    if x.dtype == torch.float32:
        x, y = x.view(torch.int32), y.view(torch.int32)
    return torch.equal(x, y)


def defaults(gym, kind):
    return np.asarray(gym.GpuVecEnv.param_defaults(kind), dtype=np.float32)


def ranges(gym, kind, spread=0.2):
    d = defaults(gym, kind)
    return d * np.float32(1 - spread), d * np.float32(1 + spread)


def ages(rng, kind, n):
    """Episode step counts spread over the kind's episode, so that envs finish during a short test."""
    return rng.integers(0, 480 if kind == 0 else 190, n).astype(np.int32)


def twins(gym, kind, n, rng, count, **kw):
    """`count` handles in the same random state (step index 0, random episode ages)."""
    es = [gym.GpuVecEnv(kind, n, seed=7, **kw) for _ in range(count)]
    st, steps = dev(random_states(rng, kind, n)), dev(ages(rng, kind, n))
    for e in es:
        e.reset()
        e.set_state(st, steps)
    return es


def assert_same_handles(*es):
    a = es[0]
    for b in es[1:]:
        for x, y in zip(a.get_state(), b.get_state()):
            assert same(x, y)
        assert same(a.get_params(), b.get_params())
        assert a.stats() == b.stats()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [1 << 20, (1 << 20) + 4, 1000])
def test_default_ranges_are_bit_identical_to_rows_and_to_no_rows(gym, kind, n):
    """Ranges [default, default] redraw the defaults at every reset: the same bits as a rows-only handle and as a
    handle without rows, on the TMA step, the ragged tail, scalar lanes, and FULL and non-FULL rollouts."""
    rng = np.random.default_rng(kind * 7 + n % 13)
    a, b, c = twins(gym, kind, n, rng, 3, track_returns=True)
    d = defaults(gym, kind)
    b.set_params(torch.tensor(d).repeat(n, 1).T.contiguous())
    c.set_param_redraw(list(d), list(d))
    for t in range(12):
        acts = dev(random_actions(rng, kind, n))
        ia, fa = a.step(acts, want_final_obs=True)
        for e in (b, c):
            ie, fe = e.step(acts, want_final_obs=True)
            assert same(ia.state, ie.state) and same(ia.reward, ie.reward) and same(ia.flags, ie.flags), t
            assert same(fa, fe), t
    assert a.stats().episodes > 0
    assert_same_handles(a, b, c)
    ra = a.rollout(16)  # FULL form when n % 128 == 0
    assert all(all(same(x, y) for x, y in zip(ra, e.rollout(16))) for e in (b, c))
    acts = dev(random_actions(rng, kind, (8, n)))
    ra = a.rollout(8, acts, want_obs=False)  # non-FULL
    for e in (b, c):
        re_ = e.rollout(8, acts, want_obs=False)
        assert same(ra.reward, re_.reward) and same(ra.flags, re_.flags) and same(ra.done_count, re_.done_count)
    assert_same_handles(a, b, c)
    for e in (a, b, c):
        e.close()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [4096, 1000, 1026])
def test_random_ranges_match_oracle(gym, kind, n):
    """200 steps with auto-resets, then a 32-step rollout, bit-exact to oracle_vec_step_r / oracle_vec_rollout_r:
    flags, rewards, observations, state and the parameter rows after every step; rows of live envs unchanged."""
    rng = np.random.default_rng(100 + kind + n)
    low, high = ranges(gym, kind, 0.3)
    env = gym.GpuVecEnv(kind, n, seed=31, env_index_base=4 * 12345, track_returns=True)
    ref = ro.VecState(kind, n, seed=31, auto_reset=1, env_index_base=4 * 12345)
    st, steps = random_states(rng, kind, n), ages(rng, kind, n)
    env.reset()  # step index 0, like the oracle's t
    env.set_state(dev(st), dev(steps))
    ref.state[:], ref.steps[:], ref.sbt[:] = st, steps, 0
    env.set_param_redraw(low, high)
    ref.set_param_redraw(low, high, defaults(gym, kind))
    finished = 0
    for t in range(200):
        acts = random_actions(rng, kind, n)
        before = host(env.get_params())
        info = env.step(dev(acts))
        obs, rew, flg = ref.step(acts)
        assert_bit_equal(host(info.flags), flg, f"flags {t}")
        assert_bit_equal(host(info.reward), rew, f"reward {t}")
        assert_bit_equal(host(info.state), obs, f"obs {t}")
        rows = host(env.get_params())
        assert_bit_equal(rows, ref.params, f"rows {t}")
        assert_bit_equal(rows[:, flg == 0], before[:, flg == 0], f"rows of live envs {t}")
        finished += int((flg != 0).sum())
    assert finished > n // 8
    acts = random_actions(rng, kind, (32, n))
    r = env.rollout(32, dev(acts))
    obs, rew, flg, dc = ref.rollout(32, acts)
    assert_bit_equal(host(r.flags), flg, "rollout flags")
    assert_bit_equal(host(r.reward), rew, "rollout reward")
    assert_bit_equal(host(r.obs), obs, "rollout obs")
    assert int(r.done_count.item()) == dc
    assert_bit_equal(host(env.get_state()[0]), ref.state, "state")
    assert_bit_equal(host(env.get_params()), ref.params, "rows after the rollout")
    s = env.stats()
    assert (s.episodes, s.length_sum) == (ref.stats.episodes, ref.stats.length_sum)
    env.close()


def test_steps_and_rollouts_leave_the_same_rows(gym):
    """CartPole (its rollout draws reset states ahead of time): 64 steps, rollout(16) x 4 and rollout(64) on three
    twins leave the same state, rows and statistics."""
    n, kind = 1 << 20, 0
    rng = np.random.default_rng(5)
    a, b, c = twins(gym, kind, n, rng, 3)
    low, high = ranges(gym, kind)
    for e in (a, b, c):
        e.set_param_redraw(low, high)
    for _ in range(64):
        a.step(a.sample_actions())  # the rollout's own device policy
    for _ in range(4):
        b.rollout(16)
    c.rollout(64)
    assert a.stats().episodes > n
    assert_same_handles(a, b, c)
    for e in (a, b, c):
        e.close()


@pytest.mark.parametrize("kind", KINDS)
def test_four_shards_equal_one_handle(gym, kind):
    n = 8192
    q = n // 4
    rng = np.random.default_rng(9)
    low, high = ranges(gym, kind, 0.5)
    whole = gym.GpuVecEnv(kind, n, seed=12)
    shards = [gym.GpuVecEnv(kind, q, seed=12, env_index_base=i * q) for i in range(4)]
    st, steps = dev(random_states(rng, kind, n)), dev(ages(rng, kind, n))
    for e, sl in [(whole, slice(0, n))] + [(s, slice(i * q, (i + 1) * q)) for i, s in enumerate(shards)]:
        e.set_param_redraw(low, high)
        e.reset()  # reset call 0 on every handle: keyed by the global env index
        e.set_state(st[:, sl].contiguous(), steps[sl].contiguous())
    assert same(torch.cat([s.get_params() for s in shards], 1), whole.get_params())
    for t in range(80):
        acts = dev(random_actions(rng, kind, n))
        iw = whole.step(acts)
        for i, s in enumerate(shards):
            si = s.step(acts[i * q:(i + 1) * q].contiguous())
            assert same(si.state, iw.state[:, i * q:(i + 1) * q]) and same(si.flags, iw.flags[i * q:(i + 1) * q]), t
    whole.rollout(16)
    for s in shards:
        s.rollout(16)
    assert same(torch.cat([s.get_params() for s in shards], 1), whole.get_params())
    assert same(torch.cat([s.get_state()[0] for s in shards], 1), whole.get_state()[0])
    for e in [whole] + shards:
        e.close()


@pytest.mark.parametrize("kind", KINDS)
def test_explicit_resets_redraw_the_masked_envs(gym, kind):
    n = 5000
    rng = np.random.default_rng(60 + kind)
    low, high = ranges(gym, kind, 0.5)
    env = gym.GpuVecEnv(kind, n, seed=77, env_index_base=12, auto_reset=False)
    ref = ro.VecState(kind, n, seed=77, env_index_base=12, auto_reset=0)
    env.set_param_redraw(low, high)
    ref.set_param_redraw(low, high, defaults(gym, kind))
    assert_bit_equal(host(env.get_params()), ref.params, "ranges leave the current episodes alone")
    assert_bit_equal(host(env.reset()), ref.reset(), "reset obs")
    assert_bit_equal(host(env.get_params()), ref.params, "reset(): every env")
    for t in range(3):
        mask = (rng.random(n) < 0.3).astype(np.uint8)
        before = host(env.get_params())
        env.reset(mask=dev(mask))
        ref.reset(mask)
        got = host(env.get_params())
        assert_bit_equal(got, ref.params, f"reset(mask) {t}")
        assert_bit_equal(got[:, mask == 0], before[:, mask == 0], f"unmasked rows {t}")
        assert_bit_equal(host(env.get_state()[0]), ref.state, f"state {t}")
    rows = env.get_params().clone()  # manual-mode steps never redraw
    for t in range(40):
        info = env.step(dev(random_actions(rng, kind, n)))
        if t % 10 == 9:
            env.reset(mask=info.flags != 0)  # the reference's caller loop
            ref.reset(host(info.flags != 0).astype(np.uint8))
            rows = torch.from_numpy(ref.params).cuda()
        assert same(env.get_params(), rows), t
    env.close()


@pytest.mark.parametrize("kind", [0, 3])
def test_reset_pool_supplies_states_parameters_come_from_philox(gym, kind):
    n, P = 4096, 777
    rng = np.random.default_rng(70 + kind)
    low, high = ranges(gym, kind)
    pool = random_states(rng, kind, P)
    env = gym.GpuVecEnv(kind, n, seed=3)
    ref = ro.VecState(kind, n, seed=3, auto_reset=1)
    env.set_reset_pool(dev(pool))
    ref.set_reset_pool(pool)
    st, steps = random_states(rng, kind, n), ages(rng, kind, n)
    env.reset()
    env.set_state(dev(st), dev(steps))
    ref.state[:], ref.steps[:], ref.sbt[:] = st, steps, 0
    env.set_param_redraw(low, high)
    ref.set_param_redraw(low, high, defaults(gym, kind))
    for t in range(60):
        acts = random_actions(rng, kind, n)
        info = env.step(dev(acts))
        obs, _, flg = ref.step(acts)
        assert_bit_equal(host(info.flags), flg, f"flags {t}")
        assert_bit_equal(host(info.state), obs, f"obs {t}")
        assert_bit_equal(host(env.get_params()), ref.params, f"rows {t}")
    acts = random_actions(rng, kind, (16, n))
    env.rollout(16, dev(acts))
    ref.rollout(16, acts)
    assert_bit_equal(host(env.get_params()), ref.params, "rows after the rollout")
    assert_bit_equal(host(env.get_state()[0]), ref.state, "state after the rollout")
    assert ref.stats.episodes > 0
    env.close()


@pytest.mark.parametrize("kind", [0, 2])
def test_step_host_chunks_match_step(gym, kind):
    n = 1 << 20  # chunked step_host: sub-range launches (first / ld)
    rng = np.random.default_rng(80 + kind)
    a, b = twins(gym, kind, n, rng, 2)
    low, high = ranges(gym, kind)
    for e in (a, b):
        e.set_param_redraw(low, high)
    od = a.obs_dim
    for t in range(6):
        acts = random_actions(rng, kind, n)
        o, r, f = np.empty((od, n), np.float32), np.empty(n, np.float32), np.empty(n, np.uint8)
        a.step_host(acts, o, r, f)
        ib = b.step(dev(acts))
        assert_bit_equal(o, host(ib.state), f"obs {t}")
        assert_bit_equal(f, host(ib.flags), f"flags {t}")
        assert same(a.get_params(), b.get_params()), t
    assert a.stats().episodes > 0
    assert_same_handles(a, b)
    a.close(), b.close()


@pytest.mark.parametrize("kind", [0, 1])
def test_graph_of_sample_and_step_replays_like_eager(gym, kind):
    n, T = 8192, 60
    rng = np.random.default_rng(90 + kind)
    a = gym.GpuVecEnv(kind, n, seed=5)
    b = gym.GpuVecEnv(kind, n, seed=5, graph_capturable=True)
    low, high = ranges(gym, kind, 0.5)
    st, steps = dev(random_states(rng, kind, n)), dev(ages(rng, kind, n))
    for e in (a, b):
        e.set_param_redraw(low, high)
        e.reset()
        e.set_state(st, steps)
    acts_b = torch.empty(n, dtype=b.action_dtype, device="cuda")
    b.step(b.sample_actions(out=acts_b))
    a.step(a.sample_actions())
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        b.sample_actions(out=acts_b)
        info_b = b.step(acts_b)
    torch.cuda.synchronize()
    for t in range(T):
        ia = a.step(a.sample_actions())
        graph.replay()
        assert same(ia.state, info_b.state) and same(ia.flags, info_b.flags), t
        assert same(a.get_params(), b.get_params()), t
    assert a.stats() == b.stats() and a.stats().episodes > 0
    a.close(), b.close()


@pytest.mark.parametrize("kind", [0, 3])
def test_checkpoints_carry_the_ranges(gym, kind):
    n = 4096
    rng = np.random.default_rng(5)
    low, high = ranges(gym, kind)
    a = gym.GpuVecEnv(kind, n, seed=8)
    a.set_param_redraw(low, high)
    a.reset()
    a.set_state(dev(random_states(rng, kind, n)), dev(ages(rng, kind, n)))
    acts = [dev(random_actions(rng, kind, n)) for _ in range(40)]
    for x in acts[:10]:
        a.step(x)
    blob = a.checkpoint()
    want = []
    for x in acts[10:]:
        want.append((a.step(x).state.clone(), a.get_params()))
    b = gym.GpuVecEnv(kind, n, seed=0)
    b.restore(blob)
    assert b.param_redraw() == a.param_redraw()
    for x, (ws, wp) in zip(acts[10:], want):
        assert same(b.step(x).state, ws) and same(b.get_params(), wp)
    assert a.stats() == b.stats() and a.stats().episodes > 0
    # without ranges the blob is the rows-only format byte for byte: has_params = 1 (bit 1 clear), no ranges after
    # the rows
    c = gym.GpuVecEnv(kind, n, seed=0)
    c.restore(blob)
    c.set_param_redraw(None)
    plain = c.checkpoint()
    assert gym.load_library().mgym_checkpoint_size(c._h) == len(plain) == len(blob) - 8 * len(low)
    has_params = 4 * 12  # offset of the has_params word in the header
    assert int.from_bytes(blob[has_params:has_params + 4], "little") == 3
    assert plain == blob[:has_params] + (1).to_bytes(4, "little") + blob[has_params + 4:len(plain)]
    # loading it turns redraw off: later resets keep the rows
    a.restore(plain)
    assert a.param_redraw() is None
    rows = a.get_params()
    for x in acts[10:]:
        a.step(x)
    assert a.stats().episodes > c.stats().episodes  # envs finished, and nothing was redrawn
    assert same(a.get_params(), rows)
    for e in (a, b, c):
        e.close()


def test_rejections_leave_the_handle_untouched(gym):
    from modurl_gym_b200._lib import MgymError

    n = 2048
    lib = gym.load_library()
    env = gym.GpuVecEnv(0, n, seed=2)
    env.reset()
    size = lib.mgym_checkpoint_size(env._h)
    low, high = ranges(gym, 0)
    bad_sets = []
    for c, lo, hi in ((0, float("nan"), None), (4, None, float("inf")), (2, 0.0, None), (1, -1.0, None),
                      (5, None, float("-inf")), (0, 11.0, 10.0)):
        bl, bh = list(low), list(high)
        if lo is not None:
            bl[c] = lo
        if hi is not None:
            bh[c] = hi
        bad_sets.append((bl, bh))
    for bl, bh in bad_sets:
        with pytest.raises(MgymError):
            env.set_param_redraw(bl, bh)
        assert env.param_redraw() is None
        assert lib.mgym_checkpoint_size(env._h) == size, "a rejected call allocates no rows"
    lo = (C.c_float * 6)(*low)
    assert lib.mgym_set_param_redraw(env._h, lo, None, None) == -1  # one of low / high NULL
    assert lib.mgym_set_param_redraw(env._h, None, lo, None) == -1
    assert lib.mgym_checkpoint_size(env._h) == size
    # a capturing stream
    x = torch.zeros(1, device="cuda")
    graph = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(graph):
        rc = lib.mgym_set_param_redraw(env._h, lo, (C.c_float * 6)(*high),
                                       C.c_void_p(torch.cuda.current_stream().cuda_stream))
        x += 1
    assert rc == -1 and env.param_redraw() is None
    assert lib.mgym_checkpoint_size(env._h) == size
    # accepted ranges, then rejected ones: the first stay
    env.set_param_redraw(low, high)
    want = (tuple(float(v) for v in low), tuple(float(v) for v in high))
    assert env.param_redraw() == want
    rows = env.get_params()
    for bl, bh in bad_sets:
        with pytest.raises(MgymError):
            env.set_param_redraw(bl, bh)
        assert env.param_redraw() == want
    assert same(env.get_params(), rows)
    # the dict form: missing names are held at their default
    env.set_param_redraw({"gravity": (9.0, 10.0), "tau": (0.01, 0.03)})
    d = defaults(gym, 0)
    lo_, hi_ = env.param_redraw()
    assert lo_[0] == np.float32(9.0) and hi_[5] == np.float32(0.03) and lo_[1:5] == tuple(d[1:5]) == hi_[1:5]
    # set_params(rows) keeps the ranges, set_params(None) clears them with the rows
    env.set_params(rows)
    assert env.param_redraw() is not None
    env.set_params(None)
    assert env.param_redraw() is None
    assert lib.mgym_checkpoint_size(env._h) == size
    env.close()
    acro = gym.GpuVecEnv(4, 128)
    with pytest.raises(MgymError, match="no per-env parameters"):
        acro.set_param_redraw([], [])
    assert acro.param_redraw() is None
    acro.close()


def test_cpp_host_layer(gym):
    """set_param_redraw / param_redraw / clear_param_redraw of include/mgym.hpp (tests/cpp/test_param_redraw.cpp)."""
    src = os.path.join(ROOT, "tests", "cpp", "test_param_redraw.cpp")
    pkg = os.path.join(ROOT, "modurl_gym_b200")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "test_param_redraw")
        r = subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-Wall", f"-I{cuda}/include", "-o", exe,
                            src, f"-L{pkg}", "-lmgym", f"-L{cuda}/lib64", "-lcudart", f"-Wl,-rpath,{pkg}",
                            f"-Wl,-rpath,{cuda}/lib64"], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ALL OK" in out.stdout, out.stdout + out.stderr
    assert out.stdout.count("ok ") >= 8
