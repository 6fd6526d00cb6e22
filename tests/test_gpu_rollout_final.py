"""Fused rollouts that keep the observation every finished episode ended on (mgym_rollout_final,
GpuVecEnv.rollout(want_final_obs=True)): only finished envs are written, bit-exact to the final observations of the
oracle's step driver, and everything else the rollout does is bit-identical to mgym_rollout."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import redraw_oracle as ro
from helpers import KIND_NAMES, assert_bit_equal, bits, random_actions, random_states
from oracle import oracle as o

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENTINEL = 0x7FA5A5A5  # a NaN with a payload no kernel produces: "not written"
K_OF = {0: 300, 1: 200, 2: 200, 3: 210, 4: 120}  # long enough that many envs finish
LIMIT = {0: 500, 1: 0, 2: 999, 3: 200, 4: 500}   # time limits; MountainCar-v0 has none
SIZES = [4096, 4000, 4099]  # FULL rollout form, V = 4 without FULL, scalar lanes


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


def sentinel(K, od, n):
    return torch.full((K, od, n), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)


def ages(rng, kind, n):
    """Episode step counts near the kind's time limit, so that truncations happen inside a short rollout."""
    lim = LIMIT[kind]
    return (rng.integers(0, lim - 10, n) if lim else np.zeros(n)).astype(np.int32)


def start(env, ref, rng, kind, n):
    """env and oracle in the same random state at step index 0."""
    st, steps = random_states(rng, kind, n), ages(rng, kind, n)
    env.reset()
    env.set_state(dev(st), dev(steps))
    if ref is not None:
        ref.state[:], ref.steps[:], ref.sbt[:] = st, steps, 0
    return st, steps


def oracle_steps(ref, actions):
    """K oracle steps with final observations: (obs, reward, flags, final) stacked time-major."""
    outs = [ref.step(a, want_final_obs=True) for a in actions]
    return tuple(np.stack([x[i] for x in outs]) for i in range(4))


def device_policy_actions(gym, kind, n, K, seed, **kw):
    """What mgym_sample_actions gives at step indices 0..K-1 (a handle of the same seed and env_index_base)."""
    src = gym.GpuVecEnv(kind, n, seed=seed, **kw)
    src.reset()
    acts = []
    for _ in range(K):
        a = src.sample_actions()
        acts.append(host(a))
        src.step(a)
    src.close()
    return np.stack(acts)


def check_final(final, flags, want, what):
    """Where flags != 0 the final observation is the oracle's, bit for bit; everywhere else the sentinel."""
    got = bits(host(final))
    hit = np.broadcast_to((flags != 0)[:, None, :], got.shape)
    assert hit.any(), f"{what}: no env finished"
    assert_bit_equal(got[hit], bits(want)[hit], f"{what}: final obs of finished envs")
    assert (got[~hit] == SENTINEL).all(), f"{what}: {int((got[~hit] != SENTINEL).sum())} entries of live envs written"


def rollout_final(env, K, actions=None, **kw):
    final = sentinel(K, env.obs_dim, env.num_envs)
    out, fin = env.rollout(K, actions, final_obs=final, want_final_obs=True, **kw)
    assert fin is final
    return out, final


@pytest.mark.parametrize("kind", range(5))
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("policy", ["caller", "device"])
def test_final_obs_match_oracle(gym, kind, n, policy):
    K, seed = K_OF[kind], 40 + kind
    rng = np.random.default_rng(1000 * kind + n)
    env = gym.GpuVecEnv(kind, n, seed=seed)
    ref = o.VecState(kind, n, auto_reset=1, seed=seed)
    ref.reset()
    start(env, ref, rng, kind, n)
    acts = random_actions(rng, kind, (K, n)) if policy == "caller" else device_policy_actions(gym, kind, n, K, seed)
    out, final = rollout_final(env, K, dev(acts) if policy == "caller" else None)
    obs, rew, flg, fin = oracle_steps(ref, acts)
    name = f"{KIND_NAMES[kind]} n={n} {policy}"
    assert_bit_equal(host(out.flags), flg, f"{name} flags")
    assert_bit_equal(host(out.obs), obs, f"{name} obs")
    assert_bit_equal(host(out.reward), rew, f"{name} reward")
    check_final(final, flg, fin, name)
    if kind != 1:
        assert (flg != 0).sum() > n // 8
    env.close()


@pytest.mark.parametrize("kind", range(5))
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("policy", ["caller", "device"])
def test_everything_else_is_mgym_rollout(gym, kind, n, policy):
    """A twin through mgym_rollout and a third handle through mgym_rollout_final(final_obs_traj = NULL): the same
    trajectories, done count, state, counters, statistics (running returns included) and step index."""
    K = K_OF[kind] // 2
    rng = np.random.default_rng(2000 * kind + n)
    es = [gym.GpuVecEnv(kind, n, seed=3, track_returns=kind in (2, 3)) for _ in range(3)]
    st, steps = dev(random_states(rng, kind, n)), dev(ages(rng, kind, n))
    for e in es:
        e.reset()
        e.set_state(st, steps)
    a = dev(random_actions(rng, kind, (K, n))) if policy == "caller" else None
    outs = [es[0].rollout(K, a), rollout_final(es[1], K, a)[0]]
    obs = torch.empty((K, es[2].obs_dim, n), device="cuda")
    rew, flg = torch.empty((K, n), device="cuda"), torch.empty((K, n), dtype=torch.uint8, device="cuda")
    dc = torch.zeros(1, dtype=torch.int64, device="cuda")
    lib, ptr = es[2]._lib, lambda t: C.c_void_p(t.data_ptr())
    assert lib.mgym_rollout_final(es[2]._h, K, None if a is None else ptr(a), ptr(obs), ptr(rew), ptr(flg), None,
                                  ptr(dc), es[2]._stream()) == 0
    outs.append((obs, rew, flg, dc))
    for out in outs[1:]:
        assert all(same(x, y) for x, y in zip(outs[0], out))
    assert int(outs[0][3].item()) > 0
    for e in es[1:]:
        assert all(same(x, y) for x, y in zip(es[0].get_state(), e.get_state()))
        assert e.stats() == es[0].stats() and e.step_index == es[0].step_index == K
    for e in es:
        e.close()


def ranges(gym, kind, spread=0.2):
    d = np.asarray(gym.GpuVecEnv.param_defaults(kind), dtype=np.float32)
    return d, d * np.float32(1 - spread), d * np.float32(1 + spread)


@pytest.mark.parametrize("kind", [0, 1, 2, 3])
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("mode", ["rows", "redraw"])
def test_parameters_and_redraw_match_oracle(gym, kind, n, mode):
    """Random per-env rows (PARAMS forms), optionally with +-20 % redraw ranges (REDRAW forms): the finishing step
    runs on the old parameters, so the final observation is the one they produced; the rows after the rollout are
    the oracle's."""
    K, seed = K_OF[kind] // 2, 60 + kind
    rng = np.random.default_rng(3000 * kind + n)
    d, low, high = ranges(gym, kind)
    env = gym.GpuVecEnv(kind, n, seed=seed)
    ref = ro.VecState(kind, n, auto_reset=1, seed=seed)
    ref.reset()
    start(env, ref, rng, kind, n)
    rows = (d[:, None] * rng.uniform(0.8, 1.2, (len(d), n))).astype(np.float32)
    env.set_params(dev(rows))
    ref.set_params(rows)
    if mode == "redraw":
        env.set_param_redraw(low, high)
        ref.set_param_redraw(low, high)
    acts = random_actions(rng, kind, (K, n))
    out, final = rollout_final(env, K, dev(acts))
    obs, rew, flg, fin = oracle_steps(ref, acts)
    assert_bit_equal(host(out.flags), flg, "flags")
    assert_bit_equal(host(out.obs), obs, "obs")
    check_final(final, flg, fin, f"{KIND_NAMES[kind]} n={n} {mode}")
    assert_bit_equal(host(env.get_params()), ref.params, "rows after the rollout")
    assert_bit_equal(host(env.get_state()[0]), ref.state, "state after the rollout")
    env.close()


@pytest.mark.parametrize("kind", range(5))
def test_reset_pool(gym, kind):
    """Pool resets replace reset states only.  MountainCar's pool holds positions far outside the track, which
    break the invariant of its trusted loop (the kernel re-tests it after pool resets)."""
    n, P, K, seed = 4096, 257, K_OF[kind] // 2, 80 + kind
    rng = np.random.default_rng(4000 + kind)
    pool = random_states(rng, kind, P)
    if kind in (1, 2):
        pool[0, rng.random(P) < 0.1] = np.float32(1e10)
    kw = {"max_episode_steps": 3} if kind == 1 else {}  # every MountainCar env resets from the pool, often
    env = gym.GpuVecEnv(kind, n, seed=seed, **kw)
    ref = o.VecState(kind, n, auto_reset=1, seed=seed, **kw)
    env.set_reset_pool(dev(pool))
    ref.set_reset_pool(pool)
    ref.reset()
    start(env, ref, rng, kind, n)
    for chunk in range(2):
        acts = random_actions(rng, kind, (K, n))
        out, final = rollout_final(env, K, dev(acts))
        obs, rew, flg, fin = oracle_steps(ref, acts)
        assert_bit_equal(host(out.flags), flg, f"flags chunk {chunk}")
        assert_bit_equal(host(out.obs), obs, f"obs chunk {chunk}")
        check_final(final, flg, fin, f"{KIND_NAMES[kind]} pool chunk {chunk}")
    assert_bit_equal(host(env.get_state()[0]), ref.state, "state")
    env.close()


@pytest.mark.parametrize("kind", range(5))
@pytest.mark.parametrize("n", [4096, 4099])
def test_k_steps_equal_one_rollout(gym, kind, n):
    """K x mgym_step(final_obs_out) and one mgym_rollout_final(K) with the device policy: the same final
    observations where an env finished, and the same handle afterwards."""
    K = K_OF[kind] // 2
    rng = np.random.default_rng(5000 * kind + n)
    a, b = gym.GpuVecEnv(kind, n, seed=17), gym.GpuVecEnv(kind, n, seed=17)
    st, steps = dev(random_states(rng, kind, n)), dev(ages(rng, kind, n))
    for e in (a, b):
        e.reset()
        e.set_state(st, steps)
    flags, finals = [], []
    for _ in range(K):
        info, fin = a.step(a.sample_actions(), want_final_obs=True)
        flags.append(info.flags.clone())
        finals.append(fin)
    out, final = rollout_final(b, K)
    flg = torch.stack(flags)
    assert same(out.flags, flg)
    check_final(final, host(flg), host(torch.stack(finals)), f"{KIND_NAMES[kind]} n={n}")
    assert all(same(x, y) for x, y in zip(a.get_state(), b.get_state()))
    assert a.stats() == b.stats()
    a.close(), b.close()


@pytest.mark.parametrize("kind", range(5))
def test_two_shards_equal_one_handle(gym, kind):
    n, K = 8192, K_OF[kind] // 2
    h = n // 2
    rng = np.random.default_rng(6000 + kind)
    whole = gym.GpuVecEnv(kind, n, seed=12)
    shards = [gym.GpuVecEnv(kind, h, seed=12, env_index_base=i * h) for i in range(2)]
    st, steps = dev(random_states(rng, kind, n)), dev(ages(rng, kind, n))
    for e, sl in [(whole, slice(0, n)), (shards[0], slice(0, h)), (shards[1], slice(h, n))]:
        e.reset()
        e.set_state(st[:, sl].contiguous(), steps[sl].contiguous())
    ow, fw = rollout_final(whole, K)  # device policy: keyed by the global env index
    parts = [rollout_final(s, K) for s in shards]
    assert same(torch.cat([p[0].flags for p in parts], 1), ow.flags)
    assert same(torch.cat([p[1] for p in parts], 2), fw)
    assert int((ow.flags != 0).sum().item()) > 0
    for e in [whole] + shards:
        e.close()


def test_graph_replay_matches_eager(gym):
    """[sample_actions, rollout_final] captured on a device-clock handle and replayed equals the eager calls of a
    default handle."""
    n, K, R, kind = 4096, 16, 6, 0
    a = gym.GpuVecEnv(kind, n, seed=9)
    b = gym.GpuVecEnv(kind, n, seed=9, graph_capturable=True)
    a.reset(), b.reset()
    acts = torch.zeros((K, n), dtype=torch.uint8, device="cuda")  # row 0 from sample_actions, the others 0
    obs = torch.empty((K, 4, n), device="cuda")
    rew = torch.empty((K, n), device="cuda")
    flg = torch.empty((K, n), dtype=torch.uint8, device="cuda")
    fin = sentinel(K, 4, n)
    b.sample_actions(out=acts[0])  # warm-up eager call (step index 0 -> K), like the default handle's below
    b.rollout(K, acts, obs=obs, reward=rew, flags=flg, final_obs=fin, want_final_obs=True)
    acts_a = torch.zeros_like(acts)
    acts_a[0] = a.sample_actions()
    a.rollout(K, acts_a, want_final_obs=True)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        b.sample_actions(out=acts[0])
        b.rollout(K, acts, obs=obs, reward=rew, flags=flg, final_obs=fin, want_final_obs=True, count_done=False)
    for r in range(R):
        fin.view(torch.int32).fill_(SENTINEL)
        graph.replay()
        acts_a = acts.clone()
        acts_a[0] = a.sample_actions()
        out, final = rollout_final(a, K, acts_a)
        assert same(acts_a, acts), f"replay {r} actions"
        assert same(out.obs, obs) and same(out.reward, rew) and same(out.flags, flg), f"replay {r}"
        assert same(final, fin), f"replay {r} final obs"
        assert int((flg != 0).sum().item()) > 0 or r < 2
    assert b.step_index == a.step_index == (R + 1) * K
    a.close(), b.close()


def test_rejections_leave_everything_untouched(gym):
    n, K = 4096, 8
    lib = gym.load_library()
    man = gym.GpuVecEnv(0, n, auto_reset=False, seed=1)
    man.reset()
    fin = sentinel(K, 4, n)
    with pytest.raises(gym.MgymError):
        man.rollout(K, final_obs=fin, want_final_obs=True)
    assert man.step_index == 0
    man.rollout(K)  # without final observations a manual handle rolls out as before
    assert man.step_index == K
    man.close()

    env = gym.GpuVecEnv(0, n, seed=2, validate_actions=True)
    env.reset()
    before = [x.clone() for x in env.get_state()]
    obs = torch.empty((K, 4, n), device="cuda")
    ptr = lambda t: C.c_void_p(t.data_ptr())
    rc = lib.mgym_rollout_final(env._h, K, None, ptr(obs), None, None, ptr(obs), None, env._stream())
    assert rc == -1  # MGYM_ERR_BAD_ARGUMENT: final_obs_traj == obs_traj
    bad = torch.zeros((K, n), dtype=torch.uint8, device="cuda")
    bad[3, 77] = 2  # not in Discrete(2)
    with pytest.raises(gym.InvalidActionError):
        env.rollout(K, bad, final_obs=fin, want_final_obs=True)
    assert lib.mgym_rollout_final(env._h, 0, None, None, None, None, ptr(fin), None, env._stream()) == 0  # K = 0
    torch.cuda.synchronize()
    assert (fin.view(torch.int32) == SENTINEL).all()
    assert env.step_index == 0 and env.stats().episodes == 0
    assert all(same(x, y) for x, y in zip(before, env.get_state()))
    env.close()


def test_full_size_cartpole(gym):
    """2^24 envs, one 32-step launch with the device policy; three windows replayed by the oracle."""
    n, K, seed, kind = 1 << 24, 32, 0xF1A1, 0
    env = gym.GpuVecEnv(kind, n, seed=seed)
    env.reset()
    out, final = rollout_final(env, K)
    torch.cuda.synchronize()
    for (lo, hi) in [(0, 1024), (n // 2 - 512 + 4, n // 2 + 512 + 4), (n - 1024, n)]:
        ref = o.VecState(kind, hi - lo, auto_reset=1, seed=seed, env_index_base=lo)
        ref.reset()
        acts = np.array([[o.sample_action(kind, seed, lo + i, t) for i in range(hi - lo)] for t in range(K)],
                        dtype=np.uint8)
        obs, rew, flg, fin = oracle_steps(ref, acts)
        assert_bit_equal(host(out.flags[:, lo:hi]), flg, f"flags [{lo},{hi})")
        check_final(final[:, :, lo:hi], flg, fin, f"window [{lo},{hi})")
    assert int(out.done_count.item()) == int((out.flags != 0).sum().item()) > 0
    env.close()


def test_iter_rollout_reuses_one_final_buffer(gym):
    n, T, chunk, kind = 4096, 230, 32, 3  # Pendulum truncates at 200; the last launch is a partial chunk
    a, b = gym.GpuVecEnv(kind, n, seed=4), gym.GpuVecEnv(kind, n, seed=4)
    a.reset(), b.reset()
    bufs, hits = set(), 0
    for first, (out, final) in a.iter_rollout(T, chunk=chunk, want_final_obs=True):
        k = out.flags.shape[0]
        want, wfin = b.rollout(k, want_final_obs=True)
        hit = (want.flags != 0).unsqueeze(1).expand_as(wfin)
        assert same(out.flags, want.flags) and same(final[hit], wfin[hit]), first
        bufs.add(final.data_ptr())
        hits += int((out.flags != 0).sum().item())
    assert len(bufs) == 1 and hits >= n
    a.close(), b.close()


def test_cpp_host_layer(gym):
    """GpuVecEnv::rollout_final of include/mgym.hpp (tests/cpp/test_rollout_final.cpp)."""
    src = os.path.join(ROOT, "tests", "cpp", "test_rollout_final.cpp")
    pkg = os.path.join(ROOT, "modurl_gym_b200")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "test_rollout_final")
        r = subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-Wall", f"-I{cuda}/include", "-o", exe,
                            src, f"-L{pkg}", "-lmgym", f"-L{cuda}/lib64", "-lcudart", f"-Wl,-rpath,{pkg}",
                            f"-Wl,-rpath,{cuda}/lib64"], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ALL OK" in out.stdout, out.stdout + out.stderr
    assert out.stdout.count("ok ") >= 4
