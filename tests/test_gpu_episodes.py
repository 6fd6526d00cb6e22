"""Per-episode returns and lengths from the step and the fused rollout (mgym_step_episodes, mgym_rollout_episodes,
GpuVecEnv.step / rollout(want_episodes=True)): written only where an env finished, bit-exact to the oracle's
episode drivers, and everything else each call does is bit-identical to mgym_step / mgym_rollout / mgym_rollout_final."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import episodes_oracle as eo
from helpers import KIND_NAMES, assert_bit_equal, bits, random_actions, random_states
from oracle import oracle as o

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RET_SENTINEL = 0x7FA5A5A5  # a NaN with a payload no kernel produces: "not written"
LEN_SENTINEL = 0xDEADBEEF
K_OF = {0: 300, 1: 200, 2: 200, 3: 210, 4: 120}  # long enough that many envs finish
LIMIT = {0: 500, 1: 0, 2: 999, 3: 200, 4: 500}   # time limits; MountainCar-v0 has none
SIZES = [4096, 4000, 4099]  # FULL rollout form / TMA step, V = 4 without FULL / TMA head + LDG tail, scalar lanes
TRACK = {2: True, 3: True}  # the kinds whose return is a running return need track_returns for ep_return


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


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def same(x, y):
    if x is None or y is None:
        return x is y
    if x.dtype == torch.float32:
        x, y = x.view(torch.int32), y.view(torch.int32)
    return torch.equal(x, y)


def sentinels(shape):
    ret = torch.full(shape, RET_SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)
    length = torch.full(shape, LEN_SENTINEL - (1 << 32), dtype=torch.int32, device="cuda")
    return ret, length


def ages(rng, kind, n):
    """Episode step counts near the kind's time limit, so that truncations happen inside a short rollout."""
    lim = LIMIT[kind]
    return (rng.integers(0, lim - 10, n) if lim else np.zeros(n)).astype(np.int32)


def make(gym, kind, n, seed, **kw):
    return gym.GpuVecEnv(kind, n, seed=seed, track_returns=TRACK.get(kind, False), **kw)


def start(env, ref, rng, kind, n):
    """env and oracle in the same random state, episodes of random ages, at step index 0."""
    st, steps = random_states(rng, kind, n), ages(rng, kind, n)
    env.reset()
    env.set_state(dev(st), dev(steps))
    if ref is not None:
        ref.state[:], ref.steps[:], ref.sbt[:], ref.ep_return[:] = st, steps, 0, 0.0
    return dev(st), dev(steps)


def check_episodes(ret, length, flags, want_ret, want_len, what):
    """Where flags != 0 the outputs are the oracle's, bit for bit; everywhere else the sentinels."""
    got_r, got_l = bits(host(ret)), host(length).view(np.uint32)
    hit = flags != 0
    assert hit.any(), f"{what}: no env finished"
    assert_bit_equal(got_l[hit], want_len[hit], f"{what}: ep_length of finished envs")
    assert_bit_equal(got_r[hit], bits(want_ret)[hit], f"{what}: ep_return of finished envs")
    assert (got_r[~hit] == RET_SENTINEL).all(), f"{what}: ep_return of {int((got_r[~hit] != RET_SENTINEL).sum())} live envs"
    assert (got_l[~hit] == LEN_SENTINEL).all(), f"{what}: ep_length of {int((got_l[~hit] != LEN_SENTINEL).sum())} live envs"


def step_raw(env, actions, episodes=None, final=False):
    """One mgym_step (episodes None) or mgym_step_episodes(ret, length) into new buffers: (obs, reward, flags, final)."""
    n = env.num_envs
    obs = torch.empty((env.obs_dim, n), device="cuda")
    rew, flg = torch.empty(n, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")
    fin = torch.empty((env.obs_dim, n), device="cuda") if final else None
    if episodes is None:
        rc = env._lib.mgym_step(env._h, ptr(actions), ptr(obs), ptr(rew), ptr(flg), ptr(fin), env._stream())
    else:
        rc = env._lib.mgym_step_episodes(env._h, ptr(actions), ptr(obs), ptr(rew), ptr(flg), ptr(fin),
                                         ptr(episodes[0]), ptr(episodes[1]), env._stream())
    assert rc == 0, env._lib.mgym_last_error()
    return obs, rew, flg, fin


def rollout_e(env, K, actions=None, **kw):
    ret, length = sentinels((K, env.num_envs))
    out, ep = env.rollout(K, actions, ep_return=ret, ep_length=length, want_episodes=True, **kw)
    assert ep.ret is ret and ep.length is length
    return out, ep


def run_both(env, ref, kind, K, acts, via):
    """K steps of `via` ("rollout" or "step") on the device and the oracle: device (flags, ret, length) and the
    oracle's (flags, ret, length), time-major.  acts None: the device policy (the rollout and the oracle's rollout
    driver draw the same Philox actions; the step takes what mgym_sample_actions gives)."""
    if via == "rollout":
        out, ep = rollout_e(env, K, None if acts is None else dev(acts))
        want = ref.rollout_e(K, acts)
        return host(out.flags), ep.ret, ep.length, want[2], want[4], want[5]
    flags, rets, lens, wf, wr, wl = [], [], [], [], [], []
    for k in range(K):
        a = env.sample_actions() if acts is None else dev(acts[k])
        ret, length = sentinels((env.num_envs,))
        _, _, flg, _ = step_raw(env, a, (ret, length))
        flags.append(host(flg)), rets.append(ret), lens.append(length)
        w = ref.step_e(host(a))
        wf.append(w[2]), wr.append(w[3]), wl.append(w[4])
    return np.stack(flags), torch.stack(rets), torch.stack(lens), np.stack(wf), np.stack(wr), np.stack(wl)


@pytest.mark.parametrize("kind", range(5))
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("policy", ["caller", "device"])
@pytest.mark.parametrize("via", ["rollout", "step"])
def test_episodes_match_oracle(gym, kind, n, policy, via):
    K, seed = K_OF[kind] // (1 if via == "rollout" else 2), 40 + kind
    rng = np.random.default_rng(1000 * kind + n)
    env = make(gym, kind, n, seed)
    ref = eo.VecState(kind, n, auto_reset=1, seed=seed)
    ref.reset()
    start(env, ref, rng, kind, n)
    acts = random_actions(rng, kind, (K, n)) if policy == "caller" else None
    flg, ret, length, wflg, wret, wlen = run_both(env, ref, kind, K, acts, via)
    name = f"{KIND_NAMES[kind]} n={n} {policy} {via}"
    assert_bit_equal(flg, wflg, f"{name} flags")
    check_episodes(ret, length, flg, wret, wlen, name)
    if kind in (2, 3, 4):  # episodes long enough that the ages force truncations
        assert (flg & o.FLAG_TRUNCATED).any(), f"{name}: no truncation"
    assert_bit_equal(host(env.get_state()[0]), ref.state, f"{name} state")
    env.close()


def ranges(gym, kind, spread=0.2):
    d = np.asarray(gym.GpuVecEnv.param_defaults(kind), dtype=np.float32)
    return d, d * np.float32(1 - spread), d * np.float32(1 + spread)


@pytest.mark.parametrize("kind", [0, 1, 2, 3])
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("mode", ["rows", "redraw"])
@pytest.mark.parametrize("via", ["rollout", "step"])
def test_parameters_and_redraw_match_oracle(gym, kind, n, mode, via):
    """Random per-env rows (PARAMS forms), optionally with +-20 % redraw ranges (REDRAW forms): the outputs and the
    rows afterwards are the oracle's."""
    K, seed = K_OF[kind] // 2, 60 + kind
    rng = np.random.default_rng(3000 * kind + n)
    d, low, high = ranges(gym, kind)
    env = make(gym, kind, n, seed)
    ref = eo.VecState(kind, n, auto_reset=1, seed=seed)
    ref.reset()
    start(env, ref, rng, kind, n)
    rows = (d[:, None] * rng.uniform(0.8, 1.2, (len(d), n))).astype(np.float32)
    env.set_params(dev(rows))
    ref.set_params(rows)
    if mode == "redraw":
        env.set_param_redraw(low, high)
        ref.set_param_redraw(low, high)
    acts = random_actions(rng, kind, (K, n))
    flg, ret, length, wflg, wret, wlen = run_both(env, ref, kind, K, acts, via)
    name = f"{KIND_NAMES[kind]} n={n} {mode} {via}"
    assert_bit_equal(flg, wflg, f"{name} flags")
    check_episodes(ret, length, flg, wret, wlen, name)
    assert_bit_equal(host(env.get_params()), ref.params, f"{name} rows")
    assert_bit_equal(host(env.get_state()[0]), ref.state, f"{name} state")
    env.close()


def twins(gym, kind, n, rng, count, **kw):
    es = [make(gym, kind, n, 3, **kw) for _ in range(count)]
    st, steps = dev(random_states(rng, kind, n)), dev(ages(rng, kind, n))
    for e in es:
        e.reset()
        e.set_state(st, steps)
    return es


def same_handles(a, b, what):
    assert all(same(x, y) for x, y in zip(a.get_state(), b.get_state())), f"{what}: state"
    assert a.stats() == b.stats(), f"{what}: statistics"
    assert a.step_index == b.step_index, f"{what}: step index"


@pytest.mark.parametrize("kind", range(5))
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("final", [False, True], ids=["no-final", "final"])
@pytest.mark.parametrize("rows", ["plain", "redraw"])
def test_everything_else_is_the_plain_call(gym, kind, n, final, rows):
    """A twin through mgym_rollout (mgym_rollout_final with final) / mgym_step and one through the episode calls: the
    same outputs, done count, state, counters, statistics (running returns included), rows and step index."""
    if rows == "redraw" and kind == 4:
        pytest.skip("Acrobot has no parameters")
    K = K_OF[kind] // 4
    rng = np.random.default_rng(2000 * kind + n)
    es = twins(gym, kind, n, rng, 4)
    if rows == "redraw":
        d, low, high = ranges(gym, kind)
        for e in es:
            e.set_params(dev(np.repeat(d[:, None], n, axis=1)))
            e.set_param_redraw(low, high)
    a = dev(random_actions(rng, kind, (K, n)))
    # rollout: plain call against the episode call
    if final:
        fa, fb = torch.zeros((K, es[0].obs_dim, n), device="cuda"), torch.zeros((K, es[0].obs_dim, n), device="cuda")
        oa, fa = es[0].rollout(K, a, final_obs=fa, want_final_obs=True)
        ob, fb, ep = es[1].rollout(K, a, final_obs=fb, want_final_obs=True, want_episodes=True)
        assert same(fa, fb)
    else:
        oa = es[0].rollout(K, a)
        ob, ep = es[1].rollout(K, a, want_episodes=True)
    assert all(same(x, y) for x, y in zip(oa, ob)) and int(oa.done_count.item()) > 0
    same_handles(es[0], es[1], "rollout")
    if rows == "redraw":
        assert same(es[0].get_params(), es[1].get_params())
    # step: K plain steps against K episode steps
    for k in range(K):
        ra = step_raw(es[2], a[k], final=final)
        rb = step_raw(es[3], a[k], sentinels((n,)), final=final)
        assert all(same(x, y) for x, y in zip(ra, rb)), f"step {k}"
    same_handles(es[2], es[3], "step")
    if rows == "redraw":
        assert same(es[2].get_params(), es[3].get_params())
    for e in es:
        e.close()


@pytest.mark.parametrize("kind", range(5))
@pytest.mark.parametrize("n", [4096, 4099])
def test_k_steps_equal_one_rollout(gym, kind, n):
    """K x mgym_step_episodes and one mgym_rollout_episodes(K) with the device policy: the same outputs where an env
    finished, and the same handle afterwards."""
    K = K_OF[kind] // 2
    rng = np.random.default_rng(5000 * kind + n)
    a, b = twins(gym, kind, n, rng, 2)
    flags, rets, lens = [], [], []
    for _ in range(K):
        ret, length = sentinels((n,))
        _, _, flg, _ = step_raw(a, a.sample_actions(), (ret, length))
        flags.append(flg), rets.append(ret), lens.append(length)
    out, ep = rollout_e(b, K)
    assert same(out.flags, torch.stack(flags))
    assert same(ep.ret, torch.stack(rets)) and same(ep.length, torch.stack(lens))
    assert int((out.flags != 0).sum().item()) > 0
    same_handles(a, b, f"{KIND_NAMES[kind]} n={n}")
    a.close(), b.close()


@pytest.mark.parametrize("kind", range(5))
def test_two_shards_equal_one_handle(gym, kind):
    n, K = 8192, K_OF[kind] // 2
    h = n // 2
    rng = np.random.default_rng(6000 + kind)
    whole = make(gym, kind, n, 12)
    shards = [make(gym, kind, h, 12, env_index_base=i * h) for i in range(2)]
    st, steps = dev(random_states(rng, kind, n)), dev(ages(rng, kind, n))
    for e, sl in [(whole, slice(0, n)), (shards[0], slice(0, h)), (shards[1], slice(h, n))]:
        e.reset()
        e.set_state(st[:, sl].contiguous(), steps[sl].contiguous())
    ow, ew = rollout_e(whole, K)  # device policy: keyed by the global env index
    parts = [rollout_e(s, K) for s in shards]
    assert same(torch.cat([p[0].flags for p in parts], 1), ow.flags)
    assert same(torch.cat([p[1].ret for p in parts], 1), ew.ret)
    assert same(torch.cat([p[1].length for p in parts], 1), ew.length)
    assert int((ow.flags != 0).sum().item()) > 0
    for e in [whole] + shards:
        e.close()


def test_graph_replay_matches_eager(gym):
    """[sample_actions, rollout_episodes] and [step_episodes] captured on a device-clock handle and replayed equal the
    eager calls of a default handle."""
    n, K, R, kind = 4096, 16, 6, 0
    a = gym.GpuVecEnv(kind, n, seed=9)
    b = gym.GpuVecEnv(kind, n, seed=9, graph_capturable=True)
    a.reset(), b.reset()
    acts = torch.zeros((K, n), dtype=torch.uint8, device="cuda")  # row 0 from sample_actions, the others 0
    obs = torch.empty((K, 4, n), device="cuda")
    rew = torch.empty((K, n), device="cuda")
    flg = torch.empty((K, n), dtype=torch.uint8, device="cuda")
    ret, length = sentinels((K, n))
    b.sample_actions(out=acts[0])  # warm-up eager call (step index 0 -> K), like the default handle's below
    b.rollout(K, acts, obs=obs, reward=rew, flags=flg, ep_return=ret, ep_length=length, want_episodes=True)
    acts_a = torch.zeros_like(acts)
    acts_a[0] = a.sample_actions()
    a.rollout(K, acts_a, want_episodes=True)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        b.sample_actions(out=acts[0])
        b.rollout(K, acts, obs=obs, reward=rew, flags=flg, ep_return=ret, ep_length=length, want_episodes=True,
                  count_done=False)
    for r in range(R):
        ret.view(torch.int32).fill_(RET_SENTINEL)
        length.fill_(LEN_SENTINEL - (1 << 32))
        graph.replay()
        acts_a = acts.clone()
        acts_a[0] = a.sample_actions()
        out, ep = rollout_e(a, K, acts_a)
        assert same(acts_a, acts), f"replay {r} actions"
        assert same(out.obs, obs) and same(out.reward, rew) and same(out.flags, flg), f"replay {r}"
        assert same(ep.ret, ret) and same(ep.length, length), f"replay {r} episodes"
        assert int((flg != 0).sum().item()) > 0 or r < 2
    assert b.step_index == a.step_index == (R + 1) * K
    # the per-call step
    sa = torch.empty(n, dtype=torch.uint8, device="cuda")
    sret, slen = sentinels((n,))
    obs1, rew1 = torch.empty((4, n), device="cuda"), torch.empty(n, device="cuda")
    flg1 = torch.empty(n, dtype=torch.uint8, device="cuda")

    def step_b():
        b.sample_actions(out=sa)
        assert b._lib.mgym_step_episodes(b._h, ptr(sa), ptr(obs1), ptr(rew1), ptr(flg1), None, ptr(sret), ptr(slen),
                                         b._stream()) == 0

    step_b()  # warm-up
    ea, eb = sentinels((n,))
    step_raw(a, a.sample_actions(), (ea, eb))
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step_b()
    hits = 0
    for r in range(3 * R):
        sret.view(torch.int32).fill_(RET_SENTINEL)
        slen.fill_(LEN_SENTINEL - (1 << 32))
        graph.replay()
        ea, eb = sentinels((n,))
        o_, r_, f_, _ = step_raw(a, a.sample_actions(), (ea, eb))
        assert same(o_, obs1) and same(r_, rew1) and same(f_, flg1), f"step replay {r}"
        assert same(ea, sret) and same(eb, slen), f"step replay {r} episodes"
        hits += int((f_ != 0).sum().item())
    assert hits > 0 and b.step_index == a.step_index
    same_handles(a, b, "after the replays")
    a.close(), b.close()


def test_rejections_leave_everything_untouched(gym):
    n, K = 4096, 8
    lib = gym.load_library()

    def untouched(env, ret, length, before, what):
        torch.cuda.synchronize()
        assert (ret.view(torch.int32) == RET_SENTINEL).all() and (length == LEN_SENTINEL - (1 << 32)).all(), what
        assert env.step_index == 0 and env.stats().episodes == 0, what
        assert all(same(x, y) for x, y in zip(before, env.get_state())), what

    def refused(env, ret, length, rollout=True, final=None, obs=None, actions=None):
        if rollout:
            return lib.mgym_rollout_episodes(env._h, K, ptr(actions), ptr(obs), None, None, ptr(final), ptr(ret),
                                             ptr(length), None, env._stream())
        a = actions if actions is not None else torch.zeros(n, dtype=env.action_dtype, device="cuda")
        return lib.mgym_step_episodes(env._h, ptr(a), None, None, None, None, ptr(ret), ptr(length), env._stream())

    # a manual-mode handle: refused for both calls, and the plain calls still run
    man = gym.GpuVecEnv(0, n, auto_reset=False, seed=1)
    man.reset()
    for rollout in (True, False):
        r, l_ = sentinels((K, n) if rollout else (n,))
        before = [x.clone() for x in man.get_state()]
        assert refused(man, r, l_, rollout) == -1 and b"auto_reset" in lib.mgym_last_error()
        assert refused(man, None, l_, rollout) == -1
        untouched(man, r, l_, before, f"manual rollout={rollout}")
    man.rollout(K)
    assert man.step_index == K
    man.close()

    # Pendulum without running returns: ep_return refused (the message names track_returns), ep_length alone runs
    for kw in ({"track_returns": False}, {"track_returns": True, "track_stats": False}):
        pen = gym.GpuVecEnv(3, n, seed=2, **kw)
        pen.reset()
        for rollout in (True, False):
            r, l_ = sentinels((K, n) if rollout else (n,))
            before = [x.clone() for x in pen.get_state()]
            assert refused(pen, r, l_, rollout) == -1 and b"track_returns" in lib.mgym_last_error()
            assert refused(pen, r, None, rollout) == -1
            untouched(pen, r, l_, before, f"Pendulum {kw} rollout={rollout}")
        r, l_ = sentinels((K, n))
        assert refused(pen, None, l_) == 0
        pen.close()

    env = gym.GpuVecEnv(0, n, seed=2, validate_actions=True)
    env.reset()
    before = [x.clone() for x in env.get_state()]
    for rollout in (True, False):
        shape = (K, n) if rollout else (n,)
        r, l_ = sentinels(shape)
        # the same buffer for both outputs
        assert refused(env, r, r.view(torch.int32), rollout) == -1 and b"different" in lib.mgym_last_error()
        # a bad batch under validate_actions
        bad = torch.zeros(shape, dtype=torch.uint8, device="cuda")
        bad.view(-1)[77] = 2  # not in Discrete(2)
        assert refused(env, r, l_, rollout, actions=bad) == -4  # MGYM_ERR_INVALID_ACTION
        untouched(env, r, l_, before, f"CartPole rollout={rollout}")
    r, l_ = sentinels((K, n))
    obs = torch.empty((K, 4, n), device="cuda")
    assert refused(env, r, l_, final=obs, obs=obs) == -1  # final_obs_traj == obs_traj
    assert lib.mgym_rollout_episodes(env._h, 0, None, None, None, None, None, ptr(r), ptr(l_), None,
                                     env._stream()) == 0  # K = 0
    untouched(env, r, l_, before, "CartPole final == obs, K = 0")
    with pytest.raises(gym.InvalidActionError):
        env.rollout(K, torch.full((K, n), 2, dtype=torch.uint8, device="cuda"), want_episodes=True)
    env.close()


def test_full_size_sums_equal_the_statistics(gym):
    """CartPole at 2^24, one 32-step launch with the device policy: the lengths and returns of the episodes add up to
    the statistics' deltas exactly; Pendulum at 2^22 with running returns, to 1e-6 relative."""
    n, K = 1 << 24, 32
    env = gym.GpuVecEnv(0, n, seed=0xF1A1)
    env.reset()
    s0 = env.stats()
    out, ep = env.rollout(K, want_episodes=True)  # all three trajectories: the FULL form
    s1 = env.stats()
    hit = out.flags != 0
    assert int(hit.sum().item()) == s1.episodes - s0.episodes > 0
    assert int(ep.length[hit].to(torch.int64).sum().item()) == s1.length_sum - s0.length_sum
    assert float(ep.ret[hit].to(torch.float64).sum().item()) == s1.return_sum - s0.return_sum
    del out, ep
    env.close()

    n, K = 1 << 22, 32
    pen = gym.GpuVecEnv(3, n, seed=5, track_returns=True)
    pen.reset()
    pen.set_state(dev(random_states(np.random.default_rng(5), 3, n)),
                  dev(np.random.default_rng(6).integers(180, 200, n).astype(np.int32)))
    s0 = pen.stats()
    out, ep = pen.rollout(K, want_episodes=True)
    s1 = pen.stats()
    hit = out.flags != 0
    assert int(hit.sum().item()) == s1.episodes - s0.episodes > 0
    assert int(ep.length[hit].to(torch.int64).sum().item()) == s1.length_sum - s0.length_sum
    got, want = float(ep.ret[hit].to(torch.float64).sum().item()), s1.return_sum - s0.return_sum
    assert abs(got - want) <= 1e-6 * abs(want)
    pen.close()


def test_python_step_and_iter_rollout(gym):
    """GpuVecEnv.step(want_episodes=True) and iter_rollout(want_episodes=True), which reuses one [chunk, N] pair."""
    n, T, chunk, kind = 4096, 230, 32, 3  # Pendulum truncates at 200; the last launch is a partial chunk
    a, b = make(gym, kind, n, 4), make(gym, kind, n, 4)
    a.reset(), b.reset()
    bufs, hits = set(), 0
    for first, (out, ep) in a.iter_rollout(T, chunk=chunk, want_episodes=True):
        k = out.flags.shape[0]
        want, wep = b.rollout(k, want_episodes=True)
        hit = want.flags != 0
        assert same(out.flags, want.flags) and same(ep.ret[hit], wep.ret[hit]) and same(ep.length[hit],
                                                                                         wep.length[hit]), first
        assert ep.ret.dtype == torch.float32 and ep.length.dtype == torch.int32
        bufs.add((ep.ret.data_ptr(), ep.length.data_ptr()))
        hits += int(hit.sum().item())
    assert len(bufs) == 1 and hits >= n
    # per-call steps: (info, episodes) and (info, final, episodes)
    c = make(gym, 0, n, 8)
    c.reset()
    seen = 0
    for t in range(60):
        acts = c.sample_actions()
        if t % 2:
            info, fin, ep = c.step(acts, want_final_obs=True, want_episodes=True)
            assert fin.shape == (4, n)
        else:
            info, ep = c.step(acts, want_episodes=True)
        hit = info.flags != 0
        seen += int(hit.sum().item())
        assert (ep.length[hit] >= 1).all() and same(ep.ret[hit], ep.length[hit].to(torch.float32))
    s = c.stats()
    assert seen == s.episodes > 0
    a.close(), b.close(), c.close()


def test_cpp_host_layer(gym):
    """GpuVecEnv::step_episodes / rollout_episodes of include/mgym.hpp (tests/cpp/test_episodes.cpp)."""
    src = os.path.join(ROOT, "tests", "cpp", "test_episodes.cpp")
    pkg = os.path.join(ROOT, "modurl_gym_b200")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "test_episodes")
        r = subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-Wall", f"-I{cuda}/include", "-o", exe,
                            src, f"-L{pkg}", "-lmgym", f"-L{cuda}/lib64", "-lcudart", f"-Wl,-rpath,{pkg}",
                            f"-Wl,-rpath,{cuda}/lib64"], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ALL OK" in out.stdout, out.stdout + out.stderr
    assert out.stdout.count("ok ") >= 3
