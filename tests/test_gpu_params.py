"""Per-env physics parameters on the device (mgym_set_params / mgym_get_params / mgym_sample_params)."""
import ctypes as C

import numpy as np
import pytest

import params_oracle as po
from helpers import assert_bit_equal, random_actions, random_states

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

KINDS = [0, 1, 2, 3]


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


def random_params(rng, gym, kind, n, spread=0.5):
    d = np.asarray(gym.GpuVecEnv.param_defaults(kind), dtype=np.float64)[:, None]
    return (d * rng.uniform(1 - spread, 1 + spread, (len(d), n))).astype(np.float32)


def make_pair(gym, kind, n, rng, **kw):
    """Two handles in the same random state: `a` without parameters, `b` with the defaults set explicitly."""
    a, b = gym.GpuVecEnv(kind, n, seed=7, **kw), gym.GpuVecEnv(kind, n, seed=7, **kw)
    st = dev(random_states(rng, kind, n))
    steps = dev(rng.integers(0, 150, n).astype(np.int32))
    for e in (a, b):
        e.reset()
        e.set_state(st, steps)
    b.set_params(torch.tensor(gym.GpuVecEnv.param_defaults(kind)).repeat(n, 1).T.contiguous())
    return a, b


def assert_same_handles(a, b):
    for x, y in zip(a.get_state(), b.get_state()):
        assert same(x, y)
    assert a.stats() == b.stats()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [1 << 20, (1 << 20) + 4, 1000])
def test_defaults_are_bit_identical_to_no_parameters(gym, kind, n):
    """TMA (N % 1024 == 0), ragged tail and scalar lanes; step with final_obs, FULL and non-FULL rollouts."""
    rng = np.random.default_rng(kind * 7 + n % 13)
    a, b = make_pair(gym, kind, n, rng, track_returns=True)
    for t in range(12):
        acts = dev(random_actions(rng, kind, n))
        ia, fa = a.step(acts, want_final_obs=True)
        ib, fb = b.step(acts, want_final_obs=True)
        assert same(ia.state, ib.state) and same(ia.reward, ib.reward) and same(ia.flags, ib.flags), t
        assert same(fa, fb), t
    assert_same_handles(a, b)
    ra, rb = a.rollout(16), b.rollout(16)  # FULL form when n % 128 == 0
    assert all(same(x, y) for x, y in zip(ra, rb))
    acts = dev(random_actions(rng, kind, (8, n)))
    ra, rb = a.rollout(8, acts, want_obs=False), b.rollout(8, acts, want_obs=False)  # non-FULL
    assert same(ra.reward, rb.reward) and same(ra.flags, rb.flags) and same(ra.done_count, rb.done_count)
    assert_same_handles(a, b)
    a.close(), b.close()


@pytest.mark.parametrize("kind", KINDS)
def test_defaults_bit_identical_manual_mode_and_step_host(gym, kind):
    n = 8192
    rng = np.random.default_rng(50 + kind)
    a, b = make_pair(gym, kind, n, rng, auto_reset=False)
    for t in range(30):
        acts = dev(random_actions(rng, kind, n))
        ia, ib = a.step(acts), b.step(acts)
        assert same(ia.state, ib.state) and same(ia.reward, ib.reward) and same(ia.flags, ib.flags), t
        mask = ia.flags != 0
        a.reset(mask=mask), b.reset(mask=mask)
    assert_same_handles(a, b)
    a.close(), b.close()
    n = 1 << 20  # chunked step_host: sub-range launches (first / ld)
    a, b = make_pair(gym, kind, n, rng)
    od = a.obs_dim
    for t in range(3):
        acts = random_actions(rng, kind, n)
        outs = []
        for e in (a, b):
            o, r, f = np.empty((od, n), np.float32), np.empty(n, np.float32), np.empty(n, np.uint8)
            e.step_host(acts, o, r, f)
            outs.append((o, r, f))
        for x, y in zip(*outs):
            assert_bit_equal(y, x, f"step_host {t}")
    assert_same_handles(a, b)
    a.close(), b.close()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [4096, 1000])
def test_random_parameters_match_oracle(gym, kind, n):
    """>= 200 steps with auto-resets, then a rollout, bit-exact to oracle_vec_step_p / oracle_vec_rollout_p."""
    rng = np.random.default_rng(100 + kind + n)
    prm = random_params(rng, gym, kind, n)
    env = gym.GpuVecEnv(kind, n, seed=31, track_returns=True)
    ref = po.VecState(kind, n, seed=31, auto_reset=1)
    st = random_states(rng, kind, n)
    env.reset()  # the step index stays 0, like the oracle's t
    env.set_state(dev(st))  # counts 0
    ref.state[:] = st
    ref.steps[:] = 0
    ref.sbt[:] = 0
    env.set_params(dev(prm))
    ref.set_params(prm)
    for t in range(200):
        acts = random_actions(rng, kind, n)
        info = env.step(dev(acts))
        obs, rew, flg = ref.step(acts)
        assert_bit_equal(host(info.flags), flg, f"flags {t}")
        assert_bit_equal(host(info.reward), rew, f"reward {t}")
        assert_bit_equal(host(info.state), obs, f"obs {t}")
    acts = random_actions(rng, kind, (32, n))
    r = env.rollout(32, dev(acts))
    obs, rew, flg, dc = ref.rollout(32, acts)
    assert_bit_equal(host(r.flags), flg, "rollout flags")
    assert_bit_equal(host(r.reward), rew, "rollout reward")
    assert_bit_equal(host(r.obs), obs, "rollout obs")
    assert int(r.done_count.item()) == dc
    assert_bit_equal(host(env.get_state()[0]), ref.state, "state")
    env.close()


@pytest.mark.parametrize("kind", KINDS)
def test_each_env_reads_only_its_own_row(gym, kind):
    n = 4096
    rng = np.random.default_rng(200 + kind)
    st, prm = random_states(rng, kind, n), random_params(rng, gym, kind, n)
    acts = random_actions(rng, kind, n)
    perm = rng.permutation(n)
    a, b = gym.GpuVecEnv(kind, n, seed=1, auto_reset=False), gym.GpuVecEnv(kind, n, seed=1, auto_reset=False)
    for e, p in ((a, np.arange(n)), (b, perm)):
        e.reset()
        e.set_state(dev(st[:, p]))
        e.set_params(dev(prm[:, p]))
    ia, ib = a.step(dev(acts)), b.step(dev(acts[perm]))
    assert_bit_equal(host(ib.state), host(ia.state)[:, perm], "obs")
    assert_bit_equal(host(ib.reward), host(ia.reward)[perm], "reward")
    assert_bit_equal(host(ib.flags), host(ia.flags)[perm], "flags")
    a.close(), b.close()


def test_set_params_rejects_bad_values_and_leaves_the_handle_untouched(gym):
    from modurl_gym_b200._lib import MgymError

    n = 2048
    rng = np.random.default_rng(3)
    lib = gym.load_library()
    env = gym.GpuVecEnv(0, n, seed=2)
    env.reset()
    good = dev(random_params(rng, gym, 0, n))
    env.set_params(good)
    before = [t.clone() for t in env.get_state()]
    for row, value in ((0, float("nan")), (2, 0.0), (1, -1.0), (5, float("inf"))):
        bad = good.clone()
        bad[row, 17] = value
        with pytest.raises(MgymError):
            env.set_params(bad)
        hb = np.ascontiguousarray(host(bad))  # host rows are checked too
        assert lib.mgym_set_params(env._h, hb.ctypes.data_as(C.c_void_p), None) == -1
        assert same(env.get_params(), good)
    assert all(same(x, y) for x, y in zip(before, env.get_state()))
    acro = gym.GpuVecEnv(4, 128)
    with pytest.raises(MgymError, match="no per-env parameters"):
        acro.set_params(torch.zeros((0, 128), device="cuda"))
    with pytest.raises(MgymError):
        acro.sample_params([], [])
    assert gym.GpuVecEnv.param_names(4) == ()
    acro.close()
    # None: back to the no-parameter kernels
    a = gym.GpuVecEnv(0, n, seed=2)
    env.reset()
    a.set_state(env.get_state()[0])  # counts 0 on both, step index 0 on both
    env.set_params(None)
    assert same(env.get_params(), torch.tensor(gym.GpuVecEnv.param_defaults(0), device="cuda")[:, None].expand(6, n))
    acts = dev(random_actions(rng, 0, n))
    ia, ib = a.step(acts), env.step(acts)
    assert same(ia.state, ib.state) and same(ia.flags, ib.flags)
    a.close(), env.close()


def test_get_params_round_trips_host_and_device(gym):
    n = 1000
    rng = np.random.default_rng(4)
    env = gym.GpuVecEnv(3, n)
    lib = gym.load_library()
    want = np.asarray(gym.GpuVecEnv.param_defaults(3), dtype=np.float32)[:, None].repeat(n, 1)
    out = np.empty((3, n), np.float32)
    assert lib.mgym_get_params(env._h, out.ctypes.data_as(C.c_void_p), None) == 0
    assert_bit_equal(out, want, "defaults, host")
    assert_bit_equal(host(env.get_params()), want, "defaults, device")
    prm = random_params(rng, gym, 3, n)
    env.set_params(prm.copy())  # numpy -> set_params takes it through torch (device)
    assert lib.mgym_set_params(env._h, prm.ctypes.data_as(C.c_void_p), None) == 0  # a host pointer
    assert lib.mgym_get_params(env._h, out.ctypes.data_as(C.c_void_p), None) == 0
    assert_bit_equal(out, prm, "host")
    assert_bit_equal(host(env.get_params()), prm, "device")
    env.set_params({"g": 9.81, "l": dev(prm[2])})
    got = host(env.get_params())
    assert (got[0] == np.float32(9.81)).all() and (got[1] == prm[1]).all() and (got[2] == prm[2]).all()
    env.close()


@pytest.mark.parametrize("kind", [0, 3])
def test_checkpoint_with_parameters_resumes_bit_identically(gym, kind):
    n = 4096
    rng = np.random.default_rng(5)
    a = gym.GpuVecEnv(kind, n, seed=8)
    a.reset()
    a.set_params(dev(random_params(rng, gym, kind, n)))
    acts = [dev(random_actions(rng, kind, n)) for _ in range(20)]
    for x in acts[:10]:
        a.step(x)
    blob = a.checkpoint()
    want = [a.step(x).state.clone() for x in acts[10:]]
    b = gym.GpuVecEnv(kind, n, seed=0)
    b.restore(blob)
    assert same(b.get_params(), a.get_params())
    for x, w in zip(acts[10:], want):
        assert same(b.step(x).state, w)
    # a blob without parameters clears them, and is as long as it always was
    c = gym.GpuVecEnv(kind, n, seed=8)
    plain = c.checkpoint()
    b.restore(plain)
    assert len(plain) == len(blob) - 4 * n * len(gym.GpuVecEnv.param_names(kind))
    assert b.checkpoint() == plain
    a.close(), b.close(), c.close()


@pytest.mark.parametrize("kind", [0, 1])
def test_graph_of_masked_sample_and_step_replays_like_eager(gym, kind):
    n, T = 8192, 40
    d = np.asarray(gym.GpuVecEnv.param_defaults(kind), dtype=np.float32)
    low, high = list(d * 0.8), list(d * 1.2)
    a = gym.GpuVecEnv(kind, n, seed=5)
    b = gym.GpuVecEnv(kind, n, seed=5, graph_capturable=True)
    a.reset(), b.reset()
    acts_b = torch.empty(n, dtype=b.action_dtype, device="cuda")
    for e in (a, b):
        e.sample_params(low, high, key=1)
    b.step(b.sample_actions(out=acts_b))
    ia = a.step(a.sample_actions())
    mask_b = torch.ones(n, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        b.sample_params(low, high, mask=mask_b, key=2)
        b.sample_actions(out=acts_b)
        info_b = b.step(acts_b)
        mask_b.copy_(info_b.flags != 0)
    mask_b.copy_((ia.flags != 0).to(torch.uint8))
    torch.cuda.synchronize()
    for t in range(T):
        a.sample_params(low, high, mask=(ia.flags != 0), key=2)
        ia = a.step(a.sample_actions())
        graph.replay()
        assert same(ia.state, info_b.state) and same(ia.flags, info_b.flags), t
        assert same(a.get_params(), b.get_params()), t
    a.close(), b.close()


@pytest.mark.parametrize("kind", KINDS)
def test_four_shards_equal_one_handle(gym, kind):
    n = 8192
    q = n // 4
    rng = np.random.default_rng(9)
    d = np.asarray(gym.GpuVecEnv.param_defaults(kind), dtype=np.float32)
    low, high = list(d * 0.5), list(d * 1.5)
    whole = gym.GpuVecEnv(kind, n, seed=12)
    shards = [gym.GpuVecEnv(kind, q, seed=12, env_index_base=i * q) for i in range(4)]
    whole.reset()
    st = whole.get_state()[0]
    whole.sample_params(low, high, key=3)
    for i, s in enumerate(shards):
        s.reset()
        s.set_state(st[:, i * q:(i + 1) * q])
        s.sample_params(low, high, key=3)
    assert same(torch.cat([s.get_params() for s in shards], 1), whole.get_params())
    for t in range(50):
        acts = dev(random_actions(rng, kind, n))
        iw = whole.step(acts)
        for i, s in enumerate(shards):
            si = s.step(acts[i * q:(i + 1) * q].contiguous())
            assert same(si.state, iw.state[:, i * q:(i + 1) * q]) and same(si.flags, iw.flags[i * q:(i + 1) * q]), t
    for e in [whole] + shards:
        e.close()


@pytest.mark.parametrize("kind", KINDS)
def test_sample_params_matches_oracle_and_respects_the_mask(gym, kind):
    n = 5000
    d = np.asarray(gym.GpuVecEnv.param_defaults(kind), dtype=np.float32)
    low, high = d * np.float32(0.5), d * np.float32(1.5)
    env = gym.GpuVecEnv(kind, n, seed=77, env_index_base=12)
    ref = po.VecState(kind, n, seed=77, env_index_base=12)
    env.sample_params(low, high, key=5)
    ref.sample_params(low, high, key=5, defaults=d)
    assert_bit_equal(host(env.get_params()), ref.params, "all envs")
    before = host(env.get_params())
    mask = (np.random.default_rng(1).random(n) < 0.3).astype(np.uint8)
    env.sample_params(low, high, mask=dev(mask), key=6)
    ref.sample_params(low, high, mask=mask, key=6)
    got = host(env.get_params())
    assert_bit_equal(got, ref.params, "masked")
    assert_bit_equal(got[:, mask == 0], before[:, mask == 0], "unmasked rows untouched")
    env.close()
