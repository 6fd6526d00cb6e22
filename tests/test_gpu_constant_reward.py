"""The handle-owned reward row (mgym_reward_ptr, mgym_reward_constant, GpuVecEnv.step's reward).

A handle whose rewards are all one value (CartPole-v1 with auto-reset and the default rewards, MountainCar-v0) fills its
row once at creation and a step given the row stores no reward.  Everything such a step returns must be bit-identical
to a twin handle with the same seed stepped into an explicit reward buffer, which every step writes; and the values
that twin's kernels write must all be the constant the handle reports."""
import ctypes as C

import pytest

torch = pytest.importorskip("torch")

SENTINEL = 7.0  # a value no step of these kinds produces


def same(x, y):
    if x.dtype == torch.float32:
        x, y = x.view(torch.int32), y.view(torch.int32)
    return torch.equal(x, y)


def mismatches(x, y):
    """Number of elements that differ bit for bit, as a device scalar (no synchronisation per step)."""
    if x.dtype == torch.float32:
        x, y = x.view(torch.int32), y.view(torch.int32)
    return (x != y).sum()


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def test_null_handle():
    from modurl_gym_b200 import build as b

    b.build()
    import modurl_gym_b200

    lib = modurl_gym_b200.load_library()
    assert lib.mgym_reward_ptr(None) is None
    v = C.c_float(3.0)
    assert lib.mgym_reward_constant(None, C.byref(v)) < 0 and v.value == 3.0


@pytest.fixture(scope="module")
def gym():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import modurl_gym_b200 as m

    m.load_library()
    return m


def with_params(env, mode, key=1):
    """mode None: the kind's constants; "rows": per-env parameters +-20 % around the defaults; "redraw": the same rows
    and +-20 % redraw ranges (every reset draws new ones)."""
    if mode is None:
        return
    d = env.param_defaults(env.kind)
    low, high = [0.8 * x for x in d], [1.2 * x for x in d]
    env.sample_params(low, high, key=key)
    if mode == "redraw":
        env.set_param_redraw(low, high)


# ---- which handles are constant ---------------------------------------------------------------------------------------

def table_cases():
    for kind in range(5):
        for auto in (True, False):
            for sb in ((False, True) if kind == 0 else (False,)):
                for mode in ((None, "rows", "redraw") if kind != 4 else (None,)):
                    yield kind, auto, sb, mode


@pytest.mark.gpu
@pytest.mark.parametrize("kind,auto,sb,mode", list(table_cases()))
def test_constancy_table(gym, kind, auto, sb, mode):
    n = 1027
    env = gym.GpuVecEnv(kind, n, seed=3, auto_reset=auto, sutton_barto_reward=sb)
    with_params(env, mode)
    want = 1.0 if (kind == 0 and auto and not sb) else (-1.0 if kind == 1 else None)
    v = C.c_float(123.0)
    rc = env._lib.mgym_reward_constant(env._h, C.byref(v))
    assert rc == (0 if want is None else 1)
    assert v.value == (123.0 if want is None else want)
    assert env._lib.mgym_reward_constant(env._h, None) == rc
    assert env.reward_constant == want
    row = env._lib.mgym_reward_ptr(env._h)
    assert row == env.step(torch.zeros(n, dtype=env.action_dtype, device="cuda")).reward.data_ptr()
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_row_filled_at_creation(gym, kind):
    env = gym.GpuVecEnv(kind, 4096, seed=1)
    row = env._reward
    assert row.dtype == torch.float32 and row.shape == (4096,) and row.is_contiguous()
    assert bool((row == env.reward_constant).all())
    env.close()


# ---- twin handles: the row against an explicit buffer, bit for bit ---------------------------------------------------

KINDS = {"cartpole": (0, {}), "mountain_car": (1, {}), "mountain_car_limit": (1, {"max_episode_steps": 200})}
SIZES = [4096, 2052, 1027, 515, 1]  # TMA tiles; TMA head + vector tail; scalar lanes; scalar lanes; one env
FORMS = ["plain", "final", "episodes", "rows", "redraw", "graph"]
STEPS = 600  # past CartPole's 500-step truncation


def force_endings(env, kind, cfg):
    """Start half of the envs near their end: CartPole and the 200-step MountainCar a few steps before the time limit,
    MountainCar-v0 (no limit) rolling into the goal."""
    n = env.num_envs
    state = env.state_view.clone()
    steps = torch.zeros(n, dtype=torch.int32, device="cuda")
    idx = torch.arange(0, n, 2, device="cuda")
    if kind == 0:
        steps[idx] = 499 - (idx % 10).to(torch.int32)  # env 0 truncates at the first step
    elif cfg.get("max_episode_steps"):
        steps[idx] = 199 - (idx % 10).to(torch.int32)
    else:
        state[0, idx] = 0.3 + 0.19 * (idx % 16).to(torch.float32) / 16
        state[1, idx] = 0.06
    env.set_state(state, steps)


@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("name", list(KINDS))
def test_twin_handles_bit_for_bit(gym, name, n, form):
    kind, cfg = KINDS[name]
    graph = form == "graph"
    a, b = (gym.GpuVecEnv(kind, n, seed=21, graph_capturable=graph, **cfg) for _ in range(2))
    assert a.reward_constant is not None
    for e in (a, b):
        with_params(e, {"rows": "rows", "redraw": "redraw"}.get(form))
        e.reset()
        force_endings(e, kind, cfg)
    od = a.obs_dim
    rb = torch.empty(n, dtype=torch.float32, device="cuda")
    fb = torch.empty(n, dtype=torch.uint8, device="cuda")
    finb = torch.empty((od, n), dtype=torch.float32, device="cuda")
    retb = torch.zeros(n, dtype=torch.float32, device="cuda")
    lenb = torch.zeros(n, dtype=torch.int32, device="cuda")
    const = torch.full((n,), a.reward_constant, dtype=torch.float32, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(n)
    pool = [torch.randint(0, 3 if kind == 1 else 2, (n,), dtype=torch.uint8, device="cuda", generator=gen)
            for _ in range(8)]
    bad = {k: torch.zeros((), dtype=torch.int64, device="cuda") for k in ("obs", "reward", "flags", "final", "ep", "const")}
    ended = torch.zeros((), dtype=torch.int64, device="cuda")

    def step_a(acts):
        if form == "final":
            info, fin = a.step(acts, want_final_obs=True)
            return info, fin, None
        if form == "episodes":
            info, ep = a.step(acts, want_episodes=True)
            return info, None, ep
        return a.step(acts), None, None

    def step_b(acts):
        if form == "episodes":
            gym._lib.check(b._lib.mgym_step_episodes(b._h, ptr(acts), None, ptr(rb), ptr(fb), None, ptr(retb),
                                                     ptr(lenb), b._stream()))
        else:
            b.step_raw(acts, reward_out=rb, flags_out=fb, final_obs_out=finb if form == "final" else None)

    def compare(info, fin, ep):
        bad["obs"] += mismatches(info.state, b.state_view)
        bad["reward"] += mismatches(info.reward, rb)
        bad["flags"] += mismatches(info.flags, fb)
        bad["const"] += mismatches(rb, const)
        if fin is not None:
            bad["final"] += mismatches(fin, finb)
        if ep is not None:
            bad["ep"] += mismatches(ep.ret, retb) + mismatches(ep.length, lenb)
        ended.add_((fb != 0).sum())

    if graph:
        acts_a = torch.empty(n, dtype=torch.uint8, device="cuda")
        acts_b = torch.empty(n, dtype=torch.uint8, device="cuda")
        step_a(a.sample_actions(out=acts_a))  # one eager step each first (occupancy queries, buffers)
        step_b(b.sample_actions(out=acts_b))
        torch.cuda.synchronize()
        ga, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(ga):
            a.sample_actions(out=acts_a)
            info, _, _ = step_a(acts_a)
        with torch.cuda.graph(gb):
            b.sample_actions(out=acts_b)
            step_b(acts_b)
        for _ in range(STEPS - 1):
            ga.replay()
            gb.replay()
            compare(info, None, None)
    else:
        for t in range(STEPS):
            acts = pool[t % len(pool)]
            info, fin, ep = step_a(acts)
            step_b(acts)
            compare(info, fin, ep)
    torch.cuda.synchronize()
    assert {k: int(v) for k, v in bad.items()} == {k: 0 for k in bad}
    assert int(ended) > 0
    sa, sb = a.stats(), b.stats()
    assert sa == sb and sa.episodes > 0
    if kind == 0:
        assert sa.truncated > 0, "no CartPole episode reached the 500-step limit"
    assert a.step_index == b.step_index == STEPS
    a.close(), b.close()


# ---- explicit buffers are still written ----------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("n", [4096, 1027])
def test_explicit_buffer_is_written(gym, kind, n):
    env = gym.GpuVecEnv(kind, n, seed=2)
    env.reset()
    buf = torch.full((n,), float("nan"), dtype=torch.float32, device="cuda")
    env.step_raw(torch.zeros(n, dtype=torch.uint8, device="cuda"), reward_out=buf)
    assert bool((buf == env.reward_constant).all())
    env.close()


# ---- handles that are not constant write the row every step ----------------------------------------------------------

NON_CONSTANT = {
    "cartpole_sutton_barto": (0, dict(sutton_barto_reward=True)),
    "cartpole_manual": (0, dict(auto_reset=False)),  # stepped past termination: r_after
    "mountain_car_continuous": (2, {}),
    "pendulum": (3, {}),
    "acrobot": (4, {}),
}


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4096, 1027])
@pytest.mark.parametrize("name", list(NON_CONSTANT))
def test_non_constant_handles_write_the_row(gym, name, n):
    kind, cfg = NON_CONSTANT[name]
    a, b = (gym.GpuVecEnv(kind, n, seed=4, **cfg) for _ in range(2))
    assert a.reward_constant is None
    a.reset(), b.reset()
    rb = torch.empty(n, dtype=torch.float32, device="cuda")
    fb = torch.empty(n, dtype=torch.uint8, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(5)
    seen = set()
    for t in range(200):
        if a.continuous:
            acts = (torch.rand(n, device="cuda", generator=gen) * 4 - 2) * (0.5 if kind == 2 else 1.0)
        else:
            acts = torch.randint(0, 3 if kind == 4 else 2, (n,), dtype=torch.uint8, device="cuda", generator=gen)
        info = a.step(acts)
        b.step_raw(acts, reward_out=rb, flags_out=fb)
        assert same(info.reward, rb) and same(info.flags, fb), f"step {t}"
        if t % 50 == 49:
            seen |= set(torch.unique(rb).tolist())
    if name == "cartpole_manual":
        assert {0.0, 1.0} <= seen, "no step past termination (r_after)"
    if name == "cartpole_sutton_barto":
        assert {0.0, -1.0} <= seen
    a.close(), b.close()


# ---- the row survives every other call ---------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("n", [4096, 1027])
def test_row_survives_other_calls(gym, kind, n):
    env = gym.GpuVecEnv(kind, n, seed=8)
    env.reset()
    acts = torch.ones(n, dtype=torch.uint8, device="cuda")
    row = env.step(acts).reward
    mask = (torch.arange(n, device="cuda") % 3 == 0).to(torch.uint8)
    d = env.param_defaults(kind)
    calls = [
        ("reset", lambda: env.reset()),
        ("reset(mask)", lambda: env.reset(mask)),
        ("checkpoint save/load", lambda: env.restore(env.checkpoint())),
        ("set_state", lambda: env.set_state(env.state_view.clone(), torch.full((n,), 3, dtype=torch.int32))),
        ("set_params", lambda: env.set_params(torch.tensor(d).unsqueeze(1).repeat(1, n) * 1.1)),
        ("set_param_redraw + reset", lambda: (env.set_param_redraw([0.9 * x for x in d], [1.1 * x for x in d]),
                                              env.reset())),
        ("rollout", lambda: env.rollout(4)),
        ("step", lambda: env.step(acts)),
    ]
    for value in (env.reward_constant, SENTINEL):  # the constant, then a value no library call would write
        row.fill_(value)
        for what, call in calls:
            call()
            torch.cuda.synchronize()
            assert bool((row == value).all()), f"{what} wrote the reward row"
    assert env.step(acts).reward.data_ptr() == row.data_ptr()
    env.close()
