"""LunarLander-v2 on the GPU against the CPU oracle (oracle/lunar_oracle.c).  `pytest -m gpu`.

PARITY UNPINNED w.r.t. the real reference: box2d-py is not available, so both the oracle and the
kernel re-derive Box2D 2.3's algorithm.  What IS checked: (1) the two independent implementations
(generic C vs specialised CUDA) agree bit for bit on float32 observations, rewards and flags over
long random and heuristic roll-outs -- every contact manifold, joint limit transition, block-solver
case and sleep event included; (2) the behavioural test the reference itself has at this boundary
(tests/envs/test_env_implementation.py:13-17: heuristic return > 100 at seed 1); (3) invariants.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _heuristic_batch(s):
    """gym/envs/box2d/lunar_lander.py:726-777 (discrete), vectorised over envs."""
    angle_targ = np.clip(s[:, 0] * 0.5 + s[:, 2] * 1.0, -0.4, 0.4)
    hover_targ = 0.55 * np.abs(s[:, 0])
    angle_todo = (angle_targ - s[:, 4]) * 0.5 - s[:, 5] * 1.0
    hover_todo = (hover_targ - s[:, 1]) * 0.5 - s[:, 3] * 0.5
    legs = (s[:, 6] != 0) | (s[:, 7] != 0)
    angle_todo = np.where(legs, 0.0, angle_todo)
    hover_todo = np.where(legs, -s[:, 3] * 0.5, hover_todo)
    a = np.zeros(len(s), dtype=np.int64)
    main = (hover_todo > np.abs(angle_todo)) & (hover_todo > 0.05)
    a[main] = 2
    a[~main & (angle_todo < -0.05)] = 3
    a[~main & ~(angle_todo < -0.05) & (angle_todo > 0.05)] = 1
    return a


def test_reference_behavioural_test_heuristic_lands():
    """tests/envs/test_env_implementation.py:13-17 on the engine's single-env facade."""
    import gym_b200
    from oracle.oracle import lunar_heuristic
    env = gym_b200.make("LunarLander-v2")
    s, info = env.reset(seed=1)
    assert s.shape == (8,) and s.dtype == np.float32 and info == {}
    total, steps = 0.0, 0
    while True:
        s, r, terminated, truncated, _ = env.step(lunar_heuristic(s))
        total += r
        steps += 1
        if terminated or truncated:
            break
    assert total > 100, (total, steps)
    env.close()


@pytest.mark.parametrize("policy", ["random", "heuristic"])
def test_bit_exact_against_oracle(policy):
    import gym_b200
    import torch
    from oracle.oracle import OracleLunar
    N, T, seed = 1024, 400, 11
    env = gym_b200.vector.make("LunarLander-v2", N)
    orc = OracleLunar(N)
    obs, _ = env.reset(seed=seed)
    ref = orc.reset(seed=seed)
    assert np.array_equal(obs.cpu().numpy(), ref), "reset observations (incl. the embedded step(0))"
    rng = np.random.default_rng(3)
    cur = ref
    n_term = n_sleep = n_crash = 0
    for t in range(T):
        a = rng.integers(0, 4, size=N) if policy == "random" else _heuristic_batch(cur)
        o, r, te, tr, info = env.step(torch.as_tensor(a, device=env.device))
        ro, rr, rte, rtr, rfo = orc.step(a)
        assert np.array_equal(te.cpu().numpy(), rte), f"step {t}: terminated"
        assert np.array_equal(tr.cpu().numpy(), rtr), f"step {t}: truncated"
        o_h = o.cpu().numpy()
        if not np.array_equal(o_h, ro):
            bad = np.argwhere(o_h != ro)
            raise AssertionError(f"step {t}: {len(bad)} observation values differ, first env {bad[0][0]} "
                                 f"got {o_h[bad[0][0]]} want {ro[bad[0][0]]}")
        assert np.array_equal(r.cpu().numpy(), rr), f"step {t}: reward"
        done = rte | rtr
        if done.any():
            assert np.array_equal(info["final_observation"].cpu().numpy()[done], rfo[done])
        n_term += int(rte.sum())
        n_sleep += int((rr[rte] == 100).sum())
        n_crash += int((rr[rte] == -100).sum())
        cur = ro
    assert n_term > 0 and n_crash > 0
    if policy == "heuristic":
        assert n_sleep > N // 2, "most heuristic episodes end asleep on the pad (+100)"
    bodies, flags = env.lunar_bodies()
    for i in (0, 1, N - 1):
        ob, of = orc.bodies(i)
        assert np.array_equal(bodies[i].cpu().numpy(), ob)
        assert flags[i, :3].tolist() == of[:3].tolist() and int(flags[i, 5]) == int(of[5])
    # the manifold table (8 touching pairs per env) never filled up, on either side
    assert env.box2d_overflows() == 0 and orc.overflows() == 0
    env.close()
    orc.close()


def test_invariants_and_api():
    import gym_b200
    import torch
    from gym_b200 import error, spaces
    N = 4096
    env = gym_b200.vector.make("LunarLander-v2", N)
    assert isinstance(env.single_action_space, spaces.Discrete) and env.single_action_space.n == 4
    assert env.single_observation_space.shape == (8,) and env.max_episode_steps == 1000
    obs, _ = env.reset(seed=0)
    assert bool((obs[:, 6:] == 0).all())                       # legs in the air at the start
    assert bool(((obs[:, 0].abs() < 0.05) & (obs[:, 1] > 1.3)).all())
    gen = torch.Generator(device="cuda").manual_seed(0)
    done_total = 0
    for t in range(250):
        a = torch.randint(0, 4, (N,), device="cuda", generator=gen)
        o, r, te, tr, info = env.step(a)
        assert bool(((o[:, 6:] == 0) | (o[:, 6:] == 1)).all())  # leg flags are 0/1
        assert bool(torch.isfinite(o).all()) and bool(torch.isfinite(r).all())
        fo = info["final_observation"]
        crashed = te & (r == -100)
        assert bool((r[te].abs() == 100).all())                 # terminal reward is +-100
        assert not bool(tr.any())
        done_total += int(te.sum())
        # a -100 ending is a body-ground contact (near the ground) or leaving the viewport sideways
        assert bool(((fo[crashed][:, 1] < 1.2) | (fo[crashed][:, 0].abs() >= 1.0)).all())
    assert done_total > N // 2                                  # random policies crash within ~100-200 steps
    with pytest.raises(AssertionError):                         # lunar_lander.py:210-212
        gym_b200.vector.make("LunarLander-v2", 4, gravity=-12.5)
    with pytest.raises(TypeError):
        gym_b200.vector.make("LunarLander-v2", 4, hardcore=True)
    env.step(torch.full((N,), 4, device="cuda"))
    with pytest.raises(error.InvalidAction):
        env.check_actions()
    env.close()
    # determinism (tests/envs/test_envs.py:60-115)
    e1, e2 = gym_b200.vector.make("LunarLander-v2", 64), gym_b200.vector.make("LunarLander-v2", 64)
    o1, _ = e1.reset(seed=5)
    o2, _ = e2.reset(seed=5)
    assert torch.equal(o1, o2)
    for t in range(100):
        a = torch.randint(0, 4, (64,), device="cuda", generator=gen)
        r1, r2 = e1.step(a), e2.step(a)
        assert all(torch.equal(x, y) for x, y in zip(r1[:4], r2[:4]))
    e1.close()
    e2.close()


def _cont_heuristic_batch(s):
    """gym/envs/box2d/lunar_lander.py:726-768 (continuous branch), vectorised over envs."""
    angle_targ = np.clip(s[:, 0] * 0.5 + s[:, 2] * 1.0, -0.4, 0.4)
    hover_targ = 0.55 * np.abs(s[:, 0])
    angle_todo = (angle_targ - s[:, 4]) * 0.5 - s[:, 5] * 1.0
    hover_todo = (hover_targ - s[:, 1]) * 0.5 - s[:, 3] * 0.5
    legs = (s[:, 6] != 0) | (s[:, 7] != 0)
    angle_todo = np.where(legs, 0.0, angle_todo)
    hover_todo = np.where(legs, -s[:, 3] * 0.5, hover_todo)
    return np.clip(np.stack([hover_todo * 20 - 1, -angle_todo * 20], axis=1), -1, +1).astype(np.float32)


VARIANTS = [
    # (id, ctor kwargs, policy)
    ("LunarLanderContinuous-v2", dict(), "random"),
    ("LunarLanderContinuous-v2", dict(), "heuristic"),
    ("LunarLander-v2", dict(continuous=True, gravity=-6.5), "heuristic"),
    ("LunarLander-v2", dict(enable_wind=True), "heuristic"),
    ("LunarLander-v2", dict(enable_wind=True, wind_power=19.0, turbulence_power=1.9, gravity=-11.5), "random"),
    ("LunarLanderContinuous-v2", dict(enable_wind=True, wind_power=5.0, turbulence_power=0.5), "random"),
]


@pytest.mark.parametrize("env_id,kwargs,policy", VARIANTS)
def test_variants_bit_exact_against_oracle(env_id, kwargs, policy):
    """continuous actions (lunar_lander.py:479-481,496-533), gravity (:210-213,240), wind (:449-477)."""
    import gym_b200
    import torch
    from gym_b200 import spaces
    from oracle.oracle import OracleLunar
    N, T, seed = 768, 350, 23
    cont = env_id.startswith("LunarLanderContinuous") or kwargs.get("continuous", False)
    wind = kwargs.get("enable_wind", False)
    rng = np.random.default_rng(17)
    extra = {}
    if wind:
        extra = dict(wind_idx=rng.integers(-9999, 9999, size=N), torque_idx=rng.integers(-9999, 9999, size=N))
    env = gym_b200.vector.make(env_id, N, **kwargs, **extra)
    okw = {k: v for k, v in kwargs.items() if k != "continuous"}
    orc = OracleLunar(N, continuous=cont, **okw, **extra)
    if cont:
        assert isinstance(env.single_action_space, spaces.Box) and env.single_action_space.shape == (2,)
        assert env.action_space.shape == (N, 2) and env.action_space.dtype == np.float32
    obs, _ = env.reset(seed=seed)
    ref = orc.reset(seed=seed)
    assert np.array_equal(obs.cpu().numpy(), ref), "reset observations"
    cur = ref
    n_done = n_sleep = 0
    for t in range(T):
        if cont:
            a = rng.uniform(-1.6, 1.6, size=(N, 2)).astype(np.float32) if policy == "random" else _cont_heuristic_batch(cur)
        else:
            a = rng.integers(0, 4, size=N) if policy == "random" else _heuristic_batch(cur)
        o, r, te, tr, info = env.step(torch.as_tensor(a, device=env.device))
        ro, rr, rte, rtr, rfo = orc.step(a)
        assert np.array_equal(te.cpu().numpy(), rte), f"step {t}: terminated"
        assert np.array_equal(tr.cpu().numpy(), rtr), f"step {t}: truncated"
        o_h = o.cpu().numpy()
        if not np.array_equal(o_h, ro):
            bad = np.argwhere(o_h != ro)
            raise AssertionError(f"step {t}: {len(bad)} observation values differ, first env {bad[0][0]} "
                                 f"got {o_h[bad[0][0]]} want {ro[bad[0][0]]}")
        assert np.array_equal(r.cpu().numpy(), rr), f"step {t}: reward"
        done = rte | rtr
        if done.any():
            assert np.array_equal(info["final_observation"].cpu().numpy()[done], rfo[done])
        n_done += int(done.sum())
        n_sleep += int((rr[rte] == 100).sum())
        cur = ro
    assert n_done > 0
    if policy == "heuristic" and not wind:
        assert n_sleep > N // 3
    if wind:
        gw, gt = env.lunar_wind_idx()
        ow, ot = orc.wind_idx()
        assert np.array_equal(gw, ow) and np.array_equal(gt, ot)
        assert (gw > extra["wind_idx"]).all()
        assert env.get_attr("wind_idx") == tuple(int(v) for v in ow)
    env.close()
    orc.close()


def test_continuous_heuristic_lands_and_numpy_backend_agrees():
    """demo_heuristic_lander(continuous env) through the single-env facade; then the host-buffer path
    (b200gym_step_host with [n][2] float32 actions) against the device path."""
    import gym_b200
    import torch
    from oracle.oracle import lunar_heuristic
    env = gym_b200.make("LunarLanderContinuous-v2")
    s, info = env.reset(seed=1)
    total, steps = 0.0, 0
    while True:
        a = lunar_heuristic(s, continuous=True).astype(np.float32)
        assert env.action_space.contains(a)
        s, r, terminated, truncated, _ = env.step(a)
        total += r
        steps += 1
        if terminated or truncated:
            break
    assert total > 100, (total, steps)
    env.close()
    N = 512
    dev = gym_b200.vector.make("LunarLanderContinuous-v2", N, enable_wind=True, wind_idx=7, torque_idx=-7)
    host = gym_b200.vector.make("LunarLanderContinuous-v2", N, enable_wind=True, wind_idx=7, torque_idx=-7, backend="numpy")
    o1, _ = dev.reset(seed=2)
    o2, _ = host.reset(seed=2)
    assert np.array_equal(o1.cpu().numpy(), o2)
    rng = np.random.default_rng(0)
    for t in range(150):
        a = rng.uniform(-1, 1, size=(N, 2)).astype(np.float32)
        r1 = dev.step(torch.as_tensor(a, device=dev.device))
        r2 = host.step(a)
        for x, y in zip(r1[:4], r2[:4]):
            assert np.array_equal(x.cpu().numpy(), y)
    dev.close()
    host.close()


def test_wind_indices_default_to_numpy_global_generator():
    """LunarLander.__init__ (lunar_lander.py:234-235): wind_idx, torque_idx = np.random.randint(-9999, 9999),
    one pair per env object in construction order."""
    import gym_b200
    np.random.seed(123)
    want = [np.random.randint(-9999, 9999) for _ in range(2 * 6)]
    np.random.seed(123)
    env = gym_b200.vector.make("LunarLander-v2", 6, enable_wind=True)
    w, t = env.lunar_wind_idx()
    assert w.tolist() == want[0::2] and t.tolist() == want[1::2]
    env.close()


@pytest.mark.parametrize("env_id", ["LunarLander-v2", "BipedalWalkerHardcore-v3"])
def test_three_launch_step_matches_oracle_and_host_path(env_id, monkeypatch):
    """The three-launch step of the Box2D tasks (step kernel -> TOI kernel over the parked envs -> compacted reset
    kernel) bit for bit against the C oracle, which runs SolveTOI and the autoreset inline, and against the chunked
    host path (every chunk has its own parked-env / reset counters).  Random play at this size goes through both
    autoresets and TOI sub-steps."""
    import os

    import gym_b200
    import torch
    from oracle.oracle import OracleLunar, OracleWalker
    N, T = 2048, 220
    monkeypatch.setenv("B200GYM_HOST_CHUNKS", "3")
    dev = gym_b200.vector.make(env_id, N)
    host = gym_b200.vector.make(env_id, N, backend="numpy")
    orc = OracleLunar(N) if dev.discrete else OracleWalker(N, hardcore=True, max_episode_steps=dev.max_episode_steps)
    nthreads = min(8, os.cpu_count() or 1)
    o0, _ = dev.reset(seed=9)
    o1, _ = host.reset(seed=9)
    ref = orc.reset(seed=9)
    assert np.array_equal(o0.cpu().numpy(), ref) and np.array_equal(o1, ref)
    rng = np.random.default_rng(4)
    n_done = 0
    for t in range(T):
        a = rng.integers(0, 4, size=N) if dev.discrete else rng.uniform(-1, 1, (N, 4)).astype(np.float32)
        r0, r1, r2 = dev.step(torch.as_tensor(a, device=dev.device)), host.step(a), orc.step(a, nthreads=nthreads)
        for k in range(4):
            assert np.array_equal(r0[k].cpu().numpy(), r2[k]), f"step {t}, output {k}: device path"
            assert np.array_equal(r1[k], r2[k]), f"step {t}, output {k}: host path"
        done = r2[2] | r2[3]
        if done.any():
            assert np.array_equal(r0[4]["final_observation"].cpu().numpy()[done], r2[4][done])
            assert np.array_equal(np.stack(r1[4]["final_observation"][done]), r2[4][done])
        n_done += int(done.sum())
    assert n_done > N // 2
    calls, events = orc.toi_stats()
    assert events > 100 and calls > events
    for e in (dev, host, orc):
        e.close()
