"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the
reference fixtures.  Needs a B200: `pytest -m gpu`.

Bars (BASELINE.json north_star): terminated / truncated / masks bit-exact;
float32 observations within 1e-5 relative, ELEMENT-wise, of the reference; float64
rewards within 1e-9.  What is actually measured is much tighter: the device evaluates
sin / cos exactly like glibc (csrc/glibc_trig.cuh), so MountainCar*, Pendulum and Acrobot
are bit-identical to the oracle -- float64 state included -- over 500 free-running steps;
CartPole keeps a faster small-angle kernel that is within 1 ulp of glibc (float32 outputs
identical in > 99.9 % of cases, float64 state within 1e-9).
"""
import numpy as np
import pytest

from conftest import GOLDEN, golden_names, load_golden

pytestmark = pytest.mark.gpu

ENV_IDS = ["CartPole-v1", "MountainCar-v0", "MountainCarContinuous-v0", "Pendulum-v1", "Acrobot-v1"]
OBS_RTOL = 1e-5   # per element
OBS_ATOL = 1e-7   # absolute floor for elements that pass through zero
REW_TOL = 1e-9


def _torch():
    import torch
    return torch


def _actions(env_id, rng, T, N, wild=False):
    if env_id.startswith("CartPole"):
        return rng.integers(0, 2, size=(T, N)).astype(np.int64)
    if env_id.startswith(("MountainCar-", "Acrobot")):
        return rng.integers(0, 3, size=(T, N)).astype(np.int64)
    lim = (3.0 if wild else 2.0) if env_id.startswith("Pendulum") else (1.5 if wild else 1.0)
    return rng.uniform(-lim, lim, size=(T, N, 1)).astype(np.float32)


def _close(a, b):
    """|a - b| <= 1e-7 + 1e-5 * |b| for every ELEMENT (north_star: "fp32 state within 1e-5 relative")."""
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    return np.abs(a64 - b64) <= OBS_ATOL + OBS_RTOL * np.abs(b64)


def _assert_obs(a, b, what):
    ok = _close(a, b)
    if not ok.all():
        a64, b64 = a.astype(np.float64), b.astype(np.float64)
        idx = np.argwhere(~ok)[0]
        raise AssertionError(
            f"{what}: {np.count_nonzero(~ok)} of {ok.size} observation elements outside rtol {OBS_RTOL}; "
            f"first at {tuple(idx)}: got {a64[tuple(idx)]!r} want {b64[tuple(idx)]!r}; "
            f"worst abs diff {np.max(np.abs(a64 - b64)):.3e}")


@pytest.mark.parametrize("env_id", ENV_IDS)
def test_free_run_parity_with_oracle(oracle_mod, env_id):
    """4096 envs x 500 steps, same seeds and actions, free-running from the first reset to the last step (no
    teacher forcing, no re-synchronisation -- Acrobot included): covers many autoresets (CartPole, Acrobot,
    MountainCarContinuous) and >= 2 TimeLimit cycles (Pendulum, MountainCar at 200)."""
    import gym_b200
    torch = _torch()
    N, T, seed = 4096, 500, 2024
    acts = _actions(env_id, np.random.default_rng(1), T, N, wild=True)
    env = gym_b200.vector.make(env_id, N)
    orc = oracle_mod.OracleVec(env_id, N)
    obs, infos = env.reset(seed=seed)
    assert infos == {}
    ref = orc.reset(seed=seed)
    assert obs.dtype == torch.float32 and tuple(obs.shape) == ref.shape
    _assert_obs(obs.cpu().numpy(), ref, "reset obs")
    if not env_id.startswith("Acrobot"):
        assert np.array_equal(obs.cpu().numpy(), ref), "reset observations must be bit-exact (pure PCG64 + cast)"
    dev_acts = torch.as_tensor(acts, device=env.device)
    n_done = n_trunc = 0
    exact = total = 0
    for t in range(T):
        o, r, te, tr, info = env.step(dev_acts[t])
        ro, rr, rte, rtr, rfo = orc.step(acts[t], nthreads=4)
        te_h, tr_h = te.cpu().numpy(), tr.cpu().numpy()
        assert te.dtype == torch.bool and tr.dtype == torch.bool and r.dtype == torch.float64
        assert np.array_equal(te_h, rte), f"step {t}: {np.count_nonzero(te_h != rte)} terminated mismatches"
        assert np.array_equal(tr_h, rtr), f"step {t}: {np.count_nonzero(tr_h != rtr)} truncated mismatches"
        o_h = o.cpu().numpy()
        _assert_obs(o_h, ro, f"step {t} obs")
        np.testing.assert_allclose(r.cpu().numpy(), rr, rtol=REW_TOL, atol=REW_TOL)
        done = rte | rtr
        assert np.array_equal(info["_final_observation"].cpu().numpy(), done)
        if done.any():
            _assert_obs(info["final_observation"].cpu().numpy()[done], rfo[done], f"step {t} final_observation")
        n_done += int(done.sum())
        n_trunc += int(rtr.sum())
        exact += int((o_h == ro).sum())
        total += o_h.size
    assert n_done > 0
    if env_id in ("Pendulum-v1", "MountainCar-v0"):
        assert n_trunc >= 2 * N
    # glibc-exact trigonometry: everything but CartPole (own small-angle kernel, <= 1 ulp) is bit-identical
    if env_id.startswith("CartPole"):
        assert exact / total > 0.999, f"only {exact / total:.5f} of the observations are bit-identical"
    else:
        assert exact == total, f"{total - exact} of {total} observation elements differ from the oracle"
    # persistent state agrees too (float64 integrator state, TimeLimit counters, PCG64 streams)
    st, el, rng = env.get_state()
    ost, oel = orc.get_state()
    assert np.array_equal(el.cpu().numpy(), oel)
    assert np.array_equal(rng.cpu().numpy().view(np.uint64), orc.get_rng())
    if env_id.startswith("CartPole"):
        np.testing.assert_allclose(st.cpu().numpy(), ost, rtol=1e-9, atol=1e-9)
    else:
        assert np.array_equal(st.cpu().numpy(), ost), "float64 integrator state must be bit-identical"
    env.close()
    orc.close()


@pytest.mark.parametrize("name", golden_names())
def test_reference_fixtures_through_the_engine(name):
    """The frozen outputs of the real reference (tests/golden) replayed on the GPU."""
    import gym_b200
    torch = _torch()
    g = load_golden(name)
    kwargs = {}
    if g["param0"] is not None:
        kwargs["g" if g["env_id"].startswith("Pendulum") else "goal_velocity"] = g["param0"]
    env = gym_b200.vector.make(g["env_id"], g["N"], max_episode_steps=g["max_episode_steps"], **kwargs)
    options = None
    if g["bounds"] is not None:
        keys = ("x_init", "y_init") if g["env_id"].startswith("Pendulum") else ("low", "high")
        options = dict(zip(keys, g["bounds"]))
    obs, _ = env.reset(seed=g["seed"], options=options)
    _assert_obs(obs.cpu().numpy(), g["obs0"], "reset obs")
    acts = torch.as_tensor(g["actions"], device=env.device)
    for t in range(g["T"]):
        o, r, te, tr, info = env.step(acts[t])
        assert np.array_equal(te.cpu().numpy(), g["terminated"][t]), f"step {t} terminated"
        assert np.array_equal(tr.cpu().numpy(), g["truncated"][t]), f"step {t} truncated"
        _assert_obs(o.cpu().numpy(), g["obs"][t], f"step {t} obs")
        np.testing.assert_allclose(r.cpu().numpy(), g["reward"][t], rtol=REW_TOL, atol=REW_TOL)
        m = g["final_mask"][t]
        assert np.array_equal(info["_final_observation"].cpu().numpy(), m)
        if m.any():
            _assert_obs(info["final_observation"].cpu().numpy()[m], g["final_obs"][t][m], f"step {t} final obs")
    env.close()


def test_device_seed_sequence_and_pcg64_known_answers(oracle_mod):
    """SeedSequence + PCG64 on the device: bit-exact integers against numpy's own values."""
    import gym_b200
    z = np.load(GOLDEN + "/rng_kat.npz")
    seeds = [(int(hi) << 64) | int(lo) for lo, hi in zip(z["seeds_lo"], z["seeds_hi"])]
    env = gym_b200.vector.make("CartPole-v1", len(seeds))
    env.seed(seeds)
    _, _, rng = env.get_state()
    rng = rng.cpu().numpy().view(np.uint64)
    orc = oracle_mod.OracleVec("CartPole-v1", len(seeds))
    orc.seed(seeds)
    assert np.array_equal(rng, orc.get_rng())
    # reset = 4 uniform draws per env from numpy's stream, cast to float32: bit-exact
    obs, _ = env.reset()
    for i, s in enumerate(seeds):
        gen = np.random.Generator(np.random.PCG64(np.random.SeedSequence(s)))
        assert np.array_equal(obs[i].cpu().numpy(), gen.uniform(-0.05, 0.05, size=4).astype(np.float32)), s
    # int seed fan-out with a base beyond 64 bits, and a sharded first_index
    base = 2**64 - 3
    env2 = gym_b200.vector.make("CartPole-v1", 8, first_index=5)
    o2, _ = env2.reset(seed=base)
    for i in range(8):
        gen = np.random.Generator(np.random.PCG64(np.random.SeedSequence(base + 5 + i)))
        assert np.array_equal(o2[i].cpu().numpy(), gen.uniform(-0.05, 0.05, size=4).astype(np.float32))
    env.close()
    env2.close()
    orc.close()


@pytest.mark.parametrize("env_id", ENV_IDS)
def test_numpy_backend_equals_torch_backend(env_id):
    """The host-buffer C-ABI path (b200gym_step_host) gives the same bits as the device path."""
    import gym_b200
    torch = _torch()
    N, T = 300, 260
    acts = _actions(env_id, np.random.default_rng(3), T, N)
    a = gym_b200.vector.make(env_id, N, max_episode_steps=60)
    b = gym_b200.vector.make(env_id, N, backend="numpy", max_episode_steps=60)
    oa, _ = a.reset(seed=17)
    ob, _ = b.reset(seed=17)
    assert isinstance(ob, np.ndarray) and np.array_equal(oa.cpu().numpy(), ob)
    saw_final = False
    for t in range(T):
        o1, r1, te1, tr1, i1 = a.step(torch.as_tensor(acts[t], device=a.device))
        o2, r2, te2, tr2, i2 = b.step(acts[t])
        assert o2.dtype == np.float32 and r2.dtype == np.float64 and te2.dtype == np.bool_ and tr2.dtype == np.bool_
        assert np.array_equal(o1.cpu().numpy(), o2) and np.array_equal(r1.cpu().numpy(), r2)
        assert np.array_equal(te1.cpu().numpy(), te2) and np.array_equal(tr1.cpu().numpy(), tr2)
        done = te2 | tr2
        if done.any():
            saw_final = True
            # reference info format: object arrays + masks (gym/vector/vector_env.py:208-258)
            assert i2["final_observation"].dtype == object and i2["final_info"].dtype == object
            assert np.array_equal(i2["_final_observation"], done) and np.array_equal(i2["_final_info"], done)
            fo = i1["final_observation"].cpu().numpy()
            for i in range(N):
                if done[i]:
                    assert np.array_equal(i2["final_observation"][i], fo[i]) and i2["final_info"][i] == {}
                else:
                    assert i2["final_observation"][i] is None and i2["final_info"][i] is None
        else:
            assert i2 == {}
    assert saw_final
    a.close()
    b.close()


def test_full_size_cartpole_properties(oracle_mod):
    """BASELINE config 2 size (2^20 envs): properties that do not need a full CPU replay."""
    import gym_b200
    torch = _torch()
    N, T, seed = 1 << 20, 64, 0
    gen = torch.Generator(device="cuda").manual_seed(0)
    acts = torch.randint(0, 2, (T, N), device="cuda", dtype=torch.int64, generator=gen)
    env = gym_b200.vector.make("CartPole-v1", N)
    twin = gym_b200.vector.make("CartPole-v1", N)
    # a shard of the same global batch: envs [3*2^18, 4*2^18)
    lo = 3 << 18
    shard = gym_b200.vector.make("CartPole-v1", 1 << 18, first_index=lo)
    sub = 4096
    orc = oracle_mod.OracleVec("CartPole-v1", sub)
    o, _ = env.reset(seed=seed)
    o2, _ = twin.reset(seed=seed)
    os_, _ = shard.reset(seed=seed)
    ro = orc.reset(seed=seed)
    assert torch.equal(o, o2) and torch.equal(o[lo:lo + (1 << 18)], os_)
    assert np.array_equal(o[:sub].cpu().numpy(), ro)
    x_thr, th_thr = 2.4, 12 * 2 * np.pi / 360
    total_done = 0
    for t in range(T):
        o, r, te, tr, info = env.step(acts[t])
        o2, r2, te2, tr2, _ = twin.step(acts[t])
        os_, rs, tes, trs, _ = shard.step(acts[t, lo:lo + (1 << 18)])
        # determinism (tests/envs/test_envs.py:60-115) and independence of the sharding
        assert torch.equal(o, o2) and torch.equal(te, te2) and torch.equal(r, r2)
        assert torch.equal(o[lo:lo + (1 << 18)], os_) and torch.equal(te[lo:lo + (1 << 18)], tes)
        # the first 4096 envs replayed on the CPU oracle
        ro, rr, rte, rtr, rfo = orc.step(acts[t, :sub].cpu().numpy(), nthreads=4)
        assert np.array_equal(te[:sub].cpu().numpy(), rte) and np.array_equal(tr[:sub].cpu().numpy(), rtr)
        _assert_obs(o[:sub].cpu().numpy(), ro, f"step {t}")
        # invariants over the whole batch
        assert bool((r == 1.0).all()) and not bool(tr.any())
        fo = info["final_observation"]
        # the float64 state crossed the threshold; after the float32 cast it is >= the float32 threshold
        out = (fo[:, 0].abs() >= np.float32(x_thr)) | (fo[:, 2].abs() >= np.float32(th_thr))
        assert torch.equal(out[te], torch.ones_like(out[te])), "terminated rows must violate a threshold"
        live = ~te
        assert bool((o[live][:, 0].abs() <= x_thr + 1e-6).all()) and bool((o[live][:, 2].abs() <= th_thr + 1e-6).all())
        # autoreset rows restart inside the reset box
        assert bool((o[te].abs() <= 0.05 + 1e-7).all())
        total_done += int(te.sum())
    assert total_done > N  # mean random-action episode is ~22 steps
    _, el, _ = env.get_state()
    assert int(el.max()) <= T and int(el.min()) >= 0
    for e in (env, twin, shard):
        e.close()
    orc.close()


@pytest.mark.parametrize("n", [1, 31, 257, 1000])
def test_ragged_batch_sizes(oracle_mod, n):
    """Batch sizes that do not fill a warp / a CTA (the tail CTA must mask correctly)."""
    import gym_b200
    torch = _torch()
    for env_id in ("CartPole-v1", "Pendulum-v1", "Acrobot-v1"):
        acts = _actions(env_id, np.random.default_rng(n), 40, n)
        env = gym_b200.vector.make(env_id, n)
        orc = oracle_mod.OracleVec(env_id, n)
        env.reset(seed=5)
        orc.reset(seed=5)
        for t in range(40):
            o, r, te, tr, _ = env.step(torch.as_tensor(acts[t], device=env.device))
            ro, rr, rte, rtr, _ = orc.step(acts[t])
            assert np.array_equal(te.cpu().numpy(), rte) and np.array_equal(tr.cpu().numpy(), rtr)
            _assert_obs(o.cpu().numpy(), ro, f"{env_id} n={n} step {t}")
        env.close()
        orc.close()


def test_state_roundtrip_and_teacher_forcing(oracle_mod):
    """set_state/get_state through the C ABI; one step from an injected oracle state."""
    import gym_b200
    torch = _torch()
    N = 512
    for env_id in ENV_IDS:
        orc = oracle_mod.OracleVec(env_id, N)
        orc.reset(seed=8)
        acts = _actions(env_id, np.random.default_rng(2), 30, N)
        for t in range(29):
            orc.step(acts[t])
        st, el = orc.get_state()
        env = gym_b200.vector.make(env_id, N)
        env.reset(seed=0)
        env.set_state(state=st, elapsed=el, rng=orc.get_rng())
        gst, gel, grng = env.get_state()
        assert np.array_equal(gst.cpu().numpy(), st) and np.array_equal(gel.cpu().numpy(), el)
        assert np.array_equal(grng.cpu().numpy().view(np.uint64), orc.get_rng())
        o, r, te, tr, _ = env.step(torch.as_tensor(acts[29], device=env.device))
        ro, rr, rte, rtr, _ = orc.step(acts[29])
        assert np.array_equal(te.cpu().numpy(), rte) and np.array_equal(tr.cpu().numpy(), rtr)
        _assert_obs(o.cpu().numpy(), ro, env_id)
        np.testing.assert_allclose(r.cpu().numpy(), rr, rtol=REW_TOL, atol=REW_TOL)
        env.close()
        orc.close()


@pytest.mark.parametrize("env_id", ENV_IDS)
def test_persistent_kernel_equals_simple_kernel(env_id, monkeypatch):
    """Kernel P (resident grid, per-thread cp.async prefetch, CTA-deferred resets; the default for large batches)
    against kernel A (one tile per CTA, plain loads): same arithmetic, so every output and the persistent state
    must be bit-identical.  N gives the resident grid several tiles per CTA plus a ragged last tile;
    max_episode_steps=40 makes the whole batch truncate in the same step twice (the dense inline-reset path and
    the overflow of the deferred-reset list), the terminations in between go through the deferred list; the
    action dtype cycles through int64 / int32 / uint8 (uint8 takes the register-prefetch path)."""
    import gym_b200
    torch = _torch()
    N, T = 148 * 256 * 9 + 178, 90
    envs = {}
    for k in ("a", "p", "l"):   # "l": the lean instantiation of kernel P (32-bit indices, no peer / episode code)
        monkeypatch.setenv("B200GYM_KERNEL", k)
        envs[k] = gym_b200.vector.make(env_id, N, max_episode_steps=40)
    monkeypatch.delenv("B200GYM_KERNEL")
    obs = {k: e.reset(seed=99)[0] for k, e in envs.items()}
    assert torch.equal(obs["a"], obs["p"]) and torch.equal(obs["a"], obs["l"])
    ea, ep, el_ = envs["a"], envs["p"], envs["l"]
    acts = torch.as_tensor(_actions(env_id, np.random.default_rng(11), T, N, wild=True), device=ea.device)
    dtypes = [torch.int64, torch.int32, torch.uint8] if ea.discrete else [torch.float32]
    n_done = 0
    for t in range(T):
        a = acts[t].to(dtypes[t % len(dtypes)])
        ra = ea.step(a)
        m = ra[4]["_final_observation"]
        for name, e in (("p", ep), ("l", el_)):
            rb = e.step(a)
            for x, y in zip(ra[:4], rb[:4]):
                assert torch.equal(x, y), f"kernel {name} step {t}"
            assert torch.equal(m, rb[4]["_final_observation"])
            assert torch.equal(ra[4]["final_observation"][m], rb[4]["final_observation"][m])
        n_done += int(m.sum())
    assert n_done >= 2 * N
    for x, y, z in zip(ea.get_state(), ep.get_state(), el_.get_state()):
        assert torch.equal(x, y), "kernel p state"
        assert torch.equal(x, z), "kernel l state"
    for e in envs.values():
        e.close()


def test_device_sin_cos_are_bit_identical_to_the_hosts_libm():
    """csrc/glibc_trig.cuh compiled by nvcc, on the device, against math.sin / math.cos of this process (the libm the
    reference's results come from): every bit, over the ranges the envs produce and beyond."""
    import ctypes
    import math
    from gym_b200 import _lib
    torch = _torch()
    lib = _lib.load()
    rng = np.random.default_rng(3)
    parts = [rng.uniform(-s, s, 200000) for s in (0.2, 1.0, 3.2, 10.0, 100.0, 1e6, 1.05e8, 1e-7)]
    parts.append(np.array([0.0, -0.0, 0.126, -0.126, 0.855469, 2.426265, math.pi, math.pi / 2, 105414349.0, 1e-300]))
    x = np.concatenate(parts)
    xd = torch.as_tensor(x, device="cuda")
    sn, cs, sq = torch.empty_like(xd), torch.empty_like(xd), torch.empty_like(xd)
    _lib.check(lib.b200gym_selftest_trig(ctypes.c_void_p(xd.data_ptr()), x.size, ctypes.c_void_p(sn.data_ptr()),
                                         ctypes.c_void_p(cs.data_ptr()), ctypes.c_void_p(sq.data_ptr()), None))
    torch.cuda.synchronize()
    ws = np.array([math.sin(v) for v in x])
    wc = np.array([math.cos(v) for v in x])
    wq = np.array([math.pow(v, 2.0) for v in x])      # what `x**2` is in the reference; differs from x*x in ~0.09 %
    bad_s = np.flatnonzero(sn.cpu().numpy().view(np.int64) != ws.view(np.int64))
    bad_c = np.flatnonzero(cs.cpu().numpy().view(np.int64) != wc.view(np.int64))
    bad_q = np.flatnonzero(sq.cpu().numpy().view(np.int64) != wq.view(np.int64))
    assert bad_s.size == 0 and bad_c.size == 0, (bad_s[:5], x[bad_s[:5]], bad_c[:5], x[bad_c[:5]])
    assert bad_q.size == 0, (bad_q[:5], x[bad_q[:5]])
    assert np.count_nonzero(wq != x * x) > 100


def test_constant_division_fast_path_is_ieee_exact():
    """csrc/envs.cuh:div_by_const (Markstein residual correction with a folded reciprocal) must be
    bit-identical to IEEE division: 2^28 pseudo-random doubles x 4 divisors on the device."""
    import ctypes
    from gym_b200 import _lib
    lib = _lib.load()
    total = 0
    for seed in (1, 2, 3, 4):
        bad = ctypes.c_int64(-1)
        _lib.check(lib.b200gym_selftest(0, 1 << 26, seed, ctypes.byref(bad)))
        total += bad.value
    assert total == 0
