"""The engine against the reference (openai/gym 0.26.2) on the GPU.

What the reference's `SyncVectorEnv` and info wrappers returned for the seeds and actions used here is stored in
tests/golden/reference (oracle/gen_reference_golden.py), so the trajectory and wrapper comparisons need no copy of
the reference.  The checks that run the reference's own code on the engine -- `check_env`, its registry, its wrappers
and `gym.vector.VectorEnv` subclassing -- need the reference installed in oracle/_ref (oracle/make_ref.py): those
tests skip without it, and the wrapper test then checks the engine's own wrappers only.
"""
import numpy as np
import pytest

from conftest import load_reference_golden
from oracle import ref_gym

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(ref_gym.reference_path() is None,
                                     reason="needs the reference installed in oracle/_ref")

CLASSIC = ["CartPole-v1", "MountainCar-v0", "MountainCarContinuous-v0", "Pendulum-v1", "Acrobot-v1"]


@pytest.fixture(scope="module")
def gym():
    return ref_gym.import_reference()


def golden_space(g, prefix):
    """The reference's space stored under `prefix`, rebuilt as a gym_b200.spaces object."""
    from gym_b200 import spaces
    kind = str(g[f"{prefix}_kind"])
    if kind == "Box":
        return spaces.Box(g[f"{prefix}_low"], g[f"{prefix}_high"], shape=tuple(g[f"{prefix}_shape"]),
                          dtype=np.dtype(str(g[f"{prefix}_dtype"])).type)
    if kind == "Discrete":
        return spaces.Discrete(int(g[f"{prefix}_n"]), start=int(g[f"{prefix}_start"]))
    return spaces.MultiDiscrete(g[f"{prefix}_nvec"], dtype=np.dtype(str(g[f"{prefix}_dtype"])).type)


@pytest.mark.parametrize("env_id", CLASSIC)
def test_engine_equals_the_references_sync_vector_env(env_id):
    """tests/vector/test_vector_env.py:14-53 of the reference compares AsyncVectorEnv with SyncVectorEnv step by
    step; here the engine takes AsyncVectorEnv's place against SyncVectorEnv's stored outputs
    (tests/golden/reference/sync_vector_<id>.npz).  Flags, masks and rewards identical; float32 observations
    identical except where CUDA's float64 sin/cos differ from glibc's by an ulp (bounded at 1e-5 relative)."""
    import gym_b200
    g = load_reference_golden(f"sync_vector_{env_id}")
    N, T, seed = 8, 320, 31337
    acts = g["actions"]
    assert acts.shape[:2] == (T, N) and int(g["seed"]) == seed
    eng = gym_b200.vector.make(env_id, N, backend="numpy")
    assert eng.is_vector_env
    assert eng.single_observation_space == golden_space(g, "single_obs")
    assert eng.single_action_space == golden_space(g, "single_act")
    assert eng.observation_space == golden_space(g, "obs") and eng.action_space == golden_space(g, "act")
    o, info = eng.reset(seed=seed)
    assert info == {}   # so was the reference's
    np.testing.assert_allclose(o, g["obs0"], rtol=1e-5, atol=1e-7)
    n_done = exact = total = 0
    for t in range(T):
        ro, rr, rte, rtr = g["obs"][t], g["reward"][t], g["terminated"][t], g["truncated"][t]
        o, r, te, tr, info = eng.step(acts[t])
        assert np.array_equal(te, rte) and np.array_equal(tr, rtr), f"step {t}"
        np.testing.assert_allclose(r, rr, rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(o, ro, rtol=1e-5, atol=1e-6, err_msg=f"step {t}")
        assert o.dtype == ro.dtype and r.dtype == rr.dtype and te.dtype == rte.dtype
        rkeys = set(str(g["info_keys"][t]).split(",")) - {""}
        assert set(info.keys()) == rkeys, f"step {t}: {info.keys()} vs {rkeys}"
        if "final_observation" in rkeys:
            assert np.array_equal(info["_final_observation"], g["final_mask"][t])
            for i in np.flatnonzero(g["final_mask"][t]):
                np.testing.assert_allclose(info["final_observation"][i], g["final_obs"][t, i], rtol=1e-5, atol=1e-6)
                assert info["final_info"][i] == {}   # the reference's final_info entries are all {} here
            n_done += int(g["final_mask"][t].sum())
        exact += int((o == ro).sum())
        total += o.size
    # Pendulum / MountainCarContinuous only truncate (200 / 999); a random Acrobot rarely swings up within 320 steps
    assert n_done > 0 or env_id.startswith(("Pendulum", "MountainCarContinuous", "Acrobot"))
    if not env_id.startswith("Acrobot"):
        assert exact / total > 0.999
    eng.close()


@needs_reference
@pytest.mark.parametrize("env_id", CLASSIC)
def test_reference_check_env_accepts_the_engine(gym, env_id):
    """gym/utils/env_checker.py:255-320 run, unmodified, on the single-env facade (a real gym.Env subclass)."""
    import warnings

    from gym.utils.env_checker import check_env

    from gym_b200.gym_compat import GymEnv
    env = GymEnv(env_id)
    assert isinstance(env, gym.Env)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        check_env(env, skip_render_check=True)
    # the generator the checker looked at is the env's own device stream: same seed -> same position
    env.reset(seed=123)
    a = env.np_random.bit_generator.state
    env.reset(seed=123)
    assert env.np_random.bit_generator.state == a
    env.close()


@needs_reference
def test_gym_make_resolves_engine_ids(gym):
    """gym/envs/registration.py:502-691: `gym.make("B200/<id>")` goes through the reference's registry into the
    engine, and the result behaves like the reference env of the same id under the same seed.  The vector facade
    is a real `gym.vector.VectorEnv` with the reference's own space objects."""
    from gym_b200 import plugin
    from gym_b200.gym_compat import GymVectorEnv
    for env_id in CLASSIC:
        eng = GymVectorEnv(env_id, 8, backend="numpy")
        ref = gym.vector.SyncVectorEnv([lambda: gym.make(env_id, disable_env_checker=True) for _ in range(8)])
        assert isinstance(eng, gym.vector.VectorEnv) and eng.is_vector_env
        assert eng.single_observation_space == ref.single_observation_space
        assert eng.single_action_space == ref.single_action_space
        assert eng.observation_space == ref.observation_space and eng.action_space == ref.action_space
        eng.close()
        ref.close()
    ids = plugin.register_all() if "B200/CartPole-v1" not in gym.envs.registry else list(gym.envs.registry)
    assert "B200/CartPole-v1" in ids
    env = gym.make("B200/CartPole-v1")
    ref = gym.make("CartPole-v1", disable_env_checker=True)
    assert isinstance(env, gym.Env) and env.spec.id == "B200/CartPole-v1"
    assert env.observation_space == ref.observation_space and env.action_space == ref.action_space
    o, _ = env.reset(seed=11)
    ro, _ = ref.reset(seed=11)
    assert np.array_equal(o, ro)
    for t in range(60):
        a = t % 2
        o, r, te, tr, _ = env.step(a)
        ro, rr, rte, rtr, _ = ref.step(a)
        assert np.array_equal(o, ro) and r == rr and te == rte and tr == rtr
        if te or tr:
            break
    with pytest.raises(Exception):
        env.step(7)       # cartpole.py:132 asserts; the engine raises InvalidAction
    env.close()
    ref.close()


def test_reference_info_wrappers_on_engine_infos():
    """What the reference's own VectorListInfo (gym/wrappers/vector_list_info.py:56-111) and RecordEpisodeStatistics
    (record_episode_statistics.py:79-151) produce around its SyncVectorEnv (tests/golden/reference/info_wrappers.npz)
    must come out of the engine's device-side re-implementations of the same wrappers (torch backend); where the
    reference is installed, also out of the reference's wrappers around the engine (numpy backend)."""
    import torch

    import gym_b200
    from gym_b200 import wrappers as own
    g = load_reference_golden("info_wrappers")
    env_id, N, T, seed = "CartPole-v1", 16, 120, 5
    acts = g["actions"]
    assert acts.shape == (T, N)
    have_ref = ref_gym.reference_path() is not None
    c = own.VectorListInfo(own.RecordEpisodeStatistics(gym_b200.vector.make(env_id, N)))
    c.reset(seed=seed)
    b = None
    if have_ref:
        from gym_b200.gym_compat import GymVectorEnv
        gym = ref_gym.import_reference()
        b = gym.wrappers.VectorListInfo(gym.wrappers.RecordEpisodeStatistics(GymVectorEnv(env_id, N, backend="numpy")))
        b.reset(seed=seed)
    episodes = 0
    for t in range(T):
        rc = c.step(torch.as_tensor(acts[t], device="cuda"))
        rb = b.step(acts[t]) if b is not None else None
        assert isinstance(rc[4], list) and (rb is None or isinstance(rb[4], list))
        for i in range(N):
            ia, ic = set(str(g["keys"][t, i]).split(",")) - {""}, rc[4][i]
            assert ia - {"final_info"} == set(ic.keys()) - {"final_info"}, f"step {t} env {i}"
            others = [ic]
            if rb is not None:
                ib = rb[4][i]
                assert ia == set(ib.keys()), f"step {t} env {i}: {ia} vs {ib.keys()}"
                others.append(ib)
            if "episode" in ia:
                episodes += 1
                for other in others:
                    assert float(other["episode"]["r"]) == g["episode_r"][t, i]
                    assert int(other["episode"]["l"]) == g["episode_l"][t, i]
            if "final_observation" in ia:
                for other in others:
                    assert np.array_equal(g["final_obs"][t, i], np.asarray(other["final_observation"]))
    assert episodes > 10
    # the 4-tuple API: the engine's converter against the reference's (gym/utils/step_api_compatibility.py:24-161)
    # on a SyncVectorEnv with max_episode_steps=7; where installed, the reference's converter on the engine too
    e = gym_b200.vector.make(env_id, N, backend="numpy", max_episode_steps=7)
    e.reset(seed=3)
    for t in range(20):
        five = e.step(acts[t])
        converted = [own.step_api_compatibility(tuple(five[:4]) + (dict(five[4]),), output_truncation_bool=False)]
        if have_ref:
            from gym.utils.step_api_compatibility import step_api_compatibility as ref_compat
            converted.append(ref_compat(five, output_truncation_bool=False, is_vector_env=True))
        for z in converted:
            assert len(z) == 4 and np.array_equal(z[2], g["compat_dones"][t])
            # the key only exists in steps where some env finished (step_api_compatibility.py:114-118)
            assert ("TimeLimit.truncated" in z[3]) == bool(g["compat_has_tl"][t])
            if g["compat_has_tl"][t]:
                assert np.array_equal(z[3]["TimeLimit.truncated"], g["compat_tl"][t])
    for w in (b, c, e):
        if w is not None:
            w.close()
