"""Oracle (and the host-side space objects) against the reference.

The first two tests compare with what the reference (openai/gym 0.26.2) returned for the same seeds and actions,
stored in tests/golden/reference by oracle/gen_reference_golden.py.  The registry test runs gym's own registry, so it
needs the reference installed in oracle/_ref (oracle/make_ref.py) and skips without it.
"""
import numpy as np
import pytest

from conftest import load_reference_golden
from oracle import ref_gym

CLASSIC = ["CartPole-v1", "MountainCar-v0", "MountainCarContinuous-v0", "Pendulum-v1", "Acrobot-v1"]


@pytest.mark.parametrize("env_id", CLASSIC)
def test_oracle_bit_exact_against_reference_golden(oracle_mod, env_id):
    """Against the golden roll-out of the reference's SyncVectorEnv: 8 envs, seed 31337, 320 random steps
    (tests/golden/reference/sync_vector_<id>.npz, also the one the engine is checked against in
    tests/test_gpu_reference_live.py)."""
    g = load_reference_golden(f"sync_vector_{env_id}")
    N, T, seed = 8, 320, 31337
    acts = g["actions"]
    assert acts.shape[:2] == (T, N) and int(g["seed"]) == seed
    v = oracle_mod.OracleVec(env_id, N)
    ref_obs = g["obs0"]
    obs = v.reset(seed=seed)
    if env_id.startswith("Acrobot"):
        np.testing.assert_allclose(obs, ref_obs, rtol=2e-7)
    else:
        assert np.array_equal(obs, ref_obs)
    for t in range(T):
        ro, rr, rte, rtr = g["obs"][t], g["reward"][t], g["terminated"][t], g["truncated"][t]
        o, r, te, tr, fo = v.step(acts[t])
        assert np.array_equal(te, rte) and np.array_equal(tr, rtr)
        assert np.array_equal(r, rr)
        done = te | tr
        if env_id.startswith("Acrobot") and done.any():
            np.testing.assert_allclose(o, ro, rtol=2e-7)  # numpy's float32 trig on reset rows
            assert np.array_equal(o[~done], ro[~done])
        else:
            assert np.array_equal(o, ro)
        assert np.array_equal(g["final_mask"][t], done)
        for i in np.flatnonzero(done):
            assert np.array_equal(g["final_obs"][t, i], fo[i])
    v.close()


def test_space_objects_sample_like_the_reference():
    """Bounds, 5 samples after action_space.seed(5), one batch_space(7) sample after seed(9), per env
    (tests/golden/reference/spaces.npz)."""
    from gym_b200 import spaces
    from gym_b200.envs import KINDS
    g = load_reference_golden("spaces")
    for kind, env_id in enumerate(CLASSIC):
        ref = {k.split("__", 1)[1]: v for k, v in g.items() if k.startswith(env_id + "__")}
        obs_space, act_space = KINDS[kind].spaces(None)
        assert obs_space.shape == tuple(ref["obs_shape"])
        assert np.array_equal(obs_space.low, ref["obs_low"])
        assert np.array_equal(obs_space.high, ref["obs_high"])
        act_space.seed(5)
        for k in range(5):
            assert np.array_equal(np.asarray(act_space.sample()), ref["samples"][k])
        mb = spaces.batch_space(act_space, 7)
        mb.seed(9)
        assert np.array_equal(mb.sample(), ref["batch_sample"])
        assert (type(mb).__name__ == str(ref["batch_type"]) and mb.shape == tuple(ref["batch_shape"])
                and str(mb.dtype) == str(ref["batch_dtype"]))


@pytest.mark.skipif(ref_gym.reference_path() is None, reason="needs the reference installed in oracle/_ref")
def test_plugin_registers_engine_ids_in_the_real_registry():
    """gym/envs/registration.py:266-309,434-499: the ids resolve through gym's own registry and gym.make
    reaches the engine's constructor (which refuses to run without a B200: no CPU fallback)."""
    gym = ref_gym.import_reference()
    import gym_b200
    from gym_b200 import error, plugin
    ids = plugin.register_all()
    assert "B200/CartPole-v1" in ids and "B200/BipedalWalkerHardcore-v3" in ids
    for env_id in ids:
        s = gym.spec(env_id)
        assert s.namespace == "B200" and s.entry_point == "gym_b200.plugin:make_env"
        assert s.max_episode_steps is None and s.order_enforce is False and s.disable_env_checker is True
        assert s.kwargs == {"env_id": env_id.split("/", 1)[1]}
        assert s.reward_threshold == gym_b200.spec(s.kwargs["env_id"]).reward_threshold
    # the reference's own ids are untouched
    assert gym.spec("CartPole-v1").entry_point == "gym.envs.classic_control.cartpole:CartPoleEnv"
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(error.DependencyNotInstalled):
            gym.make("B200/CartPole-v1")
    else:
        env = gym.make("B200/CartPole-v1")
        obs, info = env.reset(seed=0)
        assert obs.shape == (4,) and env.spec.id == "B200/CartPole-v1"
        env.close()
