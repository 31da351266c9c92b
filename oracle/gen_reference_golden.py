"""Freeze what the reference (openai/gym 0.26.2) returns in the comparisons of tests/test_oracle_vs_reference.py and
tests/test_gpu_reference_live.py, as tests/golden/reference/*.npz, so that those tests need no copy of the reference.

    python oracle/make_ref.py && python oracle/gen_reference_golden.py

Each case is the reference call a test compares against, with that test's seeds, sizes and actions; the oracle test
and the engine test share the SyncVectorEnv roll-outs.  Test infrastructure, not product code.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.ref_gym import import_reference  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference")
CLASSIC = ["CartPole-v1", "MountainCar-v0", "MountainCarContinuous-v0", "Pendulum-v1", "Acrobot-v1"]


def actions(env_id, rng, T, N):
    """Seeded random actions (stored with each case)."""
    if env_id.startswith("CartPole"):
        return rng.integers(0, 2, size=(T, N))
    if env_id.startswith(("MountainCar-", "Acrobot")):
        return rng.integers(0, 3, size=(T, N))
    lim = 2.5 if env_id.startswith("Pendulum") else 1.3
    return rng.uniform(-lim, lim, size=(T, N, 1)).astype(np.float32)


def describe_space(prefix, space):
    """A gym space as plain arrays (tests rebuild it with gym_b200.spaces and compare with ==)."""
    kind = type(space).__name__
    d = {f"{prefix}_kind": kind, f"{prefix}_shape": np.array(space.shape, np.int64), f"{prefix}_dtype": str(space.dtype)}
    if kind == "Box":
        d[f"{prefix}_low"], d[f"{prefix}_high"] = space.low, space.high
    elif kind == "Discrete":
        d[f"{prefix}_n"], d[f"{prefix}_start"] = int(space.n), int(space.start)
    elif kind == "MultiDiscrete":
        d[f"{prefix}_nvec"] = space.nvec
    else:
        raise TypeError(kind)
    return d


def sync_rollout(gym, env_id, N, T, seed, acts):
    """SyncVectorEnv of N envs: reset(seed), then T steps; everything a step returns, per step."""
    envs = gym.vector.SyncVectorEnv([lambda: gym.make(env_id, disable_env_checker=True) for _ in range(N)])
    obs0, info0 = envs.reset(seed=seed)
    assert info0 == {}
    D = envs.single_observation_space.shape[0]
    out = dict(actions=acts, obs0=obs0, obs=np.zeros((T, N, D), obs0.dtype), reward=np.zeros((T, N)),
               terminated=np.zeros((T, N), bool), truncated=np.zeros((T, N), bool),
               final_obs=np.zeros((T, N, D), obs0.dtype), final_mask=np.zeros((T, N), bool),
               info_keys=np.zeros(T, dtype="U128"))
    for t in range(T):
        o, r, te, tr, info = envs.step(acts[t])
        out["obs"][t], out["reward"][t], out["terminated"][t], out["truncated"][t] = o, r, te, tr
        assert out["reward"].dtype == r.dtype and te.dtype == tr.dtype == bool
        out["info_keys"][t] = ",".join(sorted(info.keys()))
        if "final_observation" in info:
            out["final_mask"][t] = info["_final_observation"]
            for i in np.flatnonzero(info["_final_observation"]):
                out["final_obs"][t, i] = info["final_observation"][i]
                assert info["final_info"][i] == {}   # the tests compare the engine's entries against {}
    for name, space in (("single_obs", envs.single_observation_space), ("single_act", envs.single_action_space),
                        ("obs", envs.observation_space), ("act", envs.action_space)):
        out.update(describe_space(name, space))
    envs.close()
    return out


def spaces_case(gym):
    """test_space_objects_sample_like_the_reference: bounds, seeded samples, batched samples."""
    out = {}
    for env_id in CLASSIC:
        ref = gym.make(env_id, disable_env_checker=True)
        out[f"{env_id}__obs_shape"] = np.array(ref.observation_space.shape, np.int64)
        out[f"{env_id}__obs_low"], out[f"{env_id}__obs_high"] = ref.observation_space.low, ref.observation_space.high
        ref.action_space.seed(5)
        out[f"{env_id}__samples"] = np.stack([np.asarray(ref.action_space.sample()) for _ in range(5)])
        rb = gym.vector.utils.batch_space(ref.action_space, 7)
        rb.seed(9)
        out[f"{env_id}__batch_sample"] = rb.sample()
        out[f"{env_id}__batch_type"] = type(rb).__name__
        out[f"{env_id}__batch_shape"] = np.array(rb.shape, np.int64)
        out[f"{env_id}__batch_dtype"] = str(rb.dtype)
        ref.close()
    return out


def info_wrappers_case(gym):
    """test_reference_info_wrappers_on_engine_infos: the reference's VectorListInfo(RecordEpisodeStatistics(
    SyncVectorEnv)) on CartPole-v1, and its step_api_compatibility on a SyncVectorEnv with max_episode_steps=7."""
    from gym.utils.step_api_compatibility import step_api_compatibility
    env_id, N, T, seed = "CartPole-v1", 16, 120, 5
    acts = actions(env_id, np.random.default_rng(9), T, N)
    a = gym.wrappers.VectorListInfo(gym.wrappers.RecordEpisodeStatistics(
        gym.vector.SyncVectorEnv([lambda: gym.make(env_id, disable_env_checker=True) for _ in range(N)])))
    a.reset(seed=seed)
    out = dict(actions=acts, keys=np.zeros((T, N), dtype="U64"), episode_r=np.zeros((T, N)),
               episode_l=np.zeros((T, N), np.int64), final_obs=np.zeros((T, N, 4), np.float32))
    for t in range(T):
        infos = a.step(acts[t])[4]
        assert isinstance(infos, list)
        for i, ia in enumerate(infos):
            out["keys"][t, i] = ",".join(sorted(ia.keys()))
            if "episode" in ia:
                out["episode_r"][t, i], out["episode_l"][t, i] = float(ia["episode"]["r"]), int(ia["episode"]["l"])
            if "final_observation" in ia:
                out["final_obs"][t, i] = ia["final_observation"]
    a.close()
    S = 20
    r = gym.vector.SyncVectorEnv([lambda: gym.make(env_id, disable_env_checker=True, max_episode_steps=7)
                                  for _ in range(N)])
    r.reset(seed=3)
    out.update(compat_dones=np.zeros((S, N), bool), compat_has_tl=np.zeros(S, bool), compat_tl=np.zeros((S, N), bool))
    for t in range(S):
        y = step_api_compatibility(r.step(acts[t]), output_truncation_bool=False, is_vector_env=True)
        assert len(y) == 4
        out["compat_dones"][t] = y[2]
        if "TimeLimit.truncated" in y[3]:
            out["compat_has_tl"][t] = True
            out["compat_tl"][t] = y[3]["TimeLimit.truncated"]
    r.close()
    return out


def main():
    gym = import_reference()
    os.makedirs(OUT, exist_ok=True)
    for env_id in CLASSIC:
        # test_gpu_reference_live.py::test_engine_equals_the_references_sync_vector_env and
        # test_oracle_vs_reference.py::test_oracle_bit_exact_against_reference_golden
        g = sync_rollout(gym, env_id, 8, 320, 31337, actions(env_id, np.random.default_rng(5), 320, 8))
        np.savez_compressed(os.path.join(OUT, f"sync_vector_{env_id}.npz"), seed=31337, **g)
    np.savez_compressed(os.path.join(OUT, "spaces.npz"), **spaces_case(gym))
    np.savez_compressed(os.path.join(OUT, "info_wrappers.npz"), **info_wrappers_case(gym))
    print("gym", gym.__version__, "numpy", np.__version__, "->", OUT)


if __name__ == "__main__":
    main()
