"""Time the REAL reference's vector envs on this machine's host cores and print ONE JSON object.

    python oracle/ref_timing.py [--env CartPole-v1] [--seconds 1.0] [--async-workers N]

SURVEY.md 8(d) "CPU path timing": ``gym.vector.SyncVectorEnv`` (a serial Python loop: 1 core) at num_envs in
{4, 1024} and ``gym.vector.AsyncVectorEnv`` (one worker process per env, shared-memory observations) with one env
per host core, >= `seconds` of wall time each after 3 warm-up steps, random actions from ``action_space.sample()``,
autoreset on.  Runs in its own process (bench.py spawns it before CUDA is touched: AsyncVectorEnv forks).
Test / measurement infrastructure: uses ``oracle/_ref``, never the engine.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.ref_gym import import_reference, reference_path  # noqa: E402


def host_cores():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def run(envs, n, seconds, min_steps=5):
    envs.reset(seed=0)
    envs.action_space.seed(0)
    acts = [envs.action_space.sample() for _ in range(8)]
    for k in range(3):
        envs.step(acts[k])
    steps, t0 = 0, time.perf_counter()
    while True:
        envs.step(acts[steps % 8])
        steps += 1
        el = time.perf_counter() - t0
        if steps >= min_steps and el >= seconds:
            break
    envs.close()
    return {"num_envs": n, "value": n * steps / el, "unit": "env-steps/s", "vector_steps": steps, "seconds": el}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--env", default="CartPole-v1")
    p.add_argument("--seconds", type=float, default=1.0)
    p.add_argument("--async-workers", type=int, default=0, help="0 = one per host core (at most 64)")
    args = p.parse_args()
    gym = import_reference()
    cores = host_cores()
    mk = lambda: gym.make(args.env, disable_env_checker=True)  # noqa: E731
    out = {"reference": f"openai/gym {gym.__version__} (unmodified, {reference_path()})", "env": args.env,
           "host_cores": cores, "sync": [], "async": None}
    for n in (4, 1024):
        r = run(gym.vector.SyncVectorEnv([mk] * n), n, args.seconds)
        r["cores"] = 1
        out["sync"].append(r)
    workers = args.async_workers or min(cores, 64)
    try:
        r = run(gym.vector.AsyncVectorEnv([mk] * workers, shared_memory=True), workers, args.seconds)
        r["cores"] = workers
        out["async"] = r
    except Exception as exc:  # a box that cannot fork that many workers still reports the sync numbers
        out["async"] = {"error": repr(exc)[:200]}
    # BASELINE.json configs[0]: SyncVectorEnv of 4 CartPole-v1 envs, 1000 random-action steps
    envs = gym.vector.SyncVectorEnv([lambda: gym.make("CartPole-v1", disable_env_checker=True)] * 4)
    envs.reset(seed=0)
    envs.action_space.seed(0)
    t0 = time.perf_counter()
    for _ in range(1000):
        envs.step(envs.action_space.sample())
    out["config0_ms"] = 1e3 * (time.perf_counter() - t0)
    envs.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
