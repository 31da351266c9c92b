#!/usr/bin/env python
"""bench.py -- env-steps/sec of the fused step kernel (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--env ID] [--log2-envs k]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): CartPole-v1, num_envs = 2^20 per GPU, random int64 actions resident in
HBM, fused step + TimeLimit + autoreset; a "step" is one vector step of the whole batch (one kernel launch per GPU).
For N > 1 (launched by torchrun, one rank per GPU) every rank owns 2^20 envs of a global batch and every step ends
with every rank holding the GLOBAL (obs, reward, terminated, truncated): the all-gather is fused into the step
kernel (bulk pushes over NVLink peer memory + one flag exchange) -- weak scaling; `strong_scaling` on the same line
is BASELINE.json configs[4] (2^23 envs in total, split over the N GPUs).

Prints ONE JSON line (rank 0).  Keys beyond the base contract:
  ms_per_step          N=1: MEDIAN of the K per-step CUDA-event times (L2 flushed before every step); the mean is
                       `ms_per_step_mean`.  N>1: the K steps back to back between barriers, max over ranks, / K.
  roofline             algorithmic bytes per launch / median kernel time against MEASURED_PEAKS.json's hbm_gbs
  cpu_baseline         the CPU oracle (C port of the reference path) on all host cores, bounded sample
  cpu_baseline_python  the REAL reference (oracle/_ref: unmodified openai/gym 0.26.2): SyncVectorEnv at 4 and 1024
                       envs (1 core: it is a serial Python loop), AsyncVectorEnv with one worker per core
  e2e                  the same metric through the public numpy-backend API: pinned host actions in, all results
                       to host memory, copies inside the timed region
  configs              (N=1) short runs of BASELINE.json configs[2] and [3]: Pendulum-v1 / Acrobot-v1 /
                       MountainCar-v0 at 2^18 envs, LunarLander-v2 / BipedalWalker-v3 at 2^16
  gather_verified      (N>1) every rank checks, per peer, a checksum of that peer's rows in ITS gathered copy
                       against the checksum the peer computed over its own rows

--dump-outputs DIR (N=1, --impl b200) writes what the last timed step returned as DIR/<name>.npy: obs, reward, terminated,
truncated (0/1) and final_observation (zero where the env did not finish), float32 or float64.  Above 64 MB in all,
the same seeded sample of env rows is taken from every array and its indices are written as rows.npy.  The inputs
(reset seed, action generator seed) are fixed, so two builds run with the same arguments can be compared output for
output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

ENV_ID = "CartPole-v1"
LOG2_ENVS = 20
# Algorithmic HBM bytes per env-step (DESIGN.md section 4): persistent state round trip + mandatory API I/O.
#   CartPole: read state 4 x f64 (32) + TimeLimit counter (4) + action int64 (8)            = 44
#             write state (32) + counter (4) + obs 4 x f32 (16) + reward f64 (8) + 2 flags (2) = 62  -> 106
# (SURVEY.md 8(d) counts 102 B with a float32 reward; we emit the reference's float64.)
BYTES_PER_ENV_STEP = {"CartPole-v1": 106, "CartPole-v0": 106, "Pendulum-v1": 16 * 2 + 8 + 4 + 12 + 8 + 2,
                      "Acrobot-v1": 32 * 2 + 8 + 8 + 24 + 8 + 2, "MountainCar-v0": 16 * 2 + 8 + 8 + 8 + 8 + 2,
                      "MountainCarContinuous-v0": 16 * 2 + 8 + 4 + 8 + 8 + 2,
                      # LunarLander: 103-word solver record r+w, PCG64 state (2 draws/step), counter, action, outputs
                      "LunarLander-v2": 101 * 4 * 2 + 32 + 16 + 8 + 8 + 32 + 8 + 2,
                      # BipedalWalker: 130-word record r+w (the 200 terrain words are read on demand), action, outputs
                      "BipedalWalker-v3": 130 * 4 * 2 + 8 + 16 + 96 + 8 + 2}
BYTES_PER_ENV_STEP["LunarLanderContinuous-v2"] = BYTES_PER_ENV_STEP["LunarLander-v2"]
BYTES_PER_ENV_STEP["BipedalWalkerHardcore-v3"] = BYTES_PER_ENV_STEP["BipedalWalker-v3"] + 4
# what bounds each kernel (ncu summaries in profiles/): the HBM fraction is only meaningful for the first group
BOUND = {"CartPole-v1": "hbm", "CartPole-v0": "hbm", "Pendulum-v1": "hbm (latency: 1 wave at 2^18)",
         "MountainCar-v0": "hbm (latency: 1 wave at 2^18)", "MountainCarContinuous-v0": "hbm (latency: 1 wave at 2^18)",
         "Acrobot-v1": "fp64 pipe / issue slots (4 x RK4 stage, 21 glibc-exact sin/cos + 12 glibc-exact pow(x, 2) per env-step)",
         "LunarLander-v2": "dependent-instruction latency under divergence (serial Gauss-Seidel solve + TOI sub-steps per env); "
                           "issue-slot utilisation 0.22 (step kernel) / 0.04 (TOI kernel), profiles/r2b_box2d_toi_kernel_sweep.txt",
         "LunarLanderContinuous-v2": "dependent-instruction latency under divergence (serial Gauss-Seidel solve + TOI sub-steps per env)",
         "BipedalWalker-v3": "dependent-instruction latency under divergence (serial Gauss-Seidel solve + TOI sub-steps per env); "
                             "issue-slot utilisation 0.27 (step kernel) / 0.13 (TOI kernel), profiles/r2b_box2d_toi_kernel_sweep.txt",
         "BipedalWalkerHardcore-v3": "dependent-instruction latency under divergence (serial Gauss-Seidel solve + TOI sub-steps per env)"}
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture (2^20 envs)
NCU_DRAM = {"file": "profiles/r2b_cartpole_step_kernel_L_40reg_ncu_full.txt", "read": 52.76e6, "write": 22.86e6}
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
DUMP_LIMIT_BYTES = 64 << 20
EXTRA_CONFIGS = [("Pendulum-v1", 18, 300), ("Acrobot-v1", 18, 300), ("MountainCar-v0", 18, 300),
                 ("LunarLander-v2", 16, 150), ("BipedalWalker-v3", 16, 60)]


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=1000, help="timed steps (>= 1)")
    p.add_argument("--warmup", type=int, default=100)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--env", default=ENV_ID)
    p.add_argument("--log2-envs", type=int, default=LOG2_ENVS, help="envs per GPU = 2**k")
    p.add_argument("--log2-total-strong", type=int, default=23, help="strong-scaling total (BASELINE configs[4])")
    p.add_argument("--e2e-steps", type=int, default=200)
    p.add_argument("--cpu-seconds", type=float, default=10.0, help="budget of the cpu_baseline sample")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-extra", action="store_true", help="skip the configs[2]/[3] lines and the strong-scaling run")
    p.add_argument("--gather", default="p2p", choices=["p2p", "nccl"],
                   help="N>1 exchange: fused NVLink peer pushes in the step kernel, or NCCL all-gather")
    p.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and (args.gpus != 1 or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        p.error("--dump-outputs takes --gpus 1 and a single process")
    if args.dump_outputs and args.impl != "b200":
        p.error("--dump-outputs dumps the B200 path's outputs: it takes --impl b200")
    return args


# --------------------------------------------------------------------------- helpers
class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md)."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.QUERY}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def is_box2d(env_id):
    return env_id.startswith(("LunarLander", "BipedalWalker"))


def random_actions_np(env_id, n, rng):
    if env_id.startswith("LunarLanderContinuous"):
        return rng.uniform(-1.0, 1.0, size=(n, 2)).astype(np.float32)
    if env_id.startswith("LunarLander"):
        return rng.integers(0, 4, size=n).astype(np.int64)
    if env_id.startswith("BipedalWalker"):
        return rng.uniform(-1.0, 1.0, size=(n, 4)).astype(np.float32)
    from oracle.oracle import ENV_IDS, KINDS, lib
    kind = KINDS[ENV_IDS[env_id][0]]
    nact = lib().orc_num_actions(kind)
    if nact:
        return rng.integers(0, nact, size=n).astype(np.int64)
    return rng.uniform(-2.0, 2.0, size=(n, 1)).astype(np.float32)


def make_oracle(env_id, n):
    """The C port of the reference path for `env_id` (oracle/): one object stepping n envs on host threads."""
    from oracle.oracle import OracleLunar, OracleVec, OracleWalker
    if env_id.startswith("LunarLander"):
        return OracleLunar(n, continuous="Continuous" in env_id)
    if env_id.startswith("BipedalWalker"):
        hard = "Hardcore" in env_id
        return OracleWalker(n, hardcore=hard, max_episode_steps=2000 if hard else 1600)
    return OracleVec(env_id, n)


def cpu_oracle_throughput(env_id, n, seconds, threads, min_steps=3):
    """Time the C port of the reference path (oracle/) on the host cores: bounded sample."""
    rng = np.random.default_rng(0)
    v = make_oracle(env_id, n)
    v.reset(seed=0)
    pool = [random_actions_np(env_id, n, rng) for _ in range(4)]
    kw = {"nthreads": threads}
    v.step(pool[0], **kw)  # warm-up
    steps, t0 = 0, time.perf_counter()
    while True:
        v.step(pool[steps % 4], **kw)
        steps += 1
        el = time.perf_counter() - t0
        if steps >= min_steps and el >= seconds:
            break
        if steps >= 2000:
            break
    v.close()
    return n * steps / el, steps, el


def start_python_reference(env_id):
    """Spawn oracle/ref_timing.py (the REAL reference's SyncVectorEnv / AsyncVectorEnv) in its own process."""
    script = os.path.join(ROOT, "oracle", "ref_timing.py")
    if is_box2d(env_id):
        return None  # box2d-py is not installable here: the reference cannot construct these envs
    try:
        return subprocess.Popen([sys.executable, script, "--env", env_id, "--seconds", "1.0"],
                                stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    except Exception:
        return None


def collect_python_reference(proc, timeout=180):
    if proc is None:
        return {"unavailable": "the reference cannot construct this env here (box2d-py missing)"}
    try:
        out, err = proc.communicate(timeout=timeout)
        line = [ln for ln in out.splitlines() if ln.startswith("{")]
        if proc.returncode == 0 and line:
            return json.loads(line[-1])
        return {"unavailable": (err.strip().splitlines() or ["no output"])[-1][:200]}
    except Exception as exc:
        proc.kill()
        return {"unavailable": repr(exc)[:200]}


# --------------------------------------------------------------------------- reference arm
def workload_name(env_id, log2_envs, world):
    """The workload both arms (this engine, --impl reference) name in config.workload: same string, same batch."""
    return (f"{env_id} num_envs=2^{log2_envs} per GPU x {world} GPU(s) = {(1 << log2_envs) * world} envs, random actions, "
            "step + TimeLimit + same-step autoreset, one vector step per timed step")


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores.

    openai/gym is pure Python: 2^20 SyncVectorEnv sub-environments would need ~7 s per vector step and several GB, so
    the arm that runs the FULL workload is the oracle port (oracle/gym_oracle.c: the reference's step / reset /
    TimeLimit / autoreset restated in C, bit-exact against the reference, one pthread per host core); the real
    reference (oracle/_ref) is timed beside it on the batch sizes it can hold (`cpu_baseline_python`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(1, args.gpus)
    n = (1 << args.log2_envs) * world          # the same global batch the B200 arm steps at this N
    threads = host_threads()
    py = start_python_reference(args.env)
    py_ref = collect_python_reference(py)      # before the threaded port runs: no contention
    rng = np.random.default_rng(0)
    v = make_oracle(args.env, n)
    v.reset(seed=0)
    pool = [random_actions_np(args.env, n, rng) for _ in range(4)]
    for w in range(max(args.warmup, 1)):
        v.step(pool[w % 4], nthreads=threads)
    done = args.steps
    t0 = time.perf_counter()
    for k in range(done):
        v.step(pool[k % 4], nthreads=threads)
    el = time.perf_counter() - t0
    v.close()
    value = n * done / el
    line = {
        "impl": "reference", "metric": "env-steps/sec", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": done, "warmup": args.warmup, "ms_per_step": 1e3 * el / done,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if is_box2d(args.env) else "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.env, args.log2_envs, world),
                   "arm": "the reference path on the host cores: C port of step / reset / TimeLimit / autoreset "
                          f"(oracle/, bit-exact against openai/gym 0.26.2), {threads} threads; the unmodified Python "
                          "reference is timed beside it in cpu_baseline_python"},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port",
                         "sample": f"{done} vector steps of {n} envs"},
        "cpu_baseline_python": py_ref,
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- B200 arm
def device_actions(torch, inner, n, dev, gen, count=16):
    if inner.discrete:
        return torch.randint(0, inner.single_action_space.n, (count, n), device=dev, dtype=torch.int64, generator=gen)
    scale = 2.0 if inner.act_dim == 1 else 1.0
    return (torch.rand((count, n, inner.act_dim), device=dev, generator=gen) * 2.0 - 1.0) * scale


class L2Flush:
    """write 256 MiB (> 126 MB L2), then stream-read another 256 MiB so that the lines left in L2 are CLEAN
    (otherwise the timed kernel pays the write-back of the flush's own dirty lines)."""

    def __init__(self, torch, dev):
        self.torch = torch
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        self.rd = torch.zeros(32 << 20, dtype=torch.int64, device=dev)
        self.sink = torch.zeros(1, dtype=torch.int64, device=dev)

    def __call__(self, k):
        self.buf.fill_(k & 0xFF)
        self.torch.sum(self.rd, dim=0, keepdim=True, out=self.sink)


def time_steps_flushed(torch, env, pool, K, flush):
    """K steps, L2 flushed before each, one CUDA-event pair per step -> (per-step milliseconds, what the last step
    returned)."""
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    torch.cuda.synchronize()
    for k in range(K):
        flush(k)
        starts[k].record()
        last = env.step(pool[k % len(pool)])
        ends[k].record()
    torch.cuda.synchronize()
    return np.array([s.elapsed_time(e) for s, e in zip(starts, ends)], dtype=np.float64), last


def dump_outputs(directory, step_result):
    """Write one step's (obs, reward, terminated, truncated, infos) as float32 / float64 .npy files in `directory`,
    at most DUMP_LIMIT_BYTES in all (a seeded sample of env rows beyond that)."""
    obs, rew, term, trunc, infos = step_result
    done = (term | trunc).cpu().numpy()
    final = infos["final_observation"].cpu().numpy().astype(np.float32)
    final[~done] = 0.0   # only the finished envs' rows are defined
    arrays = {"obs": obs.cpu().numpy().astype(np.float32), "reward": rew.cpu().numpy().astype(np.float64),
              "terminated": term.cpu().numpy().astype(np.float32), "truncated": trunc.cpu().numpy().astype(np.float32),
              "final_observation": final}
    n = len(done)
    row_bytes = sum(a.nbytes for a in arrays.values()) // n
    budget = DUMP_LIMIT_BYTES - 4096   # room for the .npy headers
    if row_bytes * n > budget:
        keep = budget // (row_bytes + 8)   # 8: the float64 row index written beside them
        rows = np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a))


def extra_config_line(torch, gym_b200, env_id, log2n, steps, dev, flush, peak):
    """One short single-GPU measurement of another BASELINE config (same timing rules as the headline)."""
    n = 1 << log2n
    env = gym_b200.vector.make(env_id, n)
    env.reset(seed=0)
    gen = torch.Generator(device=dev).manual_seed(99)
    pool = device_actions(torch, env, n, dev, gen, count=8)
    warm = 250 if is_box2d(env_id) else 20   # Box2D: reach the steady state of random play (contacts, resets)
    for w in range(warm):
        env.step(pool[w % 8])
    ms, _ = time_steps_flushed(torch, env, pool, steps, flush)
    env.close()
    med = float(np.median(ms))
    bpe = BYTES_PER_ENV_STEP.get(env_id, 0)
    gbs = bpe * n / (med * 1e-3) / 1e9
    return {"workload": f"{env_id} num_envs=2^{log2n}, random actions resident in HBM, fused step+TimeLimit+autoreset",
            "value": n / (med * 1e-3), "unit": "env-steps/s", "ms_per_step": med, "ms_per_step_mean": float(ms.mean()),
            "steps": steps, "warmup": warm, "bound": BOUND.get(env_id), "bytes_per_env_step": bpe,
            "hbm_gbs": gbs, "hbm_frac": gbs / peak}


def uint8_actions_line(torch, gym_b200, log2n, steps, dev, flush, peak, e2e_steps):
    """CartPole-v1 with uint8 actions, an ADDITIONAL line (the int64 line stays the headline: int64 is what
    `Discrete.sample()` and the reference's batch_space produce): 7 bytes less per env-step for the kernel to read and
    7/8 of the host->device traffic gone from the end-to-end path."""
    n = 1 << log2n
    env = gym_b200.vector.make(ENV_ID, n)
    env.reset(seed=0)
    gen = torch.Generator(device=dev).manual_seed(7)
    pool = [torch.randint(0, 2, (n,), device=dev, dtype=torch.uint8, generator=gen) for _ in range(8)]
    for w in range(20):
        env.step(pool[w % 8])
    ms, _ = time_steps_flushed(torch, env, pool, steps, flush)
    env.close()
    med = float(np.median(ms))
    bpe = BYTES_PER_ENV_STEP[ENV_ID] - 7
    line = {"workload": f"{ENV_ID} num_envs=2^{log2n}, random uint8 actions resident in HBM, fused step+TimeLimit+autoreset",
            "value": n / (med * 1e-3), "unit": "env-steps/s", "ms_per_step": med, "steps": steps, "bound": "hbm",
            "bytes_per_env_step": bpe, "hbm_gbs": bpe * n / (med * 1e-3) / 1e9, "hbm_frac": bpe * n / (med * 1e-3) / 1e9 / peak}
    host_env = gym_b200.vector.make(ENV_ID, n, backend="numpy", copy=False, dense_infos=True)
    host_env.reset(seed=0)
    hnp = [t.cpu().pin_memory().numpy() for t in pool[:4]]
    for k in range(5):
        host_env.step(hnp[k % 4])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        host_env.step(hnp[k % 4])
    torch.cuda.synchronize()
    el = time.perf_counter() - t0
    host_env.close()
    line["e2e"] = {"value": n * e2e_steps / el, "unit": "env-steps/s", "ms_per_step": 1e3 * el / e2e_steps,
                   "h2d_bytes_per_step": n, "steps": e2e_steps}
    return line


def run_b200(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # the real reference's vector envs are timed in their own process, started before CUDA exists here
    py_proc = start_python_reference(args.env) if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None
    py_ref = collect_python_reference(py_proc) if py_proc is not None else None

    import torch
    import torch.distributed as dist

    import gym_b200
    from gym_b200.distributed import ShardedVectorEnv

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", torch.cuda.current_device())
    n = 1 << args.log2_envs
    K, W = args.steps, max(args.warmup, 3)
    peak, peak_src = measured_hbm_peak()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    gather = args.gather

    def make_sharded(total):
        nonlocal gather
        try:
            return ShardedVectorEnv(args.env, total, gather=gather)
        except Exception as exc:  # e.g. CUDA IPC unavailable: fall back to the NCCL exchange
            if rank == 0:
                print(f"[bench] gather={gather} unavailable ({exc}); using nccl", file=sys.stderr)
            gather = "nccl"
            return ShardedVectorEnv(args.env, total, gather=gather)

    if world > 1:
        env = make_sharded(n * world)
        inner = env.env
    else:
        env = gym_b200.vector.make(args.env, n)
        inner = env
    env.reset(seed=0)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    pool = device_actions(torch, inner, n, dev, gen)
    flush = L2Flush(torch, dev) if world == 1 else None

    for w in range(W):
        env.step(pool[w % 16])
    barrier()

    sampler = ClockSampler(torch.cuda.current_device() if world == 1 else local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    gather_verified = None
    # kernels of this repo launched per timed step: classic control 1; the Box2D tasks 3 (step kernel, TOI kernel over
    # the parked envs, compacted reset kernel -- DESIGN.md 4.4)
    launches_per_step = 3 if is_box2d(args.env) else 1
    if world == 1:
        per_step, last = time_steps_flushed(torch, env, pool, K, flush)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last)
        ms_median, ms_mean = float(np.median(per_step)), float(per_step.mean())
        ms_per_step = ms_median
        kernel_ms = ms_median
        # the same K steps back to back with a warm L2 (reported, not the headline)
        barrier()
        s0, e0 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for k in range(K):
            env.step(pool[k % 16])
        e0.record()
        barrier()
        warm_ms = s0.elapsed_time(e0) / K
        l2_note = ("flushed before every timed step (256 MiB write, then 256 MiB read so L2 holds clean lines); "
                   "one CUDA-event pair per step on the launch stream; ms_per_step = median of the K steps")
        extra_timing = {"ms_per_step_mean": ms_mean, "ms_per_step_p10": float(np.percentile(per_step, 10)),
                        "ms_per_step_p90": float(np.percentile(per_step, 90))}
    else:
        # the gathered outputs (world x 26 MB) exceed L2; K steps back to back incl. the all-gather,
        # bracketed by barrier + synchronize, max over ranks
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        s0, e0 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for k in range(K):
            starts[k].record()
            env.step(pool[k % 16])
        e0.record()
        barrier()
        total_ms = max_over_ranks(s0.elapsed_time(e0))
        ms_per_step = total_ms / K
        gaps = [starts[k].elapsed_time(starts[k + 1]) for k in range(K - 1)] or [ms_per_step]
        extra_timing = {"ms_per_step_median": max_over_ranks(float(np.median(gaps)))}
        # fused exchange: kernel G alone when the shard is whole 256-env tiles (the step barrier runs in its tail),
        # else kernel G + kernel A for the ragged tail + p2p_sync_kernel; NCCL: the step kernel + 4 all-gathers
        fused_barrier = n % 256 == 0 and os.environ.get("B200GYM_P2P_FUSE_BARRIER", "0") == "1"
        launches_per_step = (1 if fused_barrier else 2) if gather == "p2p" else 5
        # ---- verify the gather: per peer, checksum of ITS rows in MY copy == the checksum it computed itself
        acts = pool[3]
        obs, rew, term, trunc, _ = env.step(acts)

        def sums(lo, hi):
            return torch.stack([obs[lo:hi].contiguous().view(torch.int32).to(torch.int64).sum(),
                                rew[lo:hi].contiguous().view(torch.int64).sum(),
                                term[lo:hi].to(torch.int64).sum(), trunc[lo:hi].to(torch.int64).sum()])

        mine = sums(rank * n, (rank + 1) * n)
        theirs = torch.empty((world, 4), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(theirs, mine.view(1, 4))
        seen = torch.stack([sums(r * n, (r + 1) * n) for r in range(world)])
        ok = torch.tensor([int(torch.equal(seen, theirs) and bool((rew != 0).any()))], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        gather_verified = bool(ok.item())
        # kernel-only time of this rank's shard (no exchange), for the roofline entry
        inner_s = [torch.cuda.Event(enable_timing=True) for _ in range(32)]
        inner_e = [torch.cuda.Event(enable_timing=True) for _ in range(32)]
        for k in range(32):
            inner_s[k].record()
            inner.step(pool[k % 16])
            inner_e[k].record()
        barrier()
        kernel_ms = float(np.median([s.elapsed_time(e) for s, e in zip(inner_s, inner_e)]))
        warm_ms = None
        l2_note = (f"per-step working set (gathered outputs, {world} x 26 MiB) exceeds L2; K steps back to back "
                   "between barrier+synchronize, max over ranks")
    clocks = sampler.stop() if rank == 0 else None
    value = world * n / (ms_per_step * 1e-3)

    # ---- BASELINE configs[4]: 2^23 envs in total over the N GPUs (strong scaling), exchange included
    strong = None
    if not args.no_extra and args.env.startswith("CartPole"):
        total = 1 << args.log2_total_strong
        ns = total // world
        env.close()
        env = None
        senv = make_sharded(total) if world > 1 else gym_b200.vector.make(args.env, total)
        sinner = senv.env if world > 1 else senv
        senv.reset(seed=0)
        spool = device_actions(torch, sinner, ns, dev, gen, count=4)
        for w in range(5):
            senv.step(spool[w % 4])
        SK = 40
        barrier()
        s0, e0 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for k in range(SK):
            senv.step(spool[k % 4])
        e0.record()
        barrier()
        sms = max_over_ranks(s0.elapsed_time(e0)) / SK
        strong = {"total_envs": total, "envs_per_gpu": ns, "steps": SK, "ms_per_step": sms,
                  "value": total / (sms * 1e-3), "unit": "env-steps/s", "scaling": "strong",
                  "note": "BASELINE.json configs[4]: CartPole-v1, 2^23 envs split over the GPUs, per-step all-gather "
                          "fused into the step kernel (N=1: no exchange); steps back to back, max over ranks"}
        senv.close()

    # ---- e2e: pinned host actions in, results to host, through the public API
    e2e = None
    if not args.no_e2e:
        hpool = [pool[k].cpu().pin_memory() for k in range(4)]
        E = max(10, min(args.e2e_steps, K))
        D = inner.obs_dim
        h2d = n * (8 if inner.discrete else 4 * inner.act_dim)
        if world == 1:
            host_env = gym_b200.vector.make(args.env, n, backend="numpy", copy=False, dense_infos=True)
            host_env.reset(seed=0)
            hnp = [t.numpy() for t in hpool]
            for k in range(5):
                host_env.step(hnp[k % 4])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for k in range(E):
                obs, rew, term, trunc, infos = host_env.step(hnp[k % 4])
            torch.cuda.synchronize()
            el = time.perf_counter() - t0
            n_done = int(infos["_final_observation"].sum())
            d2h = n * (4 * D + 8 + 1 + 1) + n_done * (4 + 4 * D) + 64
            api = ("B200VectorEnv(backend='numpy').step(pinned numpy actions) -> numpy obs / rewards / terminateds / "
                   "truncateds / final_observation (b200gym_step_host)")
            host_env.close()
        else:
            # N>1: the sharded env WITH the exchange: pinned host actions of this rank's shard -> H2D -> fused
            # step + all-gather -> D2H of this rank's rows of the gathered results
            if env is None:
                env = make_sharded(n * world)
                env.reset(seed=0)
            lo, hi = rank * n, (rank + 1) * n
            host_out = [torch.empty((n, D), dtype=torch.float32).pin_memory(), torch.empty(n, dtype=torch.float64).pin_memory(),
                        torch.empty(n, dtype=torch.bool).pin_memory(), torch.empty(n, dtype=torch.bool).pin_memory()]

            def host_step(k):
                a = hpool[k % 4].to(dev, non_blocking=True)
                res = env.step(a)
                for dst, src in zip(host_out, res[:4]):
                    dst.copy_(src[lo:hi], non_blocking=True)
                torch.cuda.current_stream().synchronize()

            for k in range(5):
                host_step(k)
            barrier()
            t0 = time.perf_counter()
            for k in range(E):
                host_step(k)
            el = time.perf_counter() - t0
            d2h = n * (4 * D + 8 + 1 + 1)
            api = ("ShardedVectorEnv.step(pinned host actions of the shard): H2D, fused step + all-gather over NVLink, "
                   "D2H of this rank's rows of the gathered results")
        el = max_over_ranks(el)
        e2e = {"value": world * n * E / el, "unit": "env-steps/s", "h2d_bytes_per_step": h2d * world,
               "d2h_bytes_per_step": d2h * world, "steps": E, "ms_per_step": 1e3 * el / E, "api": api,
               "exchange_included": world > 1}
    if env is not None:
        env.close()

    # ---- the other BASELINE configs (N == 1 only): short lines, same timing rules
    configs = None
    if world == 1 and not args.no_extra and args.env == ENV_ID:
        configs = {}
        for env_id, log2n, steps in EXTRA_CONFIGS:
            try:
                configs[env_id] = extra_config_line(torch, gym_b200, env_id, log2n, steps, dev, flush, peak)
            except Exception as exc:  # a failing side measurement must not lose the headline
                configs[env_id] = {"error": repr(exc)[:200]}
        try:
            configs["CartPole-v1 (uint8 actions)"] = uint8_actions_line(torch, gym_b200, args.log2_envs, 200, dev, flush, peak,
                                                                        max(10, min(args.e2e_steps, 100)))
        except Exception as exc:
            configs["CartPole-v1 (uint8 actions)"] = {"error": repr(exc)[:200]}

    # ---- cpu baseline (rank 0, N == 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        v, cpu_steps, cpu_el = cpu_oracle_throughput(args.env, n, args.cpu_seconds, threads)
        cpu = {"value": v, "unit": "env-steps/s", "cores": threads, "kind": "port",
               "sample": f"{cpu_steps} vector steps of 2^{args.log2_envs} envs ({cpu_el:.1f} s) of the same workload, "
                         + ("oracle/lunar_oracle.c / walker_oracle.c" if is_box2d(args.env) else "oracle/gym_oracle.c")
                         + " with one pthread per host core"}

    if rank == 0:
        bpe = BYTES_PER_ENV_STEP.get(args.env, 0)
        achieved = bpe * n / (kernel_ms * 1e-3) / 1e9
        kernel_name = {"a": "step_kernel", "p": "step_kernel_persistent", "l": "step_kernel_persistent<LEAN>"}[
            os.environ.get("B200GYM_KERNEL", "l")[:1]]
        if is_box2d(args.env):
            kernel_name = "lunar_step_kernel" if args.env.startswith("Lunar") else "walker_step_kernel"
        line = {
            "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if is_box2d(args.env) else "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.env, args.log2_envs, world),
                       "arm": f"{'int64' if inner.discrete else 'float32'} actions resident in HBM, fused "
                              "step+TimeLimit+autoreset kernel"
                              + ((", all-gather of (obs,reward,terminated,truncated) per step fused into the "
                                  "step kernel (bulk pushes over NVLink peer memory + one flag exchange)"
                                  if gather == "p2p" else
                                  ", NCCL all-gather of (obs,reward,terminated,truncated) per step")
                                 if world > 1 else ""),
                       "state": "float64 (reference-faithful)", "l2": l2_note,
                       "parallelism": f"env-batch data parallel x{world}"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak,
                         "traffic": (NCU_DRAM["read"] + NCU_DRAM["write"]) if (args.env == ENV_ID and args.log2_envs == 20) else None,
                         "traffic_note": f"{NCU_DRAM['file']}: dram__bytes_read.sum {NCU_DRAM['read']:.3g} + "
                                         f"dram__bytes_write.sum {NCU_DRAM['write']:.3g} of one launch; the reads exceed "
                                         "the algorithmic 46 MB by RNG records + sector slack, the writes UNDER-count: "
                                         "part of the 65 MB written is still dirty in the 126 MB L2 when the kernel ends",
                         "peak_source": peak_src, "bytes_per_env_step": bpe, "kernel_ms": kernel_ms,
                         "bound_note": BOUND.get(args.env),
                         "kernel": kernel_name + ("<CARTPOLE, int64>" if args.env.startswith("CartPole") else "")
                         + ("" if world == 1 else " (this rank's shard re-timed without the exchange)")},
            "cpu_baseline": cpu,
            "cpu_baseline_python": py_ref,
            "e2e": e2e,
            "gpu_launches": K * launches_per_step,
            "clocks": clocks,
        }
        line.update(extra_timing)
        if world > 1:
            line["gather"] = gather
            line["gather_verified"] = gather_verified
        if strong is not None:
            line["strong_scaling"] = strong
        if configs is not None:
            line["configs"] = configs
        if warm_ms is not None:
            line["warm_l2"] = {"ms_per_step": warm_ms, "value": n * 1e3 / warm_ms,
                               "note": "same K steps back to back, state resident in L2 (not the headline)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
