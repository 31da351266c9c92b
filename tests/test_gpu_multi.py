"""Multi-GPU path on real GPUs (needs >= 2 GPUs: `gpurun --gpus 2 -- pytest -m gpu tests/test_gpu_multi.py`).

Rank r owns the global envs [r*n, (r+1)*n); both exchange flavours -- the fused NVLink
peer-store kernel ("p2p") and the NCCL all-gather ("nccl") -- must deliver, on every rank, exactly
the tensors a single GPU computes for the whole batch.
"""
import os
import socket

import pytest

pytestmark = pytest.mark.gpu


def _ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, env_id, n_local, steps, q):
    import numpy as np
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import gym_b200
        from gym_b200.distributed import ShardedVectorEnv
        total = world * n_local
        rng = np.random.default_rng(0)
        full = gym_b200.vector.make(env_id, total, max_episode_steps=25)      # single-GPU reference
        if full.discrete:
            acts = torch.as_tensor(rng.integers(0, full.single_action_space.n, size=(steps, total)), device="cuda")
        else:
            acts = torch.as_tensor(rng.uniform(-2, 2, size=(steps, total, 1)).astype(np.float32), device="cuda")
        envs = {g: ShardedVectorEnv(env_id, total, gather=g, max_episode_steps=25) for g in ("p2p", "nccl")}
        ref_obs, _ = full.reset(seed=77)
        for g, e in envs.items():
            o, _ = e.reset(seed=77)
            assert torch.equal(o, ref_obs), f"{g}: reset obs differ from the single-GPU batch"
        lo, hi = rank * n_local, (rank + 1) * n_local
        n_done = 0
        for t in range(steps):
            ro, rr, rte, rtr, rinfo = full.step(acts[t])
            for g, e in envs.items():
                o, r, te, tr, info = e.step(acts[t, lo:hi])
                torch.cuda.synchronize()
                assert torch.equal(o, ro), f"{g} step {t}: obs"
                assert torch.equal(r, rr) and torch.equal(te, rte) and torch.equal(tr, rtr), f"{g} step {t}"
                m = info["_final_observation"]
                assert torch.equal(m, rinfo["_final_observation"][lo:hi])
                assert torch.equal(info["final_observation"][m], rinfo["final_observation"][lo:hi][m])
            n_done += int((rte | rtr).sum())
        assert n_done > 0
        for e in envs.values():
            e.close()
        full.close()
        q.put((rank, "ok"))
    except Exception as e:  # pragma: no cover
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def _wrapper_worker(rank, world, port, q):
    """NormalizeObservation / NormalizeReward over one rank's SHARD, batch moments all-reduced across the GPUs,
    must normalise exactly like the same wrappers over the whole batch on one GPU; and the stateless wrapper
    kernels must run on the device their buffers live on even when another device is current."""
    import numpy as np
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import gym_b200
        from gym_b200.wrappers import NormalizeObservation, NormalizeReward, RecordEpisodeStatistics
        n, T = 3000, 40
        total = world * n
        lo, hi = rank * n, (rank + 1) * n
        full = NormalizeReward(NormalizeObservation(gym_b200.vector.make("Pendulum-v1", total, max_episode_steps=13)), gamma=0.9)
        shard = NormalizeReward(NormalizeObservation(
            gym_b200.vector.make("Pendulum-v1", n, max_episode_steps=13, first_index=lo), group=True), gamma=0.9, group=True)
        fo, _ = full.reset(seed=5)
        so, _ = shard.reset(seed=5)
        torch.testing.assert_close(so, fo[lo:hi], rtol=1e-6, atol=1e-6)
        rng = np.random.default_rng(0)
        for t in range(T):
            a = torch.as_tensor(rng.uniform(-2, 2, size=(total, 1)).astype(np.float32), device="cuda")
            fo, fr, fte, ftr, _ = full.step(a)
            so, sr, ste, strn, _ = shard.step(a[lo:hi])
            torch.testing.assert_close(so, fo[lo:hi], rtol=1e-6, atol=1e-6)
            torch.testing.assert_close(sr, fr[lo:hi], rtol=1e-10, atol=1e-12)
            assert torch.equal(ste, fte[lo:hi]) and torch.equal(strn, ftr[lo:hi])
        torch.testing.assert_close(shard.env.obs_rms.mean, full.env.obs_rms.mean, rtol=1e-10, atol=1e-12)
        torch.testing.assert_close(shard.env.obs_rms.var, full.env.obs_rms.var, rtol=1e-10, atol=1e-12)
        assert abs(float(shard.env.obs_rms.count.item()) - float(full.env.obs_rms.count.item())) < 1e-6
        full.close()
        shard.close()
        # an env on ANOTHER device than the current one: every wrapper kernel must follow its buffers
        other = (rank + 1) % world
        env = RecordEpisodeStatistics(NormalizeObservation(gym_b200.vector.make("CartPole-v1", 2000, device=other)))
        twin = RecordEpisodeStatistics(NormalizeObservation(gym_b200.vector.make("CartPole-v1", 2000)))
        assert torch.cuda.current_device() == rank and env.unwrapped.device.index == other
        eo, _ = env.reset(seed=9)
        to, _ = twin.reset(seed=9)
        assert eo.device.index == other and torch.equal(eo.cpu(), to.cpu())
        for t in range(30):
            a = torch.as_tensor(rng.integers(0, 2, size=2000))
            eo, er, ete, etr, ei = env.step(a.to(f"cuda:{other}"))
            to, tr_, tte, ttr, ti = twin.step(a.cuda())
            assert torch.equal(eo.cpu(), to.cpu()) and torch.equal(ete.cpu(), tte.cpu())
            assert torch.equal(ei["episode"]["r"].cpu(), ti["episode"]["r"].cpu())
        env.close()
        twin.close()
        q.put((rank, "ok"))
    except Exception:  # pragma: no cover
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(_ngpus() < 2, reason="needs at least 2 GPUs")
@pytest.mark.timeout(300)
def test_wrappers_across_gpus():
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_wrapper_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=240) for _ in range(world))
    for p in procs:
        p.join(timeout=30)
    assert all(v == "ok" for v in results.values()), results


@pytest.mark.skipif(_ngpus() < 2, reason="needs at least 2 GPUs")
# 148*256+640: full tiles through kernel G + a ragged tail through kernel A; 5000: ragged; 300*256 / 64*256: whole tiles
# only, all through kernel G.  Every case ends the step with the p2p_sync_kernel barrier
@pytest.mark.parametrize("env_id,n_local", [("CartPole-v1", 148 * 256 + 640), ("Pendulum-v1", 5000), ("CartPole-v1", 300 * 256),
                                            ("Acrobot-v1", 64 * 256)])
@pytest.mark.timeout(300)
def test_sharded_step_matches_single_gpu(env_id, n_local):
    import torch.multiprocessing as mp
    world = min(_ngpus(), 8)   # every GPU of the box (the driver's scaling run uses 8)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, env_id, n_local, 40, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=280) for _ in range(world))
    for p in procs:
        p.join(timeout=30)
    assert all(v == "ok" for v in results.values()), results
