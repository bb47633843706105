"""Episode statistics accumulated inside the step kernels, and their sum over ranks (the only collective of the path).

Single GPU: the kernel-side totals equal a host-side accumulation from the reward / done tensors of the same rollout,
for the fused chain kernel, the single-launch trajectory kernel and the Panda task. Two GPUs (skipped on a machine with
fewer): two NCCL ranks, each stepping its shard of the env indices, all-reduce the 4 totals and
get the numbers of the unsharded run.
"""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch


def _host_totals(torch, rewards, dones):
    """Reference accumulation from [T, N] reward / done tensors (float64 on the device, exact summation order aside)."""
    from b2sim.distributed import EpisodeStats
    ref = EpisodeStats(rewards.shape[1], rewards.device)
    for t in range(rewards.shape[0]):
        ref.update(rewards[t], dones[t])
    return ref.totals.cpu().numpy()


@pytest.mark.parametrize("env_id,amp,limit", [("CartPoleContinuousSwingup-Gazebo-v0", 200.0, 37),
                                              ("Pendulum-Gazebo-v0", 50.0, 50)])
def test_kernel_side_statistics_match_host_accumulation(env_id, amp, limit, torch):
    import b2sim
    n, T = 5000, 200   # not a multiple of the block size: the last warp of the grid is partial
    env = b2sim.BatchedTaskEnv(env_id, n, seed=4, max_episode_steps=limit)
    env.enable_episode_stats()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2)
    acts = (torch.rand(T, n, device="cuda", generator=gen, dtype=torch.float64) * 2 - 1) * amp
    rew = torch.empty(T, n, dtype=torch.float64, device="cuda")
    done = torch.empty(T, n, dtype=torch.uint8, device="cuda")
    for t in range(T):
        _, r, d = env.step(acts[t])
        rew[t].copy_(r); done[t].copy_(d)
    got = np.array(env.episode_stats())
    want = _host_totals(torch, rew, done)
    assert want[2] >= n * (T // limit), "every env must have finished episodes"
    assert got[2] == want[2] and got[1] == want[1] and got[3] == want[3] == 0     # counts are exact
    assert got[0] == pytest.approx(want[0], rel=1e-12)                            # sums differ by summation order only
    # running returns of the unfinished episodes are per-env state of the kernels too
    from b2sim import _lib
    running = env.sim.tensor(env.model, _lib.BUF_EP_RETURN)
    open_len = env.elapsed.long()
    assert running.shape == (n,) and bool((running[open_len == 0] == 0).all())
    # a trajectory launch continues the same accumulators
    env.trajectory(acts[:64].contiguous(), record=False)
    o, r2, d2 = env.trajectory(acts[64:128].contiguous())
    got2 = np.array(env.episode_stats(clear=True))
    assert got2[2] > got[2] and got2[1] > got[1]
    assert env.episode_stats() == [0.0, 0.0, 0.0, 0.0]
    # non-finite rewards are counted, not summed
    env.close()


def test_panda_task_statistics(torch):
    import b2sim
    n, T, limit = 1000, 90, 40
    env = b2sim.BatchedTaskEnv("PandaReach-Gazebo-v0", n, seed=0, max_episode_steps=limit)
    env.enable_episode_stats()
    q0 = torch.tensor(b2sim.batched.PANDA_Q0, device="cuda", dtype=torch.float64)
    tg = (q0 + 0.05).repeat(n, 1).contiguous()
    tg[:, 7:] = 0.02
    rew = torch.empty(T, n, dtype=torch.float64, device="cuda")
    done = torch.empty(T, n, dtype=torch.uint8, device="cuda")
    for t in range(T):
        _, r, d = env.step(tg)
        rew[t].copy_(r); done[t].copy_(d)
    got = np.array(env.episode_stats())
    want = _host_totals(torch, rew, done)
    assert got[2] == want[2] == 2 * n and got[1] == want[1] == 2 * n * limit
    assert got[0] == pytest.approx(want[0], rel=1e-12)
    env.close()


_WORKER = r"""
import os, sys, json
sys.path.insert(0, {root!r})
import __graft_entry__; __graft_entry__.load_package()
import torch, torch.distributed as dist
import b2sim
from b2sim.distributed import EpisodeStats, shard_range
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
n_global, T, limit = 6000, 150, 41
start, stop = shard_range(n_global, rank, world)
env = b2sim.BatchedTaskEnv("CartPoleContinuousSwingup-Gazebo-v0", stop - start, device=rank, seed=8, env_offset=start,
                           max_episode_steps=limit)
stats = EpisodeStats.from_env(env)
gen = torch.Generator(device="cuda"); gen.manual_seed(3)
acts = ((torch.rand(T, n_global, device="cuda", generator=gen, dtype=torch.float64) * 2 - 1) * 200.0)[:, start:stop].contiguous()
for t in range(T):
    env.step(acts[t])
torch.cuda.synchronize()
t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
t0.record()
summary = stats.all_reduce()
t1.record(); torch.cuda.synchronize()
local = env.episode_stats()
if rank == 0:
    print("RESULT " + json.dumps(dict(summary=summary, local=local, allreduce_ms=t0.elapsed_time(t1))), flush=True)
dist.barrier()
dist.destroy_process_group()
"""


def test_two_rank_nccl_all_reduce_of_the_statistics(torch, tmp_path):
    """World size 2 over NCCL: the all-reduced totals equal those of one unsharded simulator (env-index keyed resets make
    the shards reproduce the unsharded rollout exactly, so the episode counts and lengths are identical)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import json
    import b2sim
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    procs = []
    for rank in range(2):
        envv = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1",
                    MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=envv, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                                      text=True))
    outs = [p.communicate(timeout=600)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)
    line = [l for l in outs[0].splitlines() if l.startswith("RESULT ")][0]
    res = json.loads(line[len("RESULT "):])
    # the unsharded run on one GPU
    n_global, T, limit = 6000, 150, 41
    env = b2sim.BatchedTaskEnv("CartPoleContinuousSwingup-Gazebo-v0", n_global, seed=8, max_episode_steps=limit)
    env.enable_episode_stats()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(3)
    acts = (torch.rand(T, n_global, device="cuda", generator=gen, dtype=torch.float64) * 2 - 1) * 200.0
    for t in range(T):
        env.step(acts[t])
    want = env.episode_stats()
    s = res["summary"]
    assert s["episodes"] == want[2] and s["episodes"] > n_global
    assert s["mean_length"] == pytest.approx(want[1] / want[2], rel=1e-15)
    assert s["mean_return"] == pytest.approx(want[0] / want[2], rel=1e-12)
    assert res["local"][2] < want[2]          # rank 0 alone saw only its shard
    env.close()
