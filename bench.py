#!/usr/bin/env python
"""Benchmark of the env.step hot path: batched env-steps/sec.

    python bench.py --gpus N --steps K --warmup W            # this engine (one process per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle restatement)

A "step" is one GazeboRuntime.step of every env: set_action -> one 1 kHz physics step -> observation, reward,
done -> masked auto-reset, in one kernel launch. Workload: CartPoleContinuousSwingup-Gazebo-v0 (BASELINE.json
configs[2], the config the metric's target is quoted on), envs sharded by index across ranks, no collective on
the step path. Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import __graft_entry__  # noqa: E402

METRIC = "batched env-steps/sec (Cartpole/Panda) at 1/2/4/8 B200 vs CPU Gazebo+DART"
ENV_ID = "CartPoleContinuousSwingup-Gazebo-v0"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int,
                    help="exact number of timed steps. Default 8192 for --impl b200: ~0.6 s of GPU load at the default "
                         "size, long enough for the 100 ms clock sampler (far fewer steps give few or no clock samples); "
                         "200 bounded samples for --impl reference")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=4 * 1048576,
                    help="envs per GPU; the default working set (~480 MB/step) exceeds the 126 MB L2")
    ap.add_argument("--dtype", default="float64", choices=["float64", "float32"])
    ap.add_argument("--env-id", default=ENV_ID)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target wall time of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the short measurements of the other BASELINE.json configurations (N=1 only)")
    ap.add_argument("--graph", action="store_true",
                    help="replay the steps from a CUDA graph of 4 launches (for launch-bound small batches); the "
                         "steps of a timed block beyond whole 64-step replays run as eager rollouts")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (obs, reward, done of a fixed, seeded sample of rank "
                         "0's envs, with their env_index) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 8192 if args.impl == "b200" else 200
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ---------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.samples, self._stop, self._thread = gpu_index, [], threading.Event(), None

    def _loop(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._thread = threading.Thread(target=self._loop, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=6)
        sm = sorted(int(float(s[1])) for s in self.samples if len(s) > 2 and s[1].replace(".", "").isdigit())
        mx = [int(float(s[2])) for s in self.samples if len(s) > 2 and s[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for k, name in enumerate(names):
                if len(s) > 5 + k and s[5 + k].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle restatement of the reference's path on the host cores
# ---------------------------------------------------------------------------------------------------------------
_W = {}


def _cpu_init(task, n, seed):
    """Worker initialiser: one process per core, each owning n envs of the oracle (persistent state)."""
    import multiprocessing as mp
    import numpy as np
    __graft_entry__.load_package()
    import gym_ignition_models
    from oracle import oracle as O
    ident = mp.current_process()._identity
    offset = (ident[0] if ident else 0) * n
    name = "pendulum" if task == O.TASK_PENDULUM_SWINGUP else "cartpole"
    _, model = O.load_urdf(gym_ignition_models.get_model_file(name))
    rng = np.random.default_rng(offset)
    _W.update(O=O, model=model, task=task, n=n, seed=seed, offset=offset, step=1,
              state=O.sample_reset_batch(task, seed, offset, n, 0), elapsed=np.zeros(n, np.int32),
              actions=rng.uniform(-200, 200, (64, n)))


def _cpu_step(T):
    """Advance this worker's envs by T env-steps; returns the seconds spent inside the oracle."""
    w = _W
    t0 = time.perf_counter()
    for k in range(T):
        a = w["actions"][(w["step"] + k) % 64][None, :]
        w["O"].rollout(w["model"], w["task"], a, w["state"], w["elapsed"], seed=w["seed"],
                       env_offset=w["offset"], first_step=w["step"] + k, record=False)
    w["step"] += T
    return time.perf_counter() - t0


class CpuPool:
    """The oracle restatement of the reference's path, one process per host core."""

    def __init__(self, task, n_per_core=4096, cores=None, seed=0):
        import multiprocessing as mp
        self.cores = cores or len(os.sched_getaffinity(0)) or 1
        self.n = n_per_core
        self.pool = mp.get_context("spawn").Pool(self.cores, initializer=_cpu_init, initargs=(task, n_per_core, seed))
        self.pool.map(_cpu_step, [1] * self.cores)  # make sure every worker is up

    def step(self, T=1):
        """One bounded sample: every core advances n envs by T steps. Returns (env_steps, wall seconds)."""
        t0 = time.perf_counter()
        self.pool.map(_cpu_step, [T] * self.cores, chunksize=1)
        return self.cores * self.n * T, time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_baseline(task, seconds):
    pool = CpuPool(task)
    steps, dt = pool.step(4)          # calibration
    T = max(4, int(4 * seconds / max(dt, 1e-3)))
    steps, dt = pool.step(T)
    pool.close()
    return {"value": steps / dt, "unit": "env-steps/s", "cores": pool.cores, "kind": "port",
            "sample": f"{pool.cores} processes x {pool.n} envs x {T} steps of {ENV_ID} (oracle/b2oracle.c, fp64), "
                      f"{dt:.1f} s wall"}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path. Ignition Gazebo + DART cannot be
    built in this image, so this times the oracle port (oracle/b2oracle.c) on all host cores. One step = a bounded
    sample of the workload: T env-steps of cores x 4096 envs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    pool = CpuPool(O.TASK_CARTPOLE_CONTINUOUS_SWINGUP)
    # One bench step = a bounded sample: every core advances its 4096 envs by T env-steps, T sized so that the whole
    # run takes about 90 s and the per-call process round trip does not weigh on the throughput.
    _, dt8 = pool.step(8)
    target = min(2.0, max(0.02, 90.0 / max(1, args.steps + args.warmup)))
    T = max(1, int(target / max(dt8 / 8, 1e-6)))
    for _ in range(args.warmup):
        pool.step(T)
    t0 = time.perf_counter()
    total = 0
    for _ in range(args.steps):
        total += pool.step(T)[0]
    wall = time.perf_counter() - t0
    pool.close()
    value = total / wall
    sample = f"{pool.cores} processes x {pool.n} envs x {T} env-steps per bench step (oracle/b2oracle.c, fp64)"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{ENV_ID}, {pool.cores * pool.n} envs, CPU restatement of the reference path "
                                   "(not Gazebo+DART, which cannot be built in this image)"},
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": pool.cores, "kind": "port",
                             "sample": sample},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
# the other BASELINE.json configurations, measured briefly next to the headline workload (N = 1 only)
# ---------------------------------------------------------------------------------------------------------------
def other_configs(local, peak):
    """Short CUDA-event measurements of BASELINE.json configs 1 (Pendulum, 65,536 envs), 3 (Panda position PID +
    KinDyn observation, 16,384 envs) and 4 (Panda pick scene with finger / cube / table contacts, 4,096 envs), fp64,
    one GPU. `frac` is the fraction of the HBM roofline at the algorithmic bytes per env-step of SURVEY.md 8(d); these
    small batches are launch- or latency-bound, the numbers say by how much."""
    import torch
    import b2sim

    def timed(fn, steps):
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            fn()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / steps

    def entry(workload, n, ms, nbytes, launches):
        value = n / (ms * 1e-3)
        return {"workload": workload, "envs": n, "value": value, "unit": "env-steps/s", "ms_per_step": ms,
                "launches_per_step": launches, "algorithmic_bytes_per_env_step": nbytes,
                "roofline_frac": value * nbytes / 1e9 / peak}

    out = {}
    gen = torch.Generator(device="cuda")
    gen.manual_seed(7)
    # config 1: Pendulum-Gazebo-v0, 65,536 envs
    n = 65536
    env = b2sim.BatchedTaskEnv("Pendulum-Gazebo-v0", n, device=local, seed=0)
    act4 = ((torch.rand(4, n, device="cuda", generator=gen, dtype=torch.float64) * 2 - 1) * 50.0).contiguous()
    for _ in range(10):
        env.rollout(act4)
    ms = timed(lambda: env.rollout(act4), 100) / 4
    out["pendulum_65536"] = entry("Pendulum-Gazebo-v0, 65536 envs, eager launches", n, ms, env.bytes_per_env_step, 1)
    # the same config as an open-loop rollout in ONE launch per 250 steps (k_task_trajectory: state stays in registers,
    # the full [T, N] trajectory of observations / rewards / dones is written): HBM-bound instead of launch-bound
    T = 250
    actT = ((torch.rand(T, n, device="cuda", generator=gen, dtype=torch.float64) * 2 - 1) * 50.0).contiguous()
    bufs = (torch.empty((T, n, env.nobs), dtype=torch.float64, device="cuda"),
            torch.empty((T, n), dtype=torch.float64, device="cuda"), torch.empty((T, n), dtype=torch.uint8, device="cuda"))
    for _ in range(3):
        env.trajectory(actT, out=bufs)
    ms = timed(lambda: env.trajectory(actT, out=bufs), 8) / T
    e = entry("Pendulum-Gazebo-v0, 65536 envs, open-loop rollout of 250 steps per launch, full trajectory written", n, ms,
              8 + 8 * env.nobs + 8 + 1, 1.0 / T)
    out["pendulum_65536_trajectory"] = e
    env.close()
    # the headline workload in the fp32 fast mode (reported separately, BASELINE.json north_star): 58 B per env-step
    n = 8 * 1048576
    env = b2sim.BatchedTaskEnv("CartPoleContinuousSwingup-Gazebo-v0", n, dtype="float32", device=local, seed=0)
    act4 = ((torch.rand(4, n, device="cuda", generator=gen, dtype=torch.float32) * 2 - 1) * 200.0).contiguous()
    for _ in range(5):
        env.rollout(act4)
    ms = timed(lambda: env.rollout(act4), 25) / 4
    out["cartpole_swingup_fp32_8388608"] = entry("CartPoleContinuousSwingup-Gazebo-v0, 8388608 envs, fp32 fast mode", n, ms,
                                                 env.bytes_per_env_step, 1)
    env.close()
    # config 3: Panda reach (position PID at the physics rate + end-effector pose / Jacobian observation), 16,384 envs
    n = 16384
    env = b2sim.BatchedTaskEnv("PandaReach-Gazebo-v0", n, device=local, seed=0)
    q0 = torch.tensor(b2sim.batched.PANDA_Q0, device="cuda", dtype=torch.float64)
    phase = torch.rand(n, 1, device="cuda", generator=gen, dtype=torch.float64) * 6.2831853
    tg = (q0 + 0.1 * torch.sin(phase)).contiguous()
    tg[:, 7:] = 0.02
    for _ in range(10):
        env.step(tg)
    ms = timed(lambda: env.step(tg), 100)
    out["panda_reach_16384"] = entry("PandaReach (Panda PID + ABA + KinDyn observation), 16384 envs, fingers held mid-range", n, ms,
                                     env.bytes_per_env_step, 1)
    # the same with the gripper closed against its lower joint limits (SURVEY 8d: "fingers 0"): two joint-limit rows per
    # env go through the lane-parallel constraint stage every step
    tg[:, 7:] = -0.01
    for _ in range(200):
        env.step(tg)
    ms = timed(lambda: env.step(tg), 100)
    out["panda_reach_16384_fingers_on_limits"] = entry("PandaReach, 16384 envs, both fingers pressed against their lower limits "
                                                       "(two joint-limit constraint rows per env and step)", n, ms,
                                                       env.bytes_per_env_step, 1)
    env.close()
    # the same config in the fp32 fast mode (reported separately, like the headline's)
    env = b2sim.BatchedTaskEnv("PandaReach-Gazebo-v0", n, dtype="float32", device=local, seed=0)
    tg32 = (q0 + 0.1 * torch.sin(phase)).to(torch.float32).contiguous()
    tg32[:, 7:] = 0.02
    for _ in range(10):
        env.step(tg32)
    ms = timed(lambda: env.step(tg32), 100)
    out["panda_reach_16384_fp32"] = entry("PandaReach, 16384 envs, fp32 fast mode", n, ms, env.bytes_per_env_step, 1)
    env.close()
    # config 4: pick scene, 4,096 envs: open gripper, then grasp (8 finger contact points + table contacts)
    n = 4096
    scene = b2sim.PandaPickScene(n, device=local)
    scene.step(50)
    ms_open = timed(scene.step, 50)
    scene.set_fingers(0.0)
    scene.step(300)
    ms_grasp = timed(scene.step, 100)
    z = scene.cube_state[:, 2].mean().item()
    e = entry("Panda pick scene (computed torque + finger / cube / table contacts), 4096 envs, grasp phase", n, ms_grasp,
              scene.bytes_per_env_step, 5)
    e["open_phase_ms_per_step"] = ms_open
    e["cube_height_mean"] = z
    out["panda_pick_4096"] = e
    scene.close()
    # config 0: CartPoleDiscreteBalancing-Gazebo-v0, ONE env through the unmodified gym.make / GazeboRuntime / Task
    # python over the drop-in scenario module (examples/python/launch_cartpole.py:32-75). Not a throughput workload: it
    # is the per-object API cost (ctypes calls, one small launch and a device->host read per env.step) the reference
    # pays in SWIG crossings and Gazebo's system loop.
    try:
        import functools
        import gym
        import gym_ignition_environments  # noqa: F401
        from gym_ignition_environments import randomizers
        make = functools.partial(lambda env_id, **kw: gym.make(env_id, **kw), env_id="CartPoleDiscreteBalancing-Gazebo-v0")
        genv = randomizers.cartpole_no_rand.CartpoleEnvNoRandomizations(env=make)
        genv.seed(0)
        genv.reset()
        count, t0 = 0, time.perf_counter()
        while count < 400:
            _, _, done, _ = genv.step(genv.action_space.sample())
            count += 1
            if done:
                genv.reset()
        dt = time.perf_counter() - t0
        genv.close()
        out["single_env_gym_api"] = {"workload": "CartPoleDiscreteBalancing-Gazebo-v0, 1 env, gym.make + GazeboRuntime + scenario "
                                                 "drop-in (per-object API, host wall clock incl. resets)",
                                     "envs": 1, "value": count / dt, "unit": "env-steps/s", "ms_per_step": 1e3 * dt / count}
    except Exception as exc:
        out["single_env_gym_api"] = {"error": repr(exc)}
    return out


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
def bind_near_gpu(local):
    """Pins this rank's CPU affinity (and with it the first-touch placement of the pinned host buffers it allocates
    afterwards) to the NUMA node its GPU hangs off. Returns a short description for the JSON line."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local)],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        bus = out[-12:] if len(out) >= 12 else out          # 00000000:17:00.0 -> 0000:17:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        if node < 0 or len(nodes) < 2:
            return {"numa_node": node, "numa_nodes": len(nodes), "bound": False}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "numa_nodes": len(nodes), "bound": bool(allowed), "cpus": len(allowed)}
    except Exception as exc:
        return {"bound": False, "error": repr(exc)[:80]}


def c3_strong(rank, world, local, peak, dist):
    """BASELINE.json configs[2] as written: 1,048,576 GLOBAL envs of CartPoleContinuousSwingup split by env index over the
    ranks (strong scaling: 131,072 envs per GPU at N = 8). One eager launch per step, and the same steps replayed from a
    CUDA graph of 64 launches (at 131,072 envs a launch moves 15 MB: HBM time 2.3 us against ~4 us of launch latency).
    Timed like the headline: barrier + synchronize on both sides, CUDA events, max over ranks, best of 5 blocks."""
    import torch
    import b2sim
    from b2sim.distributed import shard_range
    total = 1 << 20
    start, stop = shard_range(total, rank, world)
    n = stop - start
    env = b2sim.BatchedTaskEnv(ENV_ID, n, device=local, seed=0, env_offset=start)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(99 + rank)
    act4 = ((torch.rand(4, n, device="cuda", generator=gen, dtype=torch.float64) * 2 - 1) * 200.0).contiguous()

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, reps, steps_per_call):
        best = None
        for _ in range(5):
            sync()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(reps):
                fn()
            t1.record()
            sync()
            t = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item()) / (reps * steps_per_call)
            best = ms if best is None else min(best, ms)
        return best

    for _ in range(10):
        env.rollout(act4)
    eager_ms = timed(lambda: env.rollout(act4), 64, 4)
    side = torch.cuda.Stream()
    env.use_stream(side)
    graph = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            for _ in range(16):
                env.rollout(act4)
    torch.cuda.synchronize()
    for _ in range(3):
        graph.replay()
    graph_ms = timed(graph.replay, 8, 64)
    nbytes = env.bytes_per_env_step

    def entry(ms):
        return {"ms_per_step": ms, "value": total / (ms * 1e-3),
                "roofline_frac_per_gpu": n * nbytes / (ms * 1e-3) / 1e9 / peak}

    out = {"workload": "CartPoleContinuousSwingup-Gazebo-v0, 1048576 global envs split by env index (BASELINE configs[2] as "
                       "written)", "scaling": "strong", "global_envs": total, "envs_per_gpu": n, "unit": "env-steps/s",
           "algorithmic_bytes_per_env_step": nbytes, "hbm_us_per_step_at_peak": n * nbytes / peak / 1e3,
           "eager": entry(eager_ms), "cuda_graph_64_launches": entry(graph_ms),
           "note": "working set %.0f MB per GPU: %s the 126 MB L2" % (n * nbytes / 1e6, "inside" if n * nbytes < 126e6 else "beyond")}
    env.close()
    return out


def dump_outputs(env, directory, budget=48 << 20):
    """Writes what the last step returned to its caller (obs, reward, done) as directory/<name>.npy, for all envs or, where
    that exceeds `budget` bytes, for a fixed, seeded sample of them; env_index holds the env index of every row."""
    import numpy as np
    import torch
    n = env.num_envs
    rows = min(n, budget // (env.obs.element_size() * (env.nobs + 1) + 4 + 8))
    idx = np.arange(n) if rows == n else np.sort(np.random.default_rng(0).choice(n, rows, replace=False))
    sel = torch.as_tensor(idx, device=env.obs.device)
    out = {"obs": env.obs[sel].cpu().numpy(), "reward": env.reward[sel].cpu().numpy(),
           "done": env.done[sel].to(torch.float32).cpu().numpy(), "env_index": idx.astype(np.float64)}
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    __graft_entry__.load_package()
    import b2sim

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    torch.cuda.set_device(local)
    json_fd = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version (and any NCCL_DEBUG output) on stdout, which must carry exactly one JSON line: file
        # descriptor 1 points at stderr for the rest of the run and the line goes out through a saved copy
        sys.stdout.flush()
        json_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    n = args.envs_per_gpu
    tdt = torch.float64 if args.dtype == "float64" else torch.float32
    env = b2sim.BatchedTaskEnv(args.env_id, n, dtype=args.dtype, device=local, seed=0, env_offset=rank * n)
    amp = {"Pendulum-Gazebo-v0": 50.0, "CartPoleContinuousBalancing-Gazebo-v0": 50.0}.get(args.env_id, 200.0)
    # pre-generated action streams (the policy is outside the hot path); 4 buffers cycled
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1234 + rank)
    if args.env_id == "PandaReach-Gazebo-v0":
        # joint position targets around the initial configuration (cf. tests/test_scenario/test_pid_controllers.py:90-98),
        # fingers inside their range
        q0 = torch.tensor(b2sim.batched.PANDA_Q0, device="cuda", dtype=tdt)
        phase = torch.rand(n, 1, device="cuda", generator=gen, dtype=tdt) * 6.2831853
        acts = []
        for k in range(4):  # four consecutive samples of a 0.33 Hz sine with a per-env phase (SURVEY §8d, C4)
            wave = torch.sin(2 * 3.141592653589793 * 0.33 * k * 0.001 + phase)
            t = q0 + 0.1 * wave
            t[:, 7:] = 0.02 + 0.01 * wave
            acts.append(t.contiguous())
    elif args.env_id == "CartPoleDiscreteBalancing-Gazebo-v0":
        acts = [torch.randint(0, 2, (n,), device="cuda", generator=gen).to(tdt) for _ in range(4)]
    else:
        acts = [((torch.rand(n, device="cuda", generator=gen, dtype=tdt) * 2 - 1) * amp) for _ in range(4)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    act4 = torch.stack(acts)                      # [4, n]: one C call issues 4 consecutive step launches

    graph = None
    if args.graph:
        # the step index of the reset RNG lives in a device counter, so replays are exact
        side = torch.cuda.Stream()
        env.use_stream(side)
        graph = torch.cuda.CUDAGraph()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                for _ in range(16):
                    env.rollout(act4)
        torch.cuda.synchronize()

    def run_steps(count):
        if graph is not None:
            full, rest = divmod(count, 64)
            for _ in range(full):
                graph.replay()
            count = rest
        full, rest = divmod(count, 4)
        for _ in range(full):
            env.rollout(act4)
        for k in range(rest):
            env.step(acts[k])

    run_steps(args.warmup)
    barrier()
    # The timed region is EXACTLY args.steps steps, so that a run with the same arguments always ends in the same state.
    # It is split into up to 5 blocks of whole launch groups (4 steps per rollout call, 64 per graph replay), each
    # bracketed by barrier + synchronize and timed with CUDA events (max over ranks); the median block is reported.
    def timed_block(count):
        barrier()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        run_steps(count)
        stop.record()
        barrier()
        t = torch.tensor([start.elapsed_time(stop)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    unit = 64 if graph is not None else 4
    nblocks = max(1, min(5, args.steps // unit))
    size = args.steps // nblocks // unit * unit
    sizes = [size] * (nblocks - 1) + [args.steps - size * (nblocks - 1)]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = env.sim.launch_count()
    blocks = [timed_block(count) for count in sizes]
    launches = env.sim.launch_count() - l0
    if graph is not None:     # launches replayed from the CUDA graph are not seen by the host counter
        launches += sum(64 * (count // 64) for count in sizes)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(env, args.dump_outputs)
    per_step = sorted(ms / count for ms, count in zip(blocks, sizes))
    ms_per_step = per_step[len(per_step) // 2]    # the median block (max over ranks inside each block) is the reported one
    value = world * n / (ms_per_step * 1e-3)
    repeat_info = {"blocks": nblocks, "steps_per_block": sizes, "timed_steps": args.steps,
                   "reported": "median block, max over ranks", "best_ms_per_step": per_step[0],
                   "median_ms_per_step": ms_per_step, "worst_ms_per_step": per_step[-1], "loaded_ms": sum(blocks)}

    # dominant kernel: the step is exactly one launch of it, so its average launch duration is the CUDA-event
    # time per step of the reported block (the slowest rank's) over the launches per step
    kernel_avg_ms = ms_per_step * args.steps / max(1, launches)
    if args.env_id == "PandaReach-Gazebo-v0":
        kernel_name = "k_task_panda_lanes" if n <= 32768 else "k_task_panda"
    else:
        kernel_name = "k_task_chain"
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    algo_bytes = env.bytes_per_env_step * n
    achieved = algo_bytes / (kernel_avg_ms * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(
            f"{args.env_id}:{args.dtype}:{n}")
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": kernel_name, "kernel_ms": kernel_avg_ms,
                "algorithmic_bytes_per_env_step": env.bytes_per_env_step, "peak_source": peak_kind}

    # end to end through the C-ABI host-buffer call (pinned host memory, copies inside the timed region)
    es = 8 if args.dtype == "float64" else 4
    npdt = np.float64 if args.dtype == "float64" else np.float32
    # the pinned buffers are first touched by this rank: bind it to its GPU's NUMA node before allocating them
    binding = bind_near_gpu(local)
    h_act = torch.empty(acts[0].shape, dtype=tdt).pin_memory()
    h_obs = torch.empty((n, env.nobs), dtype=tdt).pin_memory()
    h_rew = torch.empty(n, dtype=tdt).pin_memory()
    h_done = torch.empty(n, dtype=torch.uint8).pin_memory()
    h_act.copy_(acts[0].cpu())
    a_np, o_np, r_np, d_np = h_act.numpy(), h_obs.numpy(), h_rew.numpy(), h_done.numpy()
    assert a_np.dtype == npdt
    for _ in range(3):
        env.step_host(a_np, o_np, r_np, d_np)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        env.step_host(a_np, o_np, r_np, d_np)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * n * args.e2e_steps / float(te.item())
    e2e = {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": n * env.nact * es,
           "d2h_bytes_per_step": n * (env.nobs * es + es + 1), "steps": args.e2e_steps,
           "api": "b2sim_task_step_host (C ABI, pinned host buffers)", "host_binding": binding,
           "pcie_gbs_per_gpu": n * (env.nact * es + env.nobs * es + es + 1) * args.e2e_steps / float(te.item()) / 1e9,
           "bound": ("PCIe link of the GPU (49 B per env-step; a plain pinned cudaMemcpyAsync reaches ~56 GB/s device to host)"
                     if world == 1 else
                     "host side: the GPUs of one box share the pinned-memory bandwidth of its host (8 GPUs copying at once: "
                     "121 GB/s device to host in total against 56 GB/s for one alone, profiles/r2_pcie_probe_n8.json)")}

    # the one collective of the path: episode statistics accumulated by the step kernels, summed over the ranks
    stats_info = None
    if not args.no_extra:
        from b2sim.distributed import EpisodeStats
        stats = EpisodeStats.from_env(env)
        for k in range(8):
            env.step(acts[k % 4])
        barrier()
        ts = []
        for _ in range(5):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            summary = stats.all_reduce()
            t1.record()
            torch.cuda.synchronize()
            ts.append(t0.elapsed_time(t1))
        # cost of the accumulation itself: the same kernel with the statistics on (two more scalars per env-step)
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        run_steps(args.steps)
        t1.record()
        barrier()
        stats_info = {"all_reduce_ms": sorted(ts)[len(ts) // 2], "backend": "nccl" if world > 1 else "none (one rank)",
                      "payload_bytes": 32, "includes": "sum over 32 stripes + clone + all_reduce(SUM) + D2H of 4 doubles",
                      "ms_per_step_with_statistics": t0.elapsed_time(t1) / args.steps,
                      "episodes_seen": summary["episodes"]}
        env.enable_episode_stats(False)

    extra = None
    if rank == 0 and world == 1 and not args.no_extra:
        try:
            extra = other_configs(local, peak)
        except Exception as exc:  # the headline line must not be lost to a secondary measurement
            extra = {"error": repr(exc)}
    if not args.no_extra:  # every rank takes part: the strong-scaling form of the headline config
        try:
            strong = c3_strong(rank, world, local, peak, dist)
        except Exception as exc:
            strong = {"error": repr(exc)}
        extra = dict(extra or {}, cartpole_swingup_c3_strong=strong)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O
        O.build()
        cpu = cpu_baseline(O.TASK_CARTPOLE_CONTINUOUS_SWINGUP, args.cpu_seconds)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64" if args.dtype == "float64" else "f32", "data": "synthetic",
                "config": {"workload": f"{args.env_id}, {n} envs per GPU, 1 kHz physics, 1 physics step per env step",
                           "envs_per_gpu": n, "global_envs": world * n, "parallelism": f"env-index sharding x{world}",
                           "l2": "inputs larger than L2 (per-step working set %.0f MB vs 126 MB L2)"
                                 % (env.bytes_per_env_step * n / 1e6),
                           "actions": "pre-generated on device, 4 buffers cycled",
                           "timing": "%d timed steps after %d warm-up steps, median of %d blocks, each bracketed by "
                                     "barrier + synchronize" % (args.steps, args.warmup, nblocks)},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "repeats": repeat_info}
        if stats_info is not None:
            line["episode_statistics"] = stats_info
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if extra is not None:
            line["other_configs"] = extra
        if json_fd is None:
            print(json.dumps(line))
        else:
            sys.stdout.flush()
            os.write(json_fd, (json.dumps(line) + "\n").encode())
    env.close()
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
