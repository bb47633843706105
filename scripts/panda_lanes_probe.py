"""A/B of the fused Panda task kernels (BASELINE config 4): one thread per env (k_task_panda) against G lanes per env
(k_task_panda_lanes). Each variant runs in its own process (the choice is read once from B2_PANDA_KERNEL); the parent
compares the observations after T steps and prints the time per launch.

    python scripts/panda_lanes_probe.py [n_envs] [dtype]
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def child(n, dtype, out):
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.load_package()
    import numpy as np
    import torch
    import b2sim

    tdt = torch.float64 if dtype == "float64" else torch.float32
    env = b2sim.BatchedTaskEnv("PandaReach-Gazebo-v0", n, dtype=dtype, seed=0, max_episode_steps=150)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(7)
    q0 = torch.tensor(b2sim.batched.PANDA_Q0, device="cuda", dtype=tdt)
    phase = torch.rand(n, 1, device="cuda", generator=gen, dtype=tdt) * 6.2831853
    tg = (q0 + 0.1 * torch.sin(phase)).contiguous()
    tg[:, 7:] = -0.01 if os.environ.get("PROBE_FINGERS") == "limit" else 0.02  # limit: two joint-limit rows per env
    T = 200
    for _ in range(T):
        obs, rew, done = env.step(tg)
    torch.cuda.synchronize()
    np.savez(out, obs=obs.cpu().numpy()[:4096], rew=rew.cpu().numpy()[:4096], state=env.state.cpu().numpy()[:4096],
             elapsed=env.elapsed.cpu().numpy()[:4096])
    best = 1e9
    for rep in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(100):
            env.step(tg)
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b) / 100)
    print(f"{os.environ.get('B2_PANDA_KERNEL', 'lanes'):7s} fingers={os.environ.get('PROBE_FINGERS', 'free')} n={n} {dtype}: "
          f"{best * 1e3:8.1f} us/launch  {n / best * 1e3:.3e} env-steps/s", flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--child":
        child(int(sys.argv[2]), sys.argv[3], sys.argv[4])
        sys.exit(0)
    import numpy as np
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 16384
    dtype = sys.argv[2] if len(sys.argv) > 2 else "float64"
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    outs = {}
    for variant in ("thread", "lanes"):
        out = os.path.join(ROOT, "gpurun_out", f"panda_{variant}.npz")
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--child", str(n), dtype, out],
                              env=dict(os.environ, B2_PANDA_KERNEL=variant))
        outs[variant] = np.load(out)
    a, b = outs["thread"], outs["lanes"]
    for k in ("obs", "rew", "state"):
        d = np.abs(a[k] - b[k]) / (1e-9 + np.abs(a[k]))
        print(f"{k}: max rel diff thread vs lanes = {d.max():.3e}")
    print("elapsed equal:", np.array_equal(a["elapsed"], b["elapsed"]))
