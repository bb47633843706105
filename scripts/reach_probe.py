"""PandaReach (BASELINE config 4) fused step time at several env counts."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__; __graft_entry__.load_package()
import torch, b2sim

for n in [int(a) for a in sys.argv[1:]] or (4096, 16384, 65536, 262144):
    env = b2sim.BatchedTaskEnv("PandaReach-Gazebo-v0", n, seed=0)
    q0 = torch.tensor(b2sim.batched.PANDA_Q0, device="cuda", dtype=torch.float64)
    phase = torch.rand(n, 1, device="cuda", dtype=torch.float64) * 6.2831853
    tg = (q0 + 0.1 * torch.sin(phase)).contiguous()
    tg[:, 7:] = 0.02
    for _ in range(10):
        env.step(tg)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(100):
        env.step(tg)
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 100
    print(f"n={n}: {ms * 1e3:.1f} us/step -> {n / ms * 1e3:.3e} env-steps/s", flush=True)
    env.close()
