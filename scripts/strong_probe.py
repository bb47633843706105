"""One GPU's share of BASELINE config 3 as written (1,048,576 cart-pole envs split over 8 / 4 / 2 GPUs = 131,072 / 262,144 /
524,288 envs per GPU), timed on ONE B200: eager launches and a CUDA graph of 64 launches.

    python scripts/strong_probe.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def probe(n):
    import torch
    import b2sim
    env = b2sim.BatchedTaskEnv("CartPoleContinuousSwingup-Gazebo-v0", n, seed=0, env_offset=n)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(99)
    act4 = ((torch.rand(4, n, device="cuda", generator=gen, dtype=torch.float64) * 2 - 1) * 200.0).contiguous()

    def timed(fn, reps, steps_per_call):
        best = 1e9
        for _ in range(5):
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(reps):
                fn()
            t1.record()
            torch.cuda.synchronize()
            best = min(best, t0.elapsed_time(t1) / (reps * steps_per_call))
        return best

    for _ in range(10):
        env.rollout(act4)
    eager = timed(lambda: env.rollout(act4), 64, 4)
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
    gr = timed(graph.replay, 8, 64)
    hbm = n * env.bytes_per_env_step / 6547.2e9 * 1e6
    print(f"n={n}: eager {eager * 1e3:6.2f} us/step ({hbm / (eager * 1e3):.2f} of the HBM "
          f"roofline), graph {gr * 1e3:6.2f} us/step ({hbm / (gr * 1e3):.2f}); HBM time {hbm:.2f} us", flush=True)


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.load_package()
    for n in (131072, 262144, 524288, 1048576):
        probe(n)
