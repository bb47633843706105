"""Cost of per-env physical parameters (Simulator.enable_env_params) on GazeboSimulator::run of Pandas under position PIDs,
and on the fused PandaReach step (BatchedTaskEnv.enable_env_params).

Two simulators with the same Pandas, targets and gains (those of run_probe.py), one with its own random rows per env
(masses x U(0.8, 1.2), inertias alike, damping U(0, 0.1), gravity tilted by up to ~3 degrees), the other on the shared
tables. Blocks of `runs` b2sim_run calls alternate between the two in one process and are timed with CUDA events; the
median of 5 blocks per variant is reported. The batch size selects the kernel: 4,096 and 16,384 envs run on lanes
(k_run_tree_lanes), 20,001 on k_run_tree and 65,536 on k_run_tree_local.

The reach step is timed the same way (blocks of `runs` env.step calls): 4,096 and 16,384 envs on k_task_panda_lanes with
the fingers held mid-range, 16,384 envs with the fingers driven into their lower limits (limit rows on every step) with
damped rows (the dense constraint solve) and with undamped ones (the lane-parallel stage), 65,536 envs on k_task_panda. Last, the cost of redrawing every row of 16,384 envs once (the per-episode pattern: new
rows after the step that reports done) with torch, against the step it precedes.

Worlds with free bodies (Simulator.enable_free_body_params / enable_shape_friction), timed the same way: the pick scene's
grasp step at 4,096 envs (the forked coupled pipeline), two stacked cubes at 4,096 envs (k_world_prepare / k_pgs_solve /
k_world_finish) and at 65,536 envs (k_world_free). "on": the cubes' masses x U(0.8, 1.2), centres of mass within 2 mm,
inertias x U(0.8, 1.2), and friction U(0.6, 1.2) on every shape that takes part (cube, table, finger pads; cubes, ground);
"untouched": the same rows enabled and left at their initial values (the kernels' cost without a change of the physics).

    python scripts/env_params_probe.py [runs_per_block] [all|world]
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = {4096: "k_run_tree_lanes", 16384: "k_run_tree_lanes", 20001: "k_run_tree", 65536: "k_run_tree_local"}
GAINS = [(50, 0, 20), (10000, 0, 500), (100, 0, 10), (1000, 0, 50), (100, 0, 10), (100, 0, 10), (10, 0.5, 0.1), (100, 0, 50),
         (100, 0, 50)]


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout
    return out.strip().splitlines()[0]


def panda_sim(n, env_params, seed):
    import torch
    import b2sim
    import gym_ignition_models
    from b2sim import _lib as L
    from b2sim.batched import PANDA_Q0
    sim = b2sim.Simulator(n, 0.001, 1)
    mid = sim.insert_model_file(gym_ignition_models.get_model_file("panda"))
    for j in range(9):
        sim.set_joint(mid, L.FIELD_POSITION_RESET, -1, j, PANDA_Q0[j])
    sim.run(paused=True)
    big = 1.7976931348623157e308
    sim.set_controller_period(mid, 0.001)
    for j, (p, i, d) in enumerate(GAINS):
        sim.set_pid(mid, j, p, i, d, big, -big, big, -big, 0.0)
        sim.set_control_mode(mid, j, 5)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    f64 = dict(device="cuda", dtype=torch.float64)
    tg = sim.tensor(mid, L.BUF_POS_TARGET)
    tg.copy_(torch.tensor(PANDA_Q0, **f64) + 0.1 * torch.sin(torch.rand(n, 1, generator=gen, **f64) * 6.28))
    tg[:, 7:] = 0.02
    if env_params:
        inertia, dyn, g = sim.enable_env_params(mid)
        s = 0.8 + 0.4 * torch.rand(n, 9, 1, generator=gen, **f64)
        inertia[:, :, 0:1] *= s
        inertia[:, :, 4:] *= s
        dyn[:, :, 0] = 0.1 * torch.rand(n, 9, generator=gen, **f64)
        g[:, :2] = 0.5 * (torch.rand(n, 2, generator=gen, **f64) - 0.5)
    return sim


def draw_rows(views, nominal, gen, damped=True):
    """New random rows from the nominal ones, written in place (what a caller does at its resets)."""
    import torch
    inertia, dyn, g = views
    n = inertia.shape[0]
    f64 = dict(device="cuda", dtype=torch.float64)
    s = 0.8 + 0.4 * torch.rand(n, 9, 1, generator=gen, **f64)
    inertia[:, :, 0:1] = nominal[:, :, 0:1] * s
    inertia[:, :, 1:4] = nominal[:, :, 1:4]
    inertia[:, :, 4:] = nominal[:, :, 4:] * s
    dyn[:, :, 0] = 0.1 * torch.rand(n, 9, generator=gen, **f64) if damped else 0.0
    g[:, :2] = 0.5 * (torch.rand(n, 2, generator=gen, **f64) - 0.5)


def reach_env(n, env_params, fingers, seed, damped=True):
    import torch
    import b2sim
    from b2sim.batched import PANDA_Q0
    env = b2sim.BatchedTaskEnv("PandaReach-Gazebo-v0", n)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    f64 = dict(device="cuda", dtype=torch.float64)
    tg = (torch.tensor(PANDA_Q0, **f64) + 0.1 * torch.sin(torch.rand(n, 1, generator=gen, **f64) * 6.28)).contiguous()
    tg[:, 7:] = 0.02 if fingers == "mid" else -0.05
    if env_params:
        views = env.enable_env_params()
        draw_rows(views, views[0].clone(), gen, damped)
    return env, tg


def timed(fn, runs):
    """Microseconds per call of fn over `runs` calls, CUDA events."""
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(runs):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / runs * 1e3


def reach(runs):
    import numpy as np
    import torch
    # damped=False: the rows keep the Panda's zero joint damping, so limit rows stay on the lane-parallel constraint stage
    for n, kernel, fingers, damped in ((4096, "k_task_panda_lanes", "mid", True), (16384, "k_task_panda_lanes", "mid", True),
                                       (16384, "k_task_panda_lanes", "limits", True),
                                       (16384, "k_task_panda_lanes", "limits", False), (65536, "k_task_panda", "mid", True)):
        envs = {"off": reach_env(n, False, fingers, 3), "on": reach_env(n, True, fingers, 3, damped)}
        for env, tg in envs.values():  # warm-up: module loads, clocks
            for _ in range(200):
                env.step(tg)
        torch.cuda.synchronize()
        times = {k: [] for k in envs}
        for block in range(5):
            for name, (env, tg) in envs.items():
                times[name].append(timed(lambda: env.step(tg), runs))
        off, on = (float(np.median(times[k])) for k in ("off", "on"))
        spread = {k: (min(v), max(v)) for k, v in times.items()}
        print(f"reach n={n:6d} {kernel:18s} fingers {fingers:6s} {'damped' if damped else 'undamped':8s} off {off:7.2f} us/step (blocks {spread['off'][0]:.2f}-"
              f"{spread['off'][1]:.2f})  on {on:7.2f} us/step (blocks {spread['on'][0]:.2f}-{spread['on'][1]:.2f})  "
              f"on/off {on / off:.3f}", flush=True)
        for env, _ in envs.values():
            env.close()
    n = 16384
    env, tg = reach_env(n, False, "mid", 3)
    views = env.enable_env_params()
    nominal = views[0].clone()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(5)
    for _ in range(200):
        draw_rows(views, nominal, gen)
        env.step(tg)
    torch.cuda.synchronize()
    draw = float(np.median([timed(lambda: draw_rows(views, nominal, gen), runs) for _ in range(5)]))
    step = float(np.median([timed(lambda: env.step(tg), runs) for _ in range(5)]))
    print(f"reach n={n:6d} redraw of every row {draw:7.2f} us  (one step {step:7.2f} us)", flush=True)
    env.close()


def world_rows(sim, cubes, shaped, gen):
    """Random free-body rows on `cubes` and friction rows on every model of `shaped` (rows "on")."""
    import torch
    for m in cubes:
        rows = sim.enable_free_body_params(m)
        opts = dict(device=rows.device, dtype=rows.dtype)
        n = rows.shape[0]
        s = 0.8 + 0.4 * torch.rand(n, 1, generator=gen, **opts)
        rows[:, 0:1] *= s
        rows[:, 1:4] = 0.002 * (2 * torch.rand(n, 3, generator=gen, **opts) - 1) / 3 ** 0.5
        rows[:, 4:] *= s
    for m in shaped:
        mu = sim.enable_shape_friction(m)
        mu.copy_(0.6 + 0.6 * torch.rand(mu.shape, generator=gen, device=mu.device, dtype=mu.dtype))


def pick_world(n, rows_on, seed):
    import torch
    import b2sim
    sc = b2sim.PandaPickScene(n, seed=seed)
    if rows_on == "untouched":
        sc.sim.enable_free_body_params(sc.cube)
        for m in (sc.cube, sc.table, sc.panda):
            sc.sim.enable_shape_friction(m)
    elif rows_on:
        gen = torch.Generator(device="cuda")
        gen.manual_seed(seed)
        world_rows(sc.sim, [sc.cube], [sc.cube, sc.table, sc.panda], gen)
    sc.step(30)
    sc.set_fingers(0.0)
    sc.step(150)  # grasping from here on
    return sc.sim, sc


def stacked_world(n, rows_on, seed):
    import torch
    import b2sim
    import gym_ignition_models
    from b2sim import _lib as L
    sim = b2sim.Simulator(n, 0.001, 1)
    ground = sim.insert_model_file(gym_ignition_models.get_model_file("ground_plane"))
    cube = """<robot name="cube"><link name="cube"><inertial><mass value="5.0"/>
      <inertia ixx="0.0333" ixy="0" ixz="0" iyy="0.0333" iyz="0" izz="0.0333"/></inertial>
      <collision><geometry><box size="0.2 0.2 0.2"/></geometry></collision></link></robot>"""
    cubes = [sim.insert_model(cube, pose=(0, 0, z, 1, 0, 0, 0), name=f"c{k}") for k, z in enumerate((0.1, 0.3))]
    if rows_on == "untouched":
        for m in cubes:
            sim.enable_free_body_params(m)
        for m in [ground] + cubes:
            sim.enable_shape_friction(m)
    elif rows_on:
        gen = torch.Generator(device="cuda")
        gen.manual_seed(seed)
        world_rows(sim, cubes, [ground] + cubes, gen)
    for _ in range(300):  # settle
        sim.run()
    assert sim.tensor(cubes[1], L.BUF_BASE_STATE)[:, 2].min().item() > 0.25
    return sim, None


def worlds(runs):
    import numpy as np
    import torch
    for name, n, kernels, make in (("pick grasp step", 4096, "forked coupled pipeline", pick_world),
                                   ("two stacked cubes", 4096, "k_world_prepare/k_pgs_solve/k_world_finish", stacked_world),
                                   ("two stacked cubes", 65536, "k_world_free", stacked_world)):
        worlds_ = {"off": make(n, False, 3), "untouched": make(n, "untouched", 3), "on": make(n, True, 3)}
        for sim, _ in worlds_.values():  # warm-up
            for _ in range(100):
                sim.run()
        torch.cuda.synchronize()
        times = {k: [] for k in worlds_}
        for block in range(5):
            for key, (sim, _) in worlds_.items():
                times[key].append(timed(sim.run, runs))
        med = {k: float(np.median(v)) for k, v in times.items()}
        contacts = {k: np.mean([len(sim.contacts(e)) for e in range(0, n, max(1, n // 64))]) for k, (sim, _) in worlds_.items()}
        print(f"world {name:17s} n={n:6d} {kernels:43s} " + "  ".join(
            f"{k} {med[k]:8.2f} us/step (blocks {min(v):.2f}-{max(v):.2f}, {contacts[k]:.1f} contacts)"
            for k, v in times.items()) + f"  untouched/off {med['untouched'] / med['off']:.3f}  on/off {med['on'] / med['off']:.3f}",
            flush=True)
        for sim, sc in worlds_.values():
            (sc or sim).close()


def main():
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.load_package()
    import numpy as np
    import torch
    runs = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
    section = sys.argv[2] if len(sys.argv) > 2 else "all"
    print(f"card: {card()}", flush=True)
    if section == "world":
        worlds(max(1, runs // 5))
        return
    for n, kernel in SIZES.items():
        sims = {"off": panda_sim(n, False, 3), "on": panda_sim(n, True, 3)}
        for sim in sims.values():  # warm-up: module loads, clocks
            for _ in range(200):
                sim.run()
        torch.cuda.synchronize()
        times = {k: [] for k in sims}
        for block in range(5):
            for name, sim in sims.items():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(runs):
                    sim.run()
                b.record()
                torch.cuda.synchronize()
                times[name].append(a.elapsed_time(b) / runs * 1e3)
        off, on = (float(np.median(times[k])) for k in ("off", "on"))
        spread = {k: (min(v), max(v)) for k, v in times.items()}
        print(f"n={n:6d} {kernel:17s} off {off:7.2f} us/run (blocks {spread['off'][0]:.2f}-{spread['off'][1]:.2f})  "
              f"on {on:7.2f} us/run (blocks {spread['on'][0]:.2f}-{spread['on'][1]:.2f})  on/off {on / off:.3f}", flush=True)
        for sim in sims.values():
            sim.close()
    reach(runs)
    worlds(max(1, runs // 5))


if __name__ == "__main__":
    main()
