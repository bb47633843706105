"""Per-env body inertias, joint damping / Coulomb friction and gravity (enable_env_params) on the fused reach task.

Both reach kernels read the rows on every step that runs physics. They are reached through the batch sizes at which the
engine selects them:

    k_task_panda_lanes<T, 10, 9, Panda>   the Panda, 4,095 envs (2 warps per block) and 16,381 envs (4 warps per block)
    k_task_panda_lanes<T, 8, 0>           a generated 5-joint tree, 4,093 envs
    k_task_panda_lanes<T, 10, 0>          a generated 9-joint non-Panda tree, 32,767 envs
    k_task_panda                          the Panda, 32,769 envs; B2_PANDA_KERNEL=thread at the small batches (subprocess)

Every env gets its own random rows (test_env_params_gpu.random_rows), so a kernel that reads the nominal tables, a
neighbour's row or the wrong gravity shows up in the sampled envs (first warp, a middle warp, the partial tail warp),
each compared with an oracle.Sim built from that env's own tables under the same position PIDs.
"""
import importlib.util
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _load(name, file):
    spec = importlib.util.spec_from_file_location(name, os.path.join(HERE, file))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


ep = _load("_env_params_gpu", "test_env_params_gpu.py")
gt = _load("_generated_trees_gpu", "test_generated_trees_gpu.py")

DBL_MAX = float(np.finfo(np.float64).max)
MODE_POSITION = 5
TASK_PANDA_REACH = 5
BUF_STATE, BUF_PID, BUF_OBS, BUF_REWARD, BUF_DONE, BUF_ELAPSED = 0, 5, 8, 9, 10, 11
# (model, batch size): the kernel each one selects is listed in the module docstring
CASES = [("panda", 4095), ("panda", 16381), ("g8", 4093), ("g10", 32767), ("panda", 32769)]
IDS = [f"{m}-{n}" for m, n in CASES]


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


class Reach:
    """A simulator with the reach task on `case` and what the oracle needs to follow its envs."""

    def __init__(self, torch, oracle, model_files, case, n, limit, dtype="float64", env_params_first=False):
        import b2sim
        from b2sim.batched import PANDA_PID, PANDA_Q0
        self.torch, self.oracle, self.n = torch, oracle, n
        if case == "panda":
            with open(model_files["panda"]) as f:
                self.xml = f.read()
            self.t, self.model = oracle.load_urdf(model_files["panda"])
            # resets put the fingers mid-range: a joint resting exactly on a limit (PANDA_Q0 closes the fingers) toggles
            # its row on rounding noise over the following steps, which no multi-step comparison can follow
            self.pose, self.gains, self.q0 = None, list(PANDA_PID), np.r_[PANDA_Q0[:7], 0.02, 0.02]
            self.goal = np.array([0.5, 0.0, 0.5])
            self.ee = self.t["link_names"].index("end_effector_frame")
        else:
            # "panda_tree": the Panda's body structure with random constants (the compile-time Panda lane specialisation)
            self.xml, self.t, self.model, self.ee = gt._reach_case(oracle, "panda" if case == "panda_tree" else case)
            self.pose = gt.POSE
            self.gains = [gt.GAINS] * int(self.t["nb"])
            self.q0 = np.random.default_rng(len(case)).uniform(-0.3, 0.3, int(self.t["nb"]))
            self.goal = np.array([0.3, -0.1, 0.6])
        self.nq = int(self.t["nb"])
        self.body, self.lp = int(self.t["link_body"][self.ee]), self.t["link_p"][self.ee]
        self.D = oracle.Dynamics(self.model)
        self.sim = b2sim.Simulator(n, 0.001, 1, dtype)
        self.mid = self.sim.insert_model(self.xml, **({"pose": self.pose} if self.pose else {}))
        self.rows = self.sim.enable_env_params(self.mid) if env_params_first else None
        for j, (p, i, d) in enumerate(self.gains):
            self.sim.set_pid(self.mid, j, p, i, d, DBL_MAX, -DBL_MAX, DBL_MAX, -DBL_MAX, 0.0)
        self.sim.set_task(self.mid, TASK_PANDA_REACH, max_episode_steps=limit)
        self.sim.set_task_params(self.mid, self.goal, self.q0, self.ee)
        self.sim.task_reset_all(self.mid)
        self.dtype = np.float64 if dtype == "float64" else np.float32

    def enable(self, rows=None):
        self.rows = self.sim.enable_env_params(self.mid)
        if rows is not None:
            ep.write_rows(self.torch, self.rows, rows, self.dtype)
        return self.rows

    def tensor(self, which):
        return self.sim.tensor(self.mid, which)

    def set_state(self, q, dq):
        self.tensor(BUF_STATE).copy_(self.torch.as_tensor(np.hstack([q, dq]).astype(self.dtype), device="cuda"))

    def step(self, targets):
        act = self.torch.as_tensor(targets.astype(self.dtype), device="cuda")
        self.sim.task_step(self.mid, act.data_ptr())
        self.torch.cuda.synchronize()
        return (self.tensor(BUF_OBS).cpu().numpy().astype(np.float64), self.tensor(BUF_REWARD).cpu().numpy().astype(np.float64),
                self.tensor(BUF_DONE).cpu().numpy())

    def ref(self, rows, e, q, dq):
        """oracle.Sim of env e from its own rows, position PIDs at the physics rate."""
        r = ep.oracle_sim(self.oracle, ep.env_model(self.oracle, self.t, rows, e), q, dq)
        r.set_controller_period(0.001)
        for j, (p, i, d) in enumerate(self.gains):
            r.set_pid(j, p, i, d, DBL_MAX, -DBL_MAX, DBL_MAX, -DBL_MAX, 0.0)
            r.set_control_mode(j, MODE_POSITION)
        return r

    def check(self, o, rew, r, targets, msg):
        """Steps `r` with `targets` and compares observation and reward (tolerances of test_generated_trees_gpu)."""
        nq = self.nq
        for j in range(nq):
            r.set_position_target(j, targets[j])
        r.run(False)
        qe, dqe = np.array([r.position(j) for j in range(nq)]), np.array([r.velocity(j) for j in range(nq)])
        np.testing.assert_allclose(o[:nq], qe, rtol=1e-8, atol=1e-10, err_msg=msg)
        np.testing.assert_allclose(o[nq:2 * nq], dqe, rtol=1e-7, atol=1e-9, err_msg=msg)
        R, pe = gt.link_world(self.t, self.D, qe, self.ee)
        np.testing.assert_allclose(o[2 * nq:2 * nq + 3], pe, rtol=1e-8, atol=1e-10, err_msg=msg)
        np.testing.assert_allclose(gt.quat_R(o[2 * nq + 3:2 * nq + 7]), R, atol=1e-9, err_msg=msg)
        J = o[2 * nq + 7:].reshape(6, 6 + nq)
        np.testing.assert_allclose(J[:, 6:], self.D.point_jacobian(qe, self.body, self.lp), rtol=1e-7, atol=1e-9, err_msg=msg)
        d = pe - self.t["base_p"]
        S = np.array([[0, -d[2], d[1]], [d[2], 0, -d[0]], [-d[1], d[0], 0]])
        np.testing.assert_allclose(J[:, :6], np.block([[np.eye(3), -S], [np.zeros((3, 3)), np.eye(3)]]), atol=1e-9, err_msg=msg)
        assert rew == pytest.approx(-np.linalg.norm(pe - self.goal), rel=1e-8), msg

    def random_state(self, rng):
        """Per-env states around q0 inside the joint limits, slow prismatic joints (the Panda's fingers mid-range)."""
        n, nq = self.n, self.nq
        q = self.clip(self.q0 + rng.uniform(-0.2, 0.2, (n, nq)))
        dq = rng.uniform(-0.5, 0.5, (n, nq))
        dq[:, self.t["jtype"][:nq] == 2] *= 0.1
        return q, dq

    def targets(self, rng, q):
        """Position targets near q that keep every joint off its limits over a few steps (a joint that reaches a limit
        during a multi-step comparison toggles its row on rounding: the constraint test covers the limits in one step)."""
        return self.clip(q + rng.uniform(-0.2, 0.2, q.shape))

    def clip(self, q):
        nq = self.nq
        lo, hi = self.t["lower"][:nq], self.t["upper"][:nq]
        inner = np.isfinite(lo) & np.isfinite(hi)
        mid, half = (lo[inner] + hi[inner]) / 2, (hi[inner] - lo[inner]) / 2
        q = q.copy()
        q[:, inner] = np.clip(q[:, inner], mid - 0.6 * half, mid + 0.6 * half)
        return q

    def elapsed(self):
        return self.tensor(BUF_ELAPSED).view(self.torch.int16)

    def close(self):
        self.sim.close()


def envs_of(n, nq):
    return ep.sample_envs(n, nq)


# ------------------------------------------------------------------------------------------------------------------
# 1. enabled but untouched rows = the shared tables; disabling restores the feature-off kernel
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,n", CASES, ids=IDS)
def test_untouched_rows_match_the_shared_tables(case, n, torch, oracle, model_files):
    """The rows enable_env_params fills give the feature-off results to 1e-12 over 7 steps through a TimeLimit reset; after
    enable_env_params(False) the steps are bit-identical to a simulator that never enabled."""
    a = Reach(torch, oracle, model_files, case, n, limit=5)
    b = Reach(torch, oracle, model_files, case, n, limit=5)
    b.enable()
    rng = np.random.default_rng([n, len(case)])
    q, dq = a.random_state(rng)
    for s in (a, b):
        s.set_state(q, dq)
    for step in range(7):
        tg = a.targets(rng, q)
        (oa, ra, da), (ob, rb, db) = a.step(tg), b.step(tg)
        np.testing.assert_allclose(ob, oa, rtol=1e-12, atol=1e-12 * max(1.0, np.abs(oa).max()), err_msg=f"step {step}")
        np.testing.assert_allclose(rb, ra, rtol=1e-12, atol=1e-12)
        assert np.array_equal(da, db) and da.sum() == (n if step == 4 else 0)
    assert b.sim.enable_env_params(b.mid, False) is None
    for which in (BUF_STATE, BUF_PID):
        b.tensor(which).copy_(a.tensor(which))
    for step in range(3):
        tg = a.targets(rng, q)
        a.step(tg); b.step(tg)
        for which in (BUF_STATE, BUF_PID, BUF_OBS, BUF_REWARD, BUF_DONE):
            assert torch.equal(a.tensor(which), b.tensor(which)), f"buffer {which} after disabling, step {step}"
    a.close(); b.close()


# ------------------------------------------------------------------------------------------------------------------
# 2. random rows through a TimeLimit reset
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,n", CASES, ids=IDS)
def test_random_rows_match_oracle_through_a_reset(case, n, torch, oracle, model_files):
    """7 steps with a TimeLimit of 5 and per-env targets: observation (q, dq, end-effector pose, MIXED Jacobian), reward
    and done of every sampled env against an oracle of its own rows, the reset state, and the new episode (same rows)."""
    s = Reach(torch, oracle, model_files, case, n, limit=5)
    rng = np.random.default_rng([n, len(case), 2])
    rows = ep.random_rows(rng, s.t, n)
    s.enable(rows)
    q, dq = s.random_state(rng)
    s.set_state(q, dq)
    nq = s.nq
    refs = {e: s.ref(rows, e, q[e], dq[e]) for e in envs_of(n, nq)}
    for step in range(7):
        tg = s.targets(rng, q)
        obs, rew, done = s.step(tg)
        assert done.sum() == (n if step == 4 else 0)
        for e, r in refs.items():
            s.check(obs[e], rew[e], r, tg[e], f"step {step} env {e}")
        if step == 4:
            np.testing.assert_allclose(s.tensor(BUF_STATE).cpu().numpy(), np.tile(np.r_[s.q0, np.zeros(nq)], (n, 1)))
            assert not s.tensor(BUF_PID).any() and not s.elapsed().any()
            refs = {e: s.ref(rows, e, s.q0, np.zeros(nq)) for e in refs}
    s.close()


# ------------------------------------------------------------------------------------------------------------------
# 3. constraint rows: fingers on their limits, Coulomb friction from the rows
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4095, 16381, 32769])
def test_constraint_rows_match_oracle(n, torch, oracle, model_files):
    """One step of the Panda with both fingers on a limit and driven into it, an arm joint on its upper limit in some envs,
    and the rows' Coulomb friction on half the envs. Damping is zero in every other warp of 3 envs (the lane-parallel
    constraint stage) and random elsewhere (the dense solve from the env's own inertias); on threads the impulse path and
    the dense solve split the same way. Against the oracle's dense boxed LCP at the tolerances of
    test_panda_task_limit_rows_one_step_matches_oracle."""
    s = Reach(torch, oracle, model_files, "panda", n, limit=100)
    rng = np.random.default_rng(n)
    rows = ep.random_rows(rng, s.t, n)
    rows[1][(np.arange(n) // 3) % 2 == 0, :, 0] = 0.0
    rows[1][(np.arange(n) // 3) % 2 == 1, :, 0] = rng.uniform(0.05, 0.5, ((np.arange(n) // 3) % 2 == 1).sum())[:, None]
    s.enable(rows)
    q, dq = s.random_state(rng)
    tg = np.tile(s.q0, (n, 1))
    upper = rng.random(n) < 0.5
    q[:, 7:] = np.where(upper[:, None], 0.04, 0.0)
    dq[:, 7:] = np.where(upper[:, None], 0.05, -0.05)
    tg[:, 7:] = np.where(upper[:, None], 0.09, -0.05)
    arm = rng.random(n) < 0.25
    q[arm, 3], dq[arm, 3], tg[arm, 3] = s.t["upper"][3], 0.4, s.t["upper"][3] + 0.3
    s.set_state(q, dq)
    obs, _, _ = s.step(tg)
    envs = envs_of(n, 9) + [6, 7, 8, 9, 10, 11]
    for e in envs:
        r = s.ref(rows, e, q[e], dq[e])
        for j in range(9):
            r.set_position_target(j, tg[e, j])
        r.run(False)
        qr, dqr = np.array([r.position(j) for j in range(9)]), np.array([r.velocity(j) for j in range(9)])
        np.testing.assert_allclose(obs[e, :9], qr, rtol=1e-9, atol=1e-11, err_msg=f"env {e}")
        np.testing.assert_allclose(obs[e, 9:18], dqr, rtol=1e-8, atol=1e-10, err_msg=f"env {e}")
        # the rows did act: no finger moves further into its limit (it may leave it, pushed by the arm's motion)
        assert ((obs[e, 16:18] <= 1e-12) if upper[e] else (obs[e, 16:18] >= -1e-12)).all(), f"env {e}"
    s.close()


# ------------------------------------------------------------------------------------------------------------------
# 4. rows rewritten after the step that reports done
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,n", [("panda", 4095), ("g10", 32767), ("panda", 32769)], ids=["panda-4095", "g10-32767", "panda-32769"])
def test_rows_rewritten_after_done_act_from_the_next_episode(case, n, torch, oracle, model_files):
    """Staggered episodes (ELAPSED set per env); after every step new rows are written with torch.where on the done mask.
    The terminal step of an env follows its old rows, its next episode the new ones, and the other envs keep theirs."""
    s = Reach(torch, oracle, model_files, case, n, limit=4)
    nq = s.nq
    rng = np.random.default_rng([n, 4])
    rows = s.enable(ep.random_rows(rng, s.t, n))
    elapsed = (np.arange(n) % 4).astype(np.int16)
    s.elapsed().copy_(torch.as_tensor(elapsed, device="cuda"))
    q, dq = s.random_state(rng)
    s.set_state(q, dq)
    host = [v.cpu().numpy().astype(np.float64) for v in rows]
    envs = envs_of(n, nq)
    refs = {e: s.ref(host, e, q[e], dq[e]) for e in envs}
    for step in range(6):
        tg = s.targets(rng, q)
        obs, rew, done = s.step(tg)
        assert np.array_equal(done, ((elapsed + step + 1) % 4 == 0).astype(np.uint8))
        for e, r in refs.items():
            s.check(obs[e], rew[e], r, tg[e], f"step {step} env {e}")
        fresh = ep.random_rows(rng, s.t, n)
        mask = torch.as_tensor(done, device="cuda").bool()
        for v, f in zip(rows, fresh):
            m = mask.view(-1, *([1] * (v.dim() - 1)))
            v.copy_(torch.where(m, torch.as_tensor(f.astype(s.dtype), device="cuda"), v))
        host = [v.cpu().numpy().astype(np.float64) for v in rows]
        for e in envs:
            if done[e]:
                refs[e] = s.ref(host, e, s.q0, np.zeros(nq))
    s.close()


# ------------------------------------------------------------------------------------------------------------------
# 5. a row written for one env changes that env only
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,n", CASES, ids=IDS)
def test_a_row_written_between_steps_changes_only_its_env(case, n, torch, oracle, model_files):
    """Two simulators with the same states and rows; before the second step one of them gets a heavier body, more damping,
    more friction and a tilted gravity in one env. The first step is bit-identical everywhere, the second differs in that
    env only: its neighbours in the same warp must not read its row."""
    sims = [Reach(torch, oracle, model_files, case, n, limit=100) for _ in range(2)]
    rng = np.random.default_rng([n, 5])
    rows = ep.random_rows(rng, sims[0].t, n)
    q, dq = sims[0].random_state(rng)
    for s in sims:
        s.enable(rows)
        s.set_state(q, dq)
    k = envs_of(n, sims[0].nq)[len(envs_of(n, sims[0].nq)) // 2]
    tg = sims[0].targets(rng, q)
    states = []
    for step in range(2):
        if step == 1:
            inertia, dyn, g = sims[1].rows
            inertia[k, :, 0] *= 1.5
            dyn[k, :, 0] += 0.2
            dyn[k, :, 1] += 0.1
            g[k] = torch.as_tensor([2.0, -1.0, -9.5], device="cuda")
        for s in sims:
            s.step(tg)
        states.append([np.hstack([s.tensor(BUF_STATE).cpu().numpy(), s.tensor(BUF_OBS).cpu().numpy()]) for s in sims])
    assert np.array_equal(states[0][0], states[0][1])
    a, b = states[1]
    assert list(np.nonzero((a != b).any(axis=1))[0]) == [k]
    for s in sims:
        s.close()


# ------------------------------------------------------------------------------------------------------------------
# 6. fp32
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,n", [("g8", 4093), ("panda_tree", 4095), ("panda_tree", 32769)],
                         ids=["g8-4093", "panda_tree-4095", "panda_tree-32769"])
def test_fp32_one_step_against_the_fp64_oracle(case, n, torch, oracle, model_files):
    """dtype float32 with fp32 rows (no Coulomb friction: the bound is for the smooth step), one step from the device's
    own fp32 state, against the fp64 oracle of the same (exactly converted) rows within the bound of
    test_env_params_gpu._fp32_tolerance, on the lanes (<8, 0> and the Panda specialisation) and on threads."""
    s = Reach(torch, oracle, model_files, case, n, limit=100, dtype="float32")
    nq = s.nq
    f32 = lambda a: a.astype(np.float32).astype(np.float64)
    rng = np.random.default_rng([n, 6])
    rows = ep.random_rows(rng, s.t, n)
    rows[1][..., 1] = 0.0
    rows = tuple(f32(r) for r in rows)
    s.enable(rows)
    q, dq = s.random_state(rng)
    q, dq = f32(q), f32(dq)
    tg = f32(q + rng.uniform(-0.2, 0.2, q.shape))
    s.set_state(q, dq)
    obs, _, _ = s.step(tg)
    kp, kd = np.array([g[0] for g in s.gains]), np.array([g[2] for g in s.gains])
    for e in envs_of(n, nq):
        model = ep.env_model(oracle, s.t, rows, e)
        D = oracle.Dynamics(model)
        r = s.ref(rows, e, q[e], dq[e])
        for j in range(nq):
            r.set_position_target(j, tg[e, j])
        r.run(False)
        ref = ep.oracle_state(r, nq)
        tau = kp * (tg[e] - q[e]) - kd * dq[e]
        tol_q, tol_dq = ep._fp32_tolerance(D, q[e], dq[e], D.forward_dynamics(q[e], dq[e], tau, 1e-3), nq)
        np.testing.assert_allclose(obs[e, :nq], ref[:nq], rtol=0, atol=tol_q, err_msg=f"env {e}")
        np.testing.assert_allclose(obs[e, nq:2 * nq], ref[nq:], rtol=0, atol=tol_dq, err_msg=f"env {e}")
    s.close()


# ------------------------------------------------------------------------------------------------------------------
# 7. CUDA-graph replay
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4095, 16384, 32769])
def test_steps_replayed_from_a_cuda_graph_read_the_rows_written_between_replays(n, torch):
    """Two captured steps replayed three times, new random rows written between replays (the views are the buffers the
    graph's kernels read), against eager steps with the same rows, bit for bit. 16,384 envs: the lane kernel's launch
    carries the programmatic-serialization attribute."""
    import b2sim
    from b2sim.batched import PANDA_Q0
    rng = np.random.default_rng(n)
    q0 = torch.tensor(PANDA_Q0, device="cuda", dtype=torch.float64)
    tg = (q0 + 0.1 * torch.sin(torch.arange(n, device="cuda", dtype=torch.float64)[:, None] * 0.37)).contiguous()
    tg[:, 7:] = 0.02
    envs = [b2sim.BatchedTaskEnv("PandaReach-Gazebo-v0", n, max_episode_steps=5) for _ in range(2)]
    views = [env.enable_env_params() for env in envs]
    host = [[v.cpu().numpy() for v in views[0]]]
    eager, graphed = envs
    side = torch.cuda.Stream()
    graphed.use_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            for _ in range(2):
                graphed.step(tg)
    torch.cuda.synchronize()
    graphed.reset()   # the capture does not execute: start from the same initial state
    for replay in range(3):
        inertia = host[0][0] * rng.uniform(0.7, 1.3, (n, 9, 1))
        dyn = np.stack([rng.uniform(0, 0.3, (n, 9)), rng.uniform(0, 0.2, (n, 9))], -1)
        grav = np.tile([0.0, 0.0, -9.8], (n, 1)) + rng.uniform(-0.5, 0.5, (n, 3))
        for vs in views:
            ep.write_rows(torch, vs, (inertia, dyn, grav))
        torch.cuda.synchronize()
        for _ in range(2):
            eager.step(tg)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(graphed.state, eager.state), f"replay {replay}"
        assert torch.equal(graphed.obs, eager.obs) and torch.equal(graphed.done, eager.done)
    for env in envs:
        env.close()


# ------------------------------------------------------------------------------------------------------------------
# 8. host-buffer steps in windows
# ------------------------------------------------------------------------------------------------------------------
def test_host_buffer_steps_read_each_windows_rows(torch, oracle, model_files):
    """step_host cuts 131,072 envs into two windows of 65,536 launched separately; each window must read its own envs'
    rows (offset by the window start). Against device steps with the same rows and actions, bit for bit, over 3 steps.
    The default selection runs the windows on k_task_panda; test_reach_rows_on_the_forced_kernel runs this on lanes.
    No joint reaches a constraint row (fingers mid-range, no Coulomb friction): the lane kernel picks its constraint
    path per warp, and a window that starts inside a warp of three envs groups the envs differently."""
    import b2sim
    from b2sim.batched import PANDA_Q0
    n = 131072
    rng = np.random.default_rng(8)
    envs = [b2sim.BatchedTaskEnv("PandaReach-Gazebo-v0", n, max_episode_steps=100) for _ in range(3)]
    t, _ = oracle.load_urdf(model_files["panda"])
    rows = ep.random_rows(rng, t, n)
    rows[1][..., 1] = 0.0
    q0 = torch.tensor(np.r_[PANDA_Q0[:7], 0.02, 0.02, np.zeros(9)], device="cuda")
    host, dev, plain = envs   # plain: the shared tables, to show that the rows matter
    for env in envs:
        if env is not plain:
            ep.write_rows(torch, env.enable_env_params(), rows)
        env.state.copy_(q0.expand(n, 18))
    obs, rew, done = np.empty((n, host.nobs)), np.empty(n), np.empty(n, np.uint8)
    for step in range(3):
        act = np.tile(PANDA_Q0, (n, 1)) + rng.uniform(-0.2, 0.2, (n, 9))
        act[:, 7:] = 0.02
        host.step_host(act, obs, rew, done)
        o, r, d = dev.step(torch.as_tensor(act, device="cuda"))
        plain.step(torch.as_tensor(act, device="cuda"))
        torch.cuda.synchronize()
        assert np.array_equal(obs, o.cpu().numpy()), f"step {step}"
        assert np.array_equal(rew, r.cpu().numpy()) and np.array_equal(done, d.cpu().numpy())
        assert torch.equal(host.state, dev.state)
    assert not (plain.obs == dev.obs).all(dim=1).any()
    for env in envs:
        env.close()


# ------------------------------------------------------------------------------------------------------------------
# 9. enabling with a reach task, in either order; the batched environment
# ------------------------------------------------------------------------------------------------------------------
def test_enable_and_set_task_in_either_order(torch, oracle, model_files):
    """enable_env_params before and after set_task(reach) give the same steps with the same rows; the batched environment
    forwards enable_env_params and counts the rows in bytes_per_env_step (12 nq + 3 scalars), also after
    enable_episode_stats; the cart-pole task is still refused."""
    import b2sim
    from b2sim import _lib
    n = 4095
    rng = np.random.default_rng(9)
    first = Reach(torch, oracle, model_files, "panda", n, limit=3, env_params_first=True)
    then = Reach(torch, oracle, model_files, "panda", n, limit=3)
    rows = ep.random_rows(rng, first.t, n)
    ep.write_rows(torch, first.rows, rows)
    then.enable(rows)
    q, dq = first.random_state(rng)
    for s in (first, then):
        s.set_state(q, dq)
    for step in range(4):
        tg = first.targets(rng, q)
        first.step(tg); then.step(tg)
        assert torch.equal(first.tensor(BUF_OBS), then.tensor(BUF_OBS)), f"step {step}"
    first.close(); then.close()

    env = b2sim.BatchedTaskEnv("PandaReach-Gazebo-v0", 64)
    assert env.bytes_per_env_step == 1722
    inertia, dyn, g = env.enable_env_params()
    assert tuple(inertia.shape) == (64, 9, 10) and tuple(dyn.shape) == (64, 9, 2) and tuple(g.shape) == (64, 3)
    assert env.bytes_per_env_step == 1722 + 888
    env.enable_episode_stats()
    assert env.bytes_per_env_step == 1722 + 888 + 16
    assert env.enable_env_params(False) is None and env.bytes_per_env_step == 1722 + 16
    env.close()
    env = b2sim.BatchedTaskEnv("PandaReach-Gazebo-v0", 64, dtype="float32")
    env.enable_env_params()
    assert env.bytes_per_env_step == 862 + 444
    env.close()
    env = b2sim.BatchedTaskEnv("CartPoleContinuousSwingup-Gazebo-v0", 64)
    with pytest.raises(b2sim.B2Error) as err:
        env.enable_env_params()
    assert err.value.code == _lib.ERR_UNSUPPORTED and env.bytes_per_env_step == 114
    env.close()


# ------------------------------------------------------------------------------------------------------------------
# the other kernel at the same batch sizes
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["thread", "lanes"])
def test_reach_rows_on_the_forced_kernel(variant):
    """B2_PANDA_KERNEL (read once per process) forces one reach kernel in a fresh process: "thread" runs the small-batch
    cases of this file on k_task_panda, "lanes" runs the two-window host-buffer steps on k_task_panda_lanes."""
    import subprocess
    import sys
    sel = {"thread": "(4095 or 4093 or 16381 or 16384) and not forced",
           "lanes": "test_host_buffer_steps_read_each_windows_rows"}[variant]
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", os.path.abspath(__file__), "-k", sel],
                       env=dict(os.environ, B2_PANDA_KERNEL=variant), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
