"""Per-env body inertias, joint damping / Coulomb friction and gravity (Simulator.enable_env_params) on every run kernel.

The kernels are reached through the batch sizes of test_generated_trees_gpu.py (lanes with 2 and 4 warps per block:
8,191 / 16,381 envs; k_run_tree: 20,001; k_run_tree_local: 65,537; fewer than 4 joints always run one thread per env).
Every env gets its own random rows, so a kernel that reads the nominal tables, a neighbour's row or the wrong gravity
shows up in the sampled envs (first warp, a middle warp, the partial tail warp), each compared with an oracle.Sim built
from that env's own tables.
"""
import copy
import importlib.util
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("tree_urdf", os.path.join(HERE, "helpers", "tree_urdf.py"))
tree_urdf = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(tree_urdf)

DBL_MAX = float(np.finfo(np.float64).max)
MODE_FORCE, MODE_FOLLOWER, MODE_POSITION = 2, 4, 5
F_PT, F_VT, F_AT = 5, 6, 9
BUF_STATE, BUF_FCMD, BUF_POS_T, BUF_VEL_T, BUF_ACC_T, BUF_LINK_POSE = 0, 2, 3, 4, 16, 13
POSE = (0.1, -0.2, 0.3, 0.9238795325112867, 0.0, 0.3826834323650898, 0.0)
GAINS = (20.0, 0.5, 1.0)
RUN_SIZES = [8191, 16381, 20001, 65537]
SYM = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def lane_group(nq):
    return 8 if nq <= 8 else (10 if nq <= 10 else 16)


def sample_envs(n, nq):
    """First warp, second warp of a block in the middle, partial tail warp of the lane kernels (test_generated_trees_gpu)."""
    epw = 32 // lane_group(nq)
    per_block = (2 if n <= 8192 else 4) * epw
    b = (n // per_block) // 2
    tail = (n - 1) // epw * epw
    envs = set(range(epw)) | set(range(b * per_block + epw, b * per_block + 2 * epw)) | set(range(tail, n))
    return sorted(e for e in envs if e < n)


def make_tree(oracle, nq, topology, seed, **kw):
    xml = tree_urdf.generate(nq, topology, seed=seed, **kw)
    t, model = oracle.load_urdf(xml, base_position=POSE[:3], base_orientation_wxyz=POSE[3:])
    return xml, t, model


def random_state(rng, t, n):
    nq = int(t["nb"])
    prism = t["jtype"][:nq] == 2
    q = rng.uniform(-1.5, 1.5, (n, nq))
    q[:, prism] = rng.uniform(-0.2, 0.2, (n, int(prism.sum())))
    return q, rng.uniform(-1.0, 1.0, (n, nq))


def random_rows(rng, t, n):
    """Distinct physical parameters per env: mass x U(0.5, 2) with the inertia scaled alike (even envs) or a random
    physically valid inertia (odd envs: tr(S) 1 - S for a random positive S), a shifted centre of mass, damping U(0, 0.5)
    (zero on every other group of 4 envs, whole warps, so that the undamped constraint path runs too), Coulomb friction
    U(0, 0.3) on half the envs, gravity of random direction with magnitude 9.8 +- 1."""
    nq = int(t["nb"])
    s = rng.uniform(0.5, 2.0, (n, nq))
    mass = t["mass"][:nq] * s
    com = t["com"][:nq] + rng.uniform(-0.03, 0.03, (n, nq, 3))
    Ic = t["Ic"][:nq][None] * s[..., None, None]
    A = rng.normal(size=(n, nq, 3, 3))
    S = A @ np.swapaxes(A, -1, -2) * (0.01 * np.trace(t["Ic"][:nq], axis1=1, axis2=2)[None, :, None, None] + 1e-4)
    rnd = np.trace(S, axis1=-2, axis2=-1)[..., None, None] * np.eye(3) - S
    Ic[1::2] = rnd[1::2]
    inertia = np.concatenate([mass[..., None], com, np.stack([Ic[..., i, j] for i, j in SYM], -1)], -1)
    damping = rng.uniform(0.0, 0.5, (n, nq))
    damping[(np.arange(n) // 4) % 2 == 0] = 0.0
    friction = rng.uniform(0.0, 0.3, (n, nq))
    friction[rng.random(n) < 0.5] = 0.0
    d = rng.normal(size=(n, 3))
    g = d / np.linalg.norm(d, axis=1, keepdims=True) * rng.uniform(8.8, 10.8, (n, 1))
    return inertia, np.stack([damping, friction], -1), g


def env_model(oracle, t, rows, e, gravity=None):
    """oracle.Model of env e: the nominal tables with the env's rows."""
    inertia, dyn, g = rows
    nq = int(t["nb"])
    te = copy.deepcopy(t)
    te["mass"][:nq] = inertia[e, :, 0]
    te["com"][:nq] = inertia[e, :, 1:4]
    for k, (i, j) in enumerate(SYM):
        te["Ic"][:nq, i, j] = inertia[e, :, 4 + k]
        te["Ic"][:nq, j, i] = inertia[e, :, 4 + k]
    te["damping"][:nq] = dyn[e, :, 0]
    te["friction"][:nq] = dyn[e, :, 1]
    te["gravity"] = np.array(g[e] if gravity is None else gravity, float)
    return oracle.model_from_tables(te)


def new_sim(torch, xml, n, q, dq, steps_per_run=1, dtype="float64", pose=POSE):
    import b2sim
    sim = b2sim.Simulator(n, 0.001, steps_per_run, dtype)
    mid = sim.insert_model(xml, pose=pose)
    sim.tensor(mid, BUF_STATE).copy_(torch.as_tensor(np.hstack([q, dq]), device="cuda"))
    return sim, mid


def write_rows(torch, views, rows, dtype=np.float64):
    for v, r in zip(views, rows):
        v.copy_(torch.as_tensor(r.astype(dtype), device="cuda"))


def oracle_sim(oracle, model, q, dq, steps_per_run=1):
    r = oracle.Sim(model, 0.001, steps_per_run)
    for j in range(model.nb):
        r.reset_position(j, float(q[j])); r.reset_velocity(j, float(dq[j]))
    r.run(True)
    return r


def oracle_state(r, nq):
    return np.array([r.position(j) for j in range(nq)] + [r.velocity(j) for j in range(nq)])


def assert_state(got, ref, tol, msg):
    scale = max(1.0, float(np.abs(ref).max()))
    np.testing.assert_allclose(got, ref, rtol=tol, atol=tol * scale, err_msg=msg)


def set_modes(sim, mid, refs, nq, mode=MODE_FORCE):
    for j in range(nq):
        sim.set_control_mode(mid, j, mode)
        for r in refs.values():
            r.set_control_mode(j, mode)


# ------------------------------------------------------------------------------------------------------------------
# 1. enabled but untouched rows = the shared tables
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", RUN_SIZES)
@pytest.mark.parametrize("nq,topology,kw", [(9, "random", {}), (5, "base_children", dict(damping=0.2, friction=0.05))])
def test_untouched_rows_match_the_shared_tables(nq, topology, kw, n, torch, oracle):
    """The rows enable_env_params fills (loader tables, world gravity) give the feature-off results to 1e-12 over 10 runs
    of per-env random torques, for every env."""
    xml, t, _ = make_tree(oracle, nq, topology, seed=100 + nq, **kw)
    rng = np.random.default_rng([nq, n])
    q, dq = random_state(rng, t, n)
    sims = [new_sim(torch, xml, n, q, dq) for _ in range(2)]
    inertia, dyn, g = sims[1][0].enable_env_params(sims[1][1])
    assert tuple(inertia.shape) == (n, nq, 10) and tuple(dyn.shape) == (n, nq, 2) and tuple(g.shape) == (n, 3)
    np.testing.assert_allclose(inertia[-1].cpu().numpy()[:, 0], t["mass"][:nq], rtol=1e-12)
    np.testing.assert_allclose(dyn[0].cpu().numpy(), np.stack([t["damping"][:nq], t["friction"][:nq]], -1), rtol=1e-12)
    assert np.array_equal(g.cpu().numpy(), np.tile([0.0, 0.0, -9.8], (n, 1)))
    for sim, mid in sims:
        for j in range(nq):
            sim.set_control_mode(mid, j, MODE_FORCE)
    for run in range(10):
        tau = torch.as_tensor(rng.uniform(-2, 2, (n, nq)), device="cuda")
        for sim, mid in sims:
            sim.tensor(mid, BUF_FCMD).copy_(tau)
            sim.run()
    a, b = (sim.tensor(mid, BUF_STATE).cpu().numpy() for sim, mid in sims)
    np.testing.assert_allclose(b, a, rtol=1e-12, atol=1e-12 * max(1.0, np.abs(a).max()))
    for sim, _ in sims:
        sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 2. random rows, force mode
# ------------------------------------------------------------------------------------------------------------------
RUN_TREES = [(3, "chain"), (6, "random"), (9, "random"), (13, "base_children"), (16, "random")]


@pytest.mark.parametrize("n", RUN_SIZES)
@pytest.mark.parametrize("nq,topology", RUN_TREES)
def test_random_rows_force_mode_match_oracle(nq, topology, n, torch, oracle):
    """Trees with prismatic joints and welded links, one and three physics steps per run, per-env torques: every run of
    every sampled env at 1e-9 of the state scale against an oracle.Sim of the env's own tables."""
    xml, t, _ = make_tree(oracle, nq, topology, seed=200 + nq)
    assert (t["jtype"][:nq] == 2).any() or nq <= 3
    envs = sample_envs(n, nq)
    for spr in (1, 3):
        rng = np.random.default_rng([nq, n, spr])
        q, dq = random_state(rng, t, n)
        rows = random_rows(rng, t, n)
        sim, mid = new_sim(torch, xml, n, q, dq, spr)
        write_rows(torch, sim.enable_env_params(mid), rows)
        models = {e: env_model(oracle, t, rows, e) for e in envs}
        refs = {e: oracle_sim(oracle, models[e], q[e], dq[e], spr) for e in envs}
        set_modes(sim, mid, refs, nq)
        state, fcmd = sim.tensor(mid, BUF_STATE), sim.tensor(mid, BUF_FCMD)
        for run in range(5):
            tau = rng.uniform(-2, 2, (n, nq))
            fcmd.copy_(torch.as_tensor(tau, device="cuda"))
            sim.run()
            got = state.cpu().numpy()
            for e, r in refs.items():
                for j in range(nq):
                    r.set_force_target(j, tau[e, j])
                r.run(False)
                assert_state(got[e], oracle_state(r, nq), 1e-9, f"spr {spr} run {run} env {e}")
        sim.close()


@pytest.mark.parametrize("n", [64, 20001, 65537])
@pytest.mark.parametrize("name", ["pendulum", "cartpole"])
def test_pendulum_and_cartpole_rows_match_oracle(name, n, torch, oracle, model_files):
    """The closed-form chain models outside a task run on the thread kernels: with random rows they follow the env's own
    tables (the closed-form fit of the shared tables must not be used)."""
    t, _ = oracle.load_urdf(model_files[name])
    nq = int(t["nb"])
    with open(model_files[name]) as f:
        xml = f.read()
    rng = np.random.default_rng([nq, n])
    q, dq = rng.uniform(-1, 1, (n, nq)), rng.uniform(-1, 1, (n, nq))
    rows = random_rows(rng, t, n)
    rows[1][..., 1] = 0.0   # no Coulomb friction here: the rows keep to the smooth dynamics of the closed forms
    sim, mid = new_sim(torch, xml, n, q, dq, pose=(0, 0, 0, 1, 0, 0, 0))
    write_rows(torch, sim.enable_env_params(mid), rows)
    envs = [0, 1, n // 2, n - 1]
    refs = {e: oracle_sim(oracle, env_model(oracle, t, rows, e), q[e], dq[e]) for e in envs}
    set_modes(sim, mid, refs, nq)
    for run in range(5):
        tau = rng.uniform(-2, 2, (n, nq))
        sim.tensor(mid, BUF_FCMD).copy_(torch.as_tensor(tau, device="cuda"))
        sim.run()
        got = sim.tensor(mid, BUF_STATE).cpu().numpy()
        for e, r in refs.items():
            for j in range(nq):
                r.set_force_target(j, tau[e, j])
            r.run(False)
            assert_state(got[e], oracle_state(r, nq), 1e-9, f"run {run} env {e}")
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 3. position PIDs
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4093, 20001])
@pytest.mark.parametrize("nq,topology", [(7, "base_children"), (14, "random")])
def test_random_rows_position_pids_match_oracle(nq, topology, n, torch, oracle):
    """Position PIDs at the physics rate, per-env targets, 10 runs of 2 physics steps."""
    xml, t, _ = make_tree(oracle, nq, topology, seed=500 + nq)
    envs = sample_envs(n, nq)
    rng = np.random.default_rng([nq, n])
    q, dq = random_state(rng, t, n)
    rows = random_rows(rng, t, n)
    sim, mid = new_sim(torch, xml, n, q, dq, 2)
    write_rows(torch, sim.enable_env_params(mid), rows)
    refs = {e: oracle_sim(oracle, env_model(oracle, t, rows, e), q[e], dq[e], 2) for e in envs}
    qt = q + rng.uniform(-0.1, 0.1, (n, nq))
    sim.set_controller_period(mid, 0.001)
    for j in range(nq):
        sim.set_pid(mid, j, *GAINS, DBL_MAX, -DBL_MAX, DBL_MAX, -DBL_MAX, 0.0)
        sim.set_control_mode(mid, j, MODE_POSITION)
    sim.tensor(mid, BUF_POS_T).copy_(torch.as_tensor(qt, device="cuda"))
    for e, r in refs.items():
        r.set_controller_period(0.001)
        for j in range(nq):
            r.set_pid(j, *GAINS, DBL_MAX, -DBL_MAX, DBL_MAX, -DBL_MAX, 0.0)
            r.set_control_mode(j, MODE_POSITION)
            r.set_position_target(j, qt[e, j])
    state = sim.tensor(mid, BUF_STATE)
    for run in range(10):
        sim.run()
        got = state.cpu().numpy()
        for e, r in refs.items():
            r.run(False)
            assert_state(got[e], oracle_state(r, nq), 1e-9, f"run {run} env {e}")
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 4. constraint rows: joint limits, Coulomb friction, velocity follower
# ------------------------------------------------------------------------------------------------------------------
def _limited_tree(oracle, nq, topology, need):
    for seed in range(300, 400):
        xml, t, model = make_tree(oracle, nq, topology, seed)
        limited = [j for j in range(nq) if np.isfinite(t["lower"][j])]
        if len(limited) >= need:
            return xml, t, limited
    raise AssertionError("no tree with enough limited joints")


@pytest.mark.parametrize("n", [4093, 20001])
@pytest.mark.parametrize("variant", ["limits", "follower"])
@pytest.mark.parametrize("nq,topology", [(8, "random"), (13, "base_children")])
def test_random_rows_constraint_rows_match_oracle(nq, topology, variant, n, torch, oracle):
    """One step from states with 1-4 joints (lane-parallel / impulse stage where the warp is undamped) or 5-6 joints (the
    dense solve) exactly on a limit and driven into it, with the rows' Coulomb friction on half the envs, and optionally a
    velocity-follower joint; at the tolerances of test_constraint_rows_one_step_match_oracle."""
    xml, t, limited = _limited_tree(oracle, nq, topology, 6)
    epw = 32 // lane_group(nq)
    rng = np.random.default_rng([nq, n, len(variant)])
    q, dq = random_state(rng, t, n)
    tau = rng.uniform(-2, 2, (n, nq))
    rows = random_rows(rng, t, n)
    for e in range(n):
        w = e // epw
        k = 1 + e % 4 if w % 2 == 0 else 5 + e % 2
        js = rng.choice(limited, size=k, replace=False)
        for j, u in zip(js, rng.random(k) < 0.5):
            q[e, j] = t["upper"][j] if u else t["lower"][j]
            dq[e, j] = 0.3 if u else -0.3
            tau[e, j] = 5.0 if u else -5.0
    sim, mid = new_sim(torch, xml, n, q, dq)
    write_rows(torch, sim.enable_env_params(mid), rows)
    envs = sample_envs(n, nq) + [2 * epw, 2 * epw + 1, 3 * epw, 8 * epw, 9 * epw + 1]
    refs = {e: oracle_sim(oracle, env_model(oracle, t, rows, e), q[e], dq[e]) for e in envs}
    follower = limited[0] if variant == "follower" else -1
    vt = rng.uniform(-0.5, 0.5, n)
    for j in range(nq):
        mode = MODE_FOLLOWER if j == follower else MODE_FORCE
        sim.set_control_mode(mid, j, mode)
        for r in refs.values():
            r.set_control_mode(j, mode)
    if follower >= 0:
        sim.tensor(mid, BUF_VEL_T)[:, follower].copy_(torch.as_tensor(vt, device="cuda"))
        tau[:, follower] = 0.0
    sim.tensor(mid, BUF_FCMD).copy_(torch.as_tensor(tau, device="cuda"))
    sim.run()
    got = sim.tensor(mid, BUF_STATE).cpu().numpy()
    for e, r in refs.items():
        for j in range(nq):
            if j == follower:
                r.set_velocity_target(j, vt[e])
            else:
                r.set_force_target(j, tau[e, j])
        r.run(False)
        ref = oracle_state(r, nq)
        np.testing.assert_allclose(got[e, :nq], ref[:nq], rtol=1e-9, atol=1e-11, err_msg=f"env {e}")
        np.testing.assert_allclose(got[e, nq:], ref[nq:], rtol=1e-8, atol=1e-10, err_msg=f"env {e}")
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 5. the computed-torque controller keeps the nominal model
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4093, 20001])
@pytest.mark.parametrize("nq,topology", [(7, "base_children"), (12, "random")])
def test_computed_torque_uses_the_nominal_model(nq, topology, n, torch, oracle):
    """tau = M(q) (ddq_ref - kp e - kd de) + h(q, dq) from the NOMINAL oracle.Dynamics under the controller's gravity,
    applied in force mode to an oracle.Sim of the env's own tables, every physics step of 10 runs."""
    xml, t, _ = make_tree(oracle, nq, topology, seed=550 + nq)
    envs = sample_envs(n, nq)
    rng = np.random.default_rng([nq, n])
    q, dq = random_state(rng, t, n)
    rows = random_rows(rng, t, n)
    sim, mid = new_sim(torch, xml, n, q, dq)
    write_rows(torch, sim.enable_env_params(mid), rows)
    ct_g = (0.0, 0.0, -9.80665)
    tn = copy.deepcopy(t)
    tn["gravity"] = np.array(ct_g)
    D = oracle.Dynamics(oracle.model_from_tables(tn))
    kp, kd = np.full(nq, 30.0), np.full(nq, 4.0)
    qt, vt, at = q + rng.uniform(-0.1, 0.1, (n, nq)), rng.uniform(-0.2, 0.2, (n, nq)), rng.uniform(-0.5, 0.5, (n, nq))
    sim.set_controller_period(mid, 0.001)
    sim.set_computed_torque(mid, kp, kd, ct_g)
    for j in range(nq):
        for f in (F_PT, F_VT, F_AT):
            sim.set_joint(mid, f, -1, j, 0.0)
    for buf, v in ((BUF_POS_T, qt), (BUF_VEL_T, vt), (BUF_ACC_T, at)):
        sim.tensor(mid, buf).copy_(torch.as_tensor(v, device="cuda"))
    refs = {e: oracle_sim(oracle, env_model(oracle, t, rows, e), q[e], dq[e]) for e in envs}
    for r in refs.values():
        for j in range(nq):
            r.set_control_mode(j, MODE_FORCE)
    state = sim.tensor(mid, BUF_STATE)
    for run in range(10):
        sim.run()
        got = state.cpu().numpy()
        for e, r in refs.items():
            x = oracle_state(r, nq)
            qe, dqe = x[:nq], x[nq:]
            tau = D.mass_matrix(qe) @ (at[e] - kp * (qe - qt[e]) - kd * (dqe - vt[e])) + D.inverse_dynamics(qe, dqe, np.zeros(nq))
            for j in range(nq):
                r.set_force_target(j, tau[j])
            r.run(False)
            assert_state(got[e], oracle_state(r, nq), 1e-9, f"run {run} env {e}")
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 6. fp32
# ------------------------------------------------------------------------------------------------------------------
def _fp32_tolerance(D, q, dq, ddq, nq):
    """The bound of test_generated_trees_gpu._fp32_tolerance (u = 2^-24, 50 covers the constants of the recursions)."""
    u = 2.0 ** -24
    k = np.linalg.cond(D.mass_matrix(q))
    err_ddq = 50 * nq * u * k * (1.0 + np.abs(ddq).max())
    tol_dq = 50 * u * (1.0 + np.abs(dq).max()) + 1e-3 * err_ddq
    tol_q = 50 * u * (1.0 + np.abs(q).max()) + 1e-3 * tol_dq
    return tol_q, tol_dq


@pytest.mark.parametrize("n", [4093, 20001])
@pytest.mark.parametrize("nq,topology", [(6, "random"), (15, "random")])
def test_fp32_random_rows_one_step_against_the_fp64_oracle(nq, topology, n, torch, oracle):
    """dtype float32 with fp32 rows, one step from the device's own fp32 state, against the fp64 oracle built from the same
    (exactly converted) rows, within the derived rounding bound."""
    xml, t, _ = make_tree(oracle, nq, topology, seed=800 + nq)
    rng = np.random.default_rng([nq, n])
    q, dq = random_state(rng, t, n)
    f32 = lambda a: a.astype(np.float32).astype(np.float64)
    q, dq = f32(q), f32(dq)
    tau = f32(rng.uniform(-2, 2, (n, nq)))
    rows = random_rows(rng, t, n)
    rows[1][..., 1] = 0.0   # smooth dynamics: the bound is for the unconstrained step
    rows = tuple(f32(r) for r in rows)
    sim, mid = new_sim(torch, xml, n, q.astype(np.float32), dq.astype(np.float32), dtype="float32")
    write_rows(torch, sim.enable_env_params(mid), rows, np.float32)
    for j in range(nq):
        sim.set_control_mode(mid, j, MODE_FORCE)
    sim.tensor(mid, BUF_FCMD).copy_(torch.as_tensor(tau.astype(np.float32), device="cuda"))
    sim.run()
    got = sim.tensor(mid, BUF_STATE).cpu().numpy().astype(np.float64)
    for e in sample_envs(n, nq):
        model = env_model(oracle, t, rows, e)
        D = oracle.Dynamics(model)
        r = oracle_sim(oracle, model, q[e], dq[e])
        for j in range(nq):
            r.set_control_mode(j, MODE_FORCE); r.set_force_target(j, tau[e, j])
        r.run(False)
        ref = oracle_state(r, nq)
        tol_q, tol_dq = _fp32_tolerance(D, q[e], dq[e], D.forward_dynamics(q[e], dq[e], tau[e], 1e-3), nq)
        np.testing.assert_allclose(got[e, :nq], ref[:nq], rtol=0, atol=tol_q, err_msg=f"env {e}")
        np.testing.assert_allclose(got[e, nq:], ref[nq:], rtol=0, atol=tol_dq, err_msg=f"env {e}")
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 7. semantics of the rows
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", RUN_SIZES)
def test_a_row_written_between_runs_changes_only_its_env(n, torch, oracle):
    """Two simulators from the same states and rows; between runs one of them gets a heavier body, more damping and a
    tilted gravity in one env. The first run is bit-identical everywhere, the second differs in that env only (its
    neighbours included: they must not read its row)."""
    nq = 10
    xml, t, _ = make_tree(oracle, nq, "random", seed=1000)
    rng = np.random.default_rng(n)
    q, dq = random_state(rng, t, n)
    rows = random_rows(rng, t, n)
    sims = [new_sim(torch, xml, n, q, dq) for _ in range(2)]
    views = []
    for sim, mid in sims:
        views.append(sim.enable_env_params(mid))
        write_rows(torch, views[-1], rows)
        for j in range(nq):
            sim.set_control_mode(mid, j, MODE_FORCE)
    tau = torch.as_tensor(rng.uniform(-2, 2, (n, nq)), device="cuda")
    k = sample_envs(n, nq)[len(sample_envs(n, nq)) // 2]
    states = []
    for run in range(2):
        if run == 1:
            inertia, dyn, g = views[1]
            inertia[k, :, 0] *= 1.5
            dyn[k, :, 0] += 0.2
            g[k] = torch.as_tensor([2.0, -1.0, -9.5], device="cuda")
        for sim, mid in sims:
            sim.tensor(mid, BUF_FCMD).copy_(tau)
            sim.run()
        states.append([sim.tensor(mid, BUF_STATE).cpu().numpy() for sim, mid in sims])
    assert np.array_equal(states[0][0], states[0][1])
    a, b = states[1]
    differ = np.nonzero((a != b).any(axis=1))[0]
    assert list(differ) == [k]
    for sim, _ in sims:
        sim.close()


@pytest.mark.parametrize("n", [4093, 65537])
def test_every_env_setters_update_every_row_and_disabling_restores_the_tables(n, torch, oracle):
    """set_gravity and the joint friction setter keep their every-env meaning while the feature is on: every row takes the
    new value and the runs match a feature-off simulator with the same edits. enable_env_params(False) returns None, the
    buffers are unset again, and runs from equal states are bit-identical to the feature-off simulator."""
    import b2sim
    from b2sim import _lib
    nq = 6
    xml, t, _ = make_tree(oracle, nq, "random", seed=1100)
    rng = np.random.default_rng(n)
    q, dq = random_state(rng, t, n)
    sims = [new_sim(torch, xml, n, q, dq) for _ in range(2)]
    sim_on, mid_on = sims[1]
    inertia, dyn, g = sim_on.enable_env_params(mid_on)
    write_rows(torch, (inertia, dyn, g), random_rows(rng, t, n))
    for sim, mid in sims:
        sim.set_gravity([0.5, -0.3, -9.6])
        for j in (1, 4):
            assert sim.lib.b2sim_set_joint_friction(sim.handle, mid, j, 0.02 * j, 0.1 * j) == 0
        for j in range(nq):
            sim.set_control_mode(mid, j, MODE_FORCE)
    assert np.array_equal(g.cpu().numpy(), np.tile([0.5, -0.3, -9.6], (n, 1)))
    for j in (1, 4):
        assert np.array_equal(dyn[:, j].cpu().numpy(), np.tile([0.1 * j, 0.02 * j], (n, 1)))
    inertia.copy_(torch.as_tensor(np.tile(np.concatenate(
        [t["mass"][:nq, None], t["com"][:nq], np.stack([t["Ic"][:nq, i, j] for i, j in SYM], -1)], -1), (n, 1, 1)), device="cuda"))
    dyn.copy_(torch.as_tensor(np.tile(np.stack([t["damping"][:nq], t["friction"][:nq]], -1), (n, 1, 1)), device="cuda"))
    dyn[:, [1, 4]] = torch.as_tensor([[0.1, 0.02], [0.4, 0.08]], dtype=torch.float64, device="cuda")
    for run in range(5):
        tau = torch.as_tensor(rng.uniform(-2, 2, (n, nq)), device="cuda")
        for sim, mid in sims:
            sim.tensor(mid, BUF_FCMD).copy_(tau)
            sim.run()
    a, b = (sim.tensor(mid, BUF_STATE).cpu().numpy() for sim, mid in sims)
    np.testing.assert_allclose(b, a, rtol=1e-12, atol=1e-12 * max(1.0, np.abs(a).max()))
    assert sim_on.enable_env_params(mid_on, False) is None
    for which in (_lib.BUF_BODY_INERTIA, _lib.BUF_JOINT_DYNAMICS, _lib.BUF_GRAVITY):
        with pytest.raises(b2sim.B2Error) as err:
            sim_on.buffer(mid_on, which)
        assert err.value.code == _lib.ERR_UNSET
    sim_on.tensor(mid_on, BUF_STATE).copy_(sims[0][0].tensor(sims[0][1], BUF_STATE))
    for run in range(3):
        tau = torch.as_tensor(rng.uniform(-2, 2, (n, nq)), device="cuda")
        for sim, mid in sims:
            sim.tensor(mid, BUF_FCMD).copy_(tau)
            sim.run()
    assert torch.equal(*(sim.tensor(mid, BUF_STATE) for sim, mid in sims))
    for sim, _ in sims:
        sim.close()


def test_kindyn_queries_stay_nominal(torch, oracle):
    """KinDynComputations is built from the model file: with random rows the KinDyn outputs equal the feature-off ones
    bit for bit and the nominal oracle."""
    nq, n = 9, 257
    xml, t, model = make_tree(oracle, nq, "random", seed=1200)
    D = oracle.Dynamics(model)
    rng = np.random.default_rng(3)
    q, dq = random_state(rng, t, n)
    sims = [new_sim(torch, xml, n, q, dq) for _ in range(2)]
    write_rows(torch, sims[1][0].enable_env_params(sims[1][1]), random_rows(rng, t, n))
    f64 = dict(dtype=torch.float64, device="cuda")
    outs = []
    for sim, mid in sims:
        M, h, J = torch.empty((n, nq * nq), **f64), torch.empty((n, nq), **f64), torch.empty((n, 6 * nq), **f64)
        sim.kindyn(mid, nq - 1, M, h, J)
        com, vel, mom, cJ = (torch.empty((n, k), **f64) for k in (3, 3, 12, 3 * nq))
        sim.centroidal(mid, com, vel, mom, cJ)
        mJ, locked = torch.empty((n, 6 * nq), **f64), torch.empty((n, 10), **f64)
        sim.momentum_jacobian(mid, mJ, locked)
        sim.update_kinematics(mid)
        outs.append([M, h, J, com, vel, mom, cJ, mJ, locked, sim.tensor(mid, BUF_LINK_POSE).clone()])
    for x, y in zip(*outs):
        assert torch.equal(x, y)
    M, h = outs[1][0].cpu().numpy(), outs[1][1].cpu().numpy()
    for e in (0, n // 2, n - 1):
        np.testing.assert_allclose(M[e].reshape(nq, nq), D.mass_matrix(q[e]), rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(h[e], D.inverse_dynamics(q[e], dq[e], np.zeros(nq)), rtol=1e-10, atol=1e-11)
    for sim, _ in sims:
        sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 8. refusals
# ------------------------------------------------------------------------------------------------------------------
CUBE_URDF = """<robot name="cube"><link name="cube"><inertial><origin xyz="0 0 0"/><mass value="1.0"/>
<inertia ixx="0.01" ixy="0" ixz="0" iyy="0.01" iyz="0" izz="0.01"/></inertial>
<collision><geometry><box size="0.1 0.1 0.1"/></geometry></collision></link></robot>"""


def test_refusals(torch, oracle, model_files):
    """B2_ERR_UNSUPPORTED for a static model, a free-floating model, a model with a fused task (either order) and a world
    with free bodies, at enable time and at the first run after a free body was inserted."""
    import b2sim
    from b2sim import _lib

    def refused(fn, *a):
        with pytest.raises(b2sim.B2Error) as err:
            fn(*a)
        assert err.value.code == _lib.ERR_UNSUPPORTED

    xml, t, _ = make_tree(oracle, 5, "random", seed=1300)
    sim = b2sim.Simulator(64, 0.001, 1)
    ground = sim.insert_model_file(model_files["ground_plane"])
    refused(sim.enable_env_params, ground)
    arm = sim.insert_model(xml, pose=POSE)
    assert sim.enable_env_params(arm) is not None
    sim.run()
    cube = sim.insert_model(CUBE_URDF, pose=(0, 0, 1.0, 1, 0, 0, 0), name="cube")
    refused(sim.enable_env_params, cube)
    refused(sim.run)
    sim.remove_model(cube)
    sim.run()
    cube = sim.insert_model(CUBE_URDF, pose=(0, 0, 1.0, 1, 0, 0, 0), name="cube2")
    sim.enable_env_params(arm, False)
    refused(sim.enable_env_params, arm)
    sim.close()

    with open(model_files["pendulum"]) as f:
        pend = f.read()
    sim = b2sim.Simulator(64, 0.001, 1)
    mid = sim.insert_model(pend)
    sim.enable_env_params(mid)
    refused(sim.set_task, mid, 1)
    sim.enable_env_params(mid, False)
    sim.set_task(mid, 1)
    refused(sim.enable_env_params, mid)
    sim.close()
