"""Every tree kernel on generated kinematic trees of 3-16 joints (tests/helpers/tree_urdf.py) against the oracle.

The kernels are reached through the batch-size selection the engine makes (no environment switches):

    run path      k_run_tree_lanes<G>  n <= 16,384 and >= 4 joints (G = 8 / 10 / 16 lanes per env by joint count; 2 warps
                                       per block and no programmatic dependent launch up to 8,192 envs, 4 warps above)
                  k_run_tree           n = 20,001, or fewer than 4 joints (scratch in shared memory)
                  k_run_tree_local     n >= 65,536 (scratch in local memory)
    reach task    k_task_panda_lanes   n <= 32,768 (the Panda's exact body structure is a compile-time specialisation)
                  k_task_panda         n = 32,769

Batch sizes leave the last warp partial for every G (G = 8: n % 4 != 0, G = 10: n % 3 != 0, G = 16: n odd). Every env has
its own random state and commands, so a lane that reads another env's strip or slot shows up; the sampled envs are the
first warp, a warp in the middle of a block and the partial tail warp, each against one oracle.Sim.
"""
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
BUF_STATE, BUF_ACC, BUF_FCMD, BUF_POS_T, BUF_VEL_T, BUF_PID, BUF_OBS, BUF_REWARD, BUF_DONE, BUF_LINK_POSE = 0, 1, 2, 3, 4, 5, 8, 9, 10, 13
TASK_PANDA_REACH = 5
# a translated and rotated base: world placements carry the base pose
POSE = (0.1, -0.2, 0.3, 0.9238795325112867, 0.0, 0.3826834323650898, 0.0)
GAINS = (20.0, 0.5, 1.0)


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def make_tree(oracle, nq, topology, seed, **kw):
    xml = tree_urdf.generate(nq, topology, seed=seed, **kw)
    t, model = oracle.load_urdf(xml, base_position=POSE[:3], base_orientation_wxyz=POSE[3:])
    return xml, t, model


def lane_group(nq):
    return 8 if nq <= 8 else (10 if nq <= 10 else 16)


def sample_envs(n, nq):
    """The first warp, the second warp of a block in the middle of the batch and the (partial) tail warp of the lane
    kernels with `nq` joints."""
    epw = 32 // lane_group(nq)
    per_block = (2 if n <= 8192 else 4) * epw
    b = (n // per_block) // 2
    tail = (n - 1) // epw * epw
    envs = set(range(epw)) | set(range(b * per_block + epw, b * per_block + 2 * epw)) | set(range(tail, n))
    return sorted(e for e in envs if e < n)


def random_state(rng, t, n):
    nq = int(t["nb"])
    prism = t["jtype"][:nq] == 2
    q = rng.uniform(-1.5, 1.5, (n, nq))
    q[:, prism] = rng.uniform(-0.2, 0.2, (n, int(prism.sum())))
    return q, rng.uniform(-1.0, 1.0, (n, nq))


def new_sim(torch, xml, n, q, dq, steps_per_run=1, dtype="float64"):
    import b2sim
    sim = b2sim.Simulator(n, 0.001, steps_per_run, dtype)
    mid = sim.insert_model(xml, pose=POSE)
    sim.tensor(mid, BUF_STATE).copy_(torch.as_tensor(np.hstack([q, dq]), device="cuda"))
    return sim, mid


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


def link_world(t, D, q, link):
    """World pose (R, p) of `link` from the oracle's forward kinematics."""
    b = int(t["link_body"][link])
    if b < 0:
        return t["base_R"] @ t["link_R"][link], t["base_p"] + t["base_R"] @ t["link_p"][link]
    Rw, pw = D.forward_kinematics(q)
    return Rw[b] @ t["link_R"][link], pw[b] + Rw[b] @ t["link_p"][link]


def quat_R(q):
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def side_branch_link(t):
    """A link of a body off the path from the base to body 0 whose parent is not the previous body, if there is one."""
    nq = int(t["nb"])
    par = t["parent"][:nq]
    cands = [i for i in range(nq) if par[i] >= 0 and par[i] != i - 1] or [nq - 1]
    b = cands[-1]
    return next(l for l in range(len(t["link_body"])) if t["link_body"][l] == b)


def welded_links(t):
    """(a link welded to a moving body other than its body's own link, a link welded to the base)."""
    names = t["link_names"]
    body = next((l for l, nm in enumerate(names) if nm.startswith("tool")), None)
    base = next((l for l, nm in enumerate(names) if t["link_body"][l] < 0), None)
    return body, base


# ------------------------------------------------------------------------------------------------------------------
# 1. KinDyn queries
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nq,topology", [(3, "star"), (6, "base_children"), (9, "random"), (10, "random"), (13, "base_children"),
                                         (16, "random")])
def test_kindyn_queries_match_oracle(nq, topology, torch, oracle):
    import b2sim
    xml, t, model = make_tree(oracle, nq, topology, seed=100 + nq)
    D = oracle.Dynamics(model)
    n = 131
    rng = np.random.default_rng(nq)
    q, dq = random_state(rng, t, n)
    ddq = rng.uniform(-2, 2, (n, nq))
    sim, mid = new_sim(torch, xml, n, q, dq)
    sim.tensor(mid, BUF_ACC).copy_(torch.as_tensor(ddq, device="cuda"))
    tool, plate = welded_links(t)
    side = side_branch_link(t)
    envs = [0, 1, 2, 3, 64, 65, n - 2, n - 1]
    sim.update_kinematics(mid)
    poses = sim.tensor(mid, BUF_LINK_POSE).cpu().numpy().reshape(n, -1, 7)
    f64 = dict(dtype=torch.float64, device="cuda")
    com, vel, mom, cJ = (torch.empty((n, k), **f64) for k in (3, 3, 12, 3 * nq))
    sim.centroidal(mid, com, vel, mom, cJ)
    mJ, locked = torch.empty((n, 6 * nq), **f64), torch.empty((n, 10), **f64)
    sim.momentum_jacobian(mid, mJ, locked)
    cen = [x.cpu().numpy() for x in (com, vel, mom, cJ, mJ, locked)]
    for link in (side, tool):
        M, h, J = torch.empty((n, nq * nq), **f64), torch.empty((n, nq), **f64), torch.empty((n, 6 * nq), **f64)
        sim.kindyn(mid, link, M, h, J)
        tw, ac = torch.empty((n, 6), **f64), torch.empty((n, 6), **f64)
        sim.link_motion(mid, link, tw, ac)
        M, h, J, tw, ac = (x.cpu().numpy() for x in (M, h, J, tw, ac))
        b, lp = int(t["link_body"][link]), t["link_p"][link]
        for e in envs:
            msg = f"env {e} link {t['link_names'][link]}"
            np.testing.assert_allclose(M[e].reshape(nq, nq), D.mass_matrix(q[e]), rtol=1e-10, atol=1e-12, err_msg=msg)
            np.testing.assert_allclose(h[e], D.inverse_dynamics(q[e], dq[e], np.zeros(nq)), rtol=1e-10, atol=1e-11, err_msg=msg)
            np.testing.assert_allclose(J[e].reshape(6, nq), D.point_jacobian(q[e], b, lp), rtol=1e-10, atol=1e-12, err_msg=msg)
            ref = D.link_motion(q[e], dq[e], ddq[e], b, lp)
            np.testing.assert_allclose(tw[e], np.r_[ref[0], ref[1]], rtol=1e-10, atol=1e-11, err_msg=msg)
            np.testing.assert_allclose(ac[e], np.r_[ref[2], ref[3]], rtol=1e-10, atol=1e-10, err_msg=msg)
    for e in envs:
        for l in range(len(t["link_names"])):
            R, p = link_world(t, D, q[e], l)
            np.testing.assert_allclose(poses[e, l, :3], p, rtol=1e-10, atol=1e-12, err_msg=f"env {e} link {l}")
            np.testing.assert_allclose(quat_R(poses[e, l, 3:]), R, atol=1e-10, err_msg=f"env {e} link {l}")
        rc, rv, rm, rg, rJ = D.centroidal(q[e], dq[e], t["base_mass"], t["base_mc"])
        np.testing.assert_allclose(cen[0][e], rc, rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(cen[1][e], rv, rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(cen[2][e], np.r_[rm, rg], rtol=1e-10, atol=1e-11)
        np.testing.assert_allclose(cen[3][e].reshape(3, nq), rJ, rtol=1e-10, atol=1e-12)
        rJm, rl = D.momentum_jacobian(q[e], t["base_mass"], t["base_mc"], t["base_Io"])
        np.testing.assert_allclose(cen[4][e].reshape(6, nq), rJm, rtol=1e-10, atol=1e-11)
        np.testing.assert_allclose(cen[5][e], rl, rtol=1e-10, atol=1e-11)
    assert plate is not None and int(t["link_body"][plate]) < 0
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 2. run path, force mode
# ------------------------------------------------------------------------------------------------------------------
RUN_TREES = [(3, "chain"), (4, "star"), (5, "base_children"), (8, "random"), (9, "random"), (10, "base_children"),
             (11, "random"), (16, "random")]
# lanes with 2 warps per block, lanes with 4 warps and programmatic dependent launch, k_run_tree, k_run_tree_local
RUN_SIZES = [8191, 16381, 20001, 65537]


@pytest.mark.parametrize("n", RUN_SIZES)
@pytest.mark.parametrize("nq,topology", RUN_TREES)
def test_run_force_mode_matches_oracle(nq, topology, n, torch, oracle):
    """One run from identical states at 1e-9 of the state scale, then 20 consecutive runs at 1e-8, with one and three
    physics steps per run; per-env random torques every run."""
    xml, t, model = make_tree(oracle, nq, topology, seed=200 + nq)
    if nq == 9:
        assert list(t["parent"][:9]) != [-1, 0, 1, 2, 3, 4, 5, 6, 6]   # not the Panda's specialised structure
    envs = sample_envs(n, nq)
    for spr in (1, 3):
        rng = np.random.default_rng([nq, n, spr])
        q, dq = random_state(rng, t, n)
        sim, mid = new_sim(torch, xml, n, q, dq, spr)
        refs = {e: oracle_sim(oracle, model, q[e], dq[e], spr) for e in envs}
        for j in range(nq):
            sim.set_control_mode(mid, j, MODE_FORCE)
            for r in refs.values():
                r.set_control_mode(j, MODE_FORCE)
        state, fcmd = sim.tensor(mid, BUF_STATE), sim.tensor(mid, BUF_FCMD)
        for run in range(20):
            tau = rng.uniform(-2, 2, (n, nq))
            fcmd.copy_(torch.as_tensor(tau, device="cuda"))
            sim.run()
            for e, r in refs.items():
                for j in range(nq):
                    r.set_force_target(j, tau[e, j])
                r.run(False)
            if run in (0, 19):
                got = state.cpu().numpy()
                for e, r in refs.items():
                    assert_state(got[e], oracle_state(r, nq), 1e-9 if run == 0 else 1e-8, f"spr {spr} run {run} env {e}")
        sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 3. constraint rows
# ------------------------------------------------------------------------------------------------------------------
def _limited_tree(oracle, nq, topology, need, **kw):
    for seed in range(300, 400):
        xml, t, model = make_tree(oracle, nq, topology, seed, **kw)
        limited = [j for j in range(nq) if np.isfinite(t["lower"][j])]
        if len(limited) >= need:
            return xml, t, model, limited
    raise AssertionError("no tree with enough limited joints")


@pytest.mark.parametrize("variant", ["limits", "friction", "follower", "damped"])
@pytest.mark.parametrize("nq,topology", [(8, "random"), (13, "base_children")])
def test_constraint_rows_one_step_match_oracle(nq, topology, variant, torch, oracle):
    """One step from states in which joints sit exactly on a limit, moving and driven into it. By warp: every env with 1-4
    such joints (the lane-parallel stage, lanes_constraints_fast), every env with 5-6 (the dense solve on lane 0), and a
    warp mixing both. Variants add Coulomb friction on every joint, a velocity-follower joint, or joint damping (dense path
    for the whole warp). Against the oracle's dense boxed LCP, at the tolerances of
    test_panda_task_limit_rows_one_step_matches_oracle."""
    kw = dict(friction=0.05) if variant == "friction" else (dict(damping=0.3) if variant == "damped" else {})
    xml, t, model, limited = _limited_tree(oracle, nq, topology, 6, **kw)
    n = 4093
    epw = 32 // lane_group(nq)
    rng = np.random.default_rng([nq, len(variant)])
    q, dq = random_state(rng, t, n)
    tau = rng.uniform(-2, 2, (n, nq))
    on_limit = []
    for e in range(n):
        w, slot = divmod(e, epw)
        k = (1 + e % 4) if w % 3 == 0 else (5 + e % 2 if w % 3 == 1 else (5 if slot == 0 else 1 + e % 4))
        js = rng.choice(limited, size=k, replace=False)
        up = rng.random(k) < 0.5
        for j, u in zip(js, up):
            q[e, j] = t["upper"][j] if u else t["lower"][j]
            dq[e, j] = 0.3 if u else -0.3
            tau[e, j] = 5.0 if u else -5.0
        on_limit.append((js, up))
    sim, mid = new_sim(torch, xml, n, q, dq)
    envs = sample_envs(n, nq) + [3 * epw, 3 * epw + 1, 4 * epw, 5 * epw, 5 * epw + 1]
    refs = {e: oracle_sim(oracle, model, q[e], dq[e]) for e in envs}
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
    if variant == "limits":   # the rows acted: no joint on a limit moves further into it
        for e in envs:
            for j, u in zip(*on_limit[e]):
                assert (got[e, nq + j] <= 1e-9) if u else (got[e, nq + j] >= -1e-9), (e, j)
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 4. controllers
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("controller", ["pid1", "pid3", "computed_torque"])
@pytest.mark.parametrize("nq,topology", [(7, "base_children"), (14, "random")])
def test_controllers_match_oracle(nq, topology, controller, torch, oracle):
    """Position PIDs with a controller period of 1 and 3 physics steps, and the computed-torque controller
    (k_run_tree_lanes<CT>), per-env targets, 20 runs of 2 physics steps against oracle.Sim."""
    xml, t, model = make_tree(oracle, nq, topology, seed=500 + nq)
    n = 4093 if nq <= 8 else 4095
    envs = sample_envs(n, nq)
    rng = np.random.default_rng([nq, len(controller)])
    q, dq = random_state(rng, t, n)
    sim, mid = new_sim(torch, xml, n, q, dq, 2)
    refs = {e: oracle_sim(oracle, model, q[e], dq[e], 2) for e in envs}
    qt = q + rng.uniform(-0.1, 0.1, (n, nq))
    if controller == "computed_torque":
        kp, kd = [30.0] * nq, [4.0] * nq
        vt, at = rng.uniform(-0.2, 0.2, (n, nq)), rng.uniform(-0.5, 0.5, (n, nq))
        sim.set_controller_period(mid, 0.001)
        sim.set_computed_torque(mid, kp, kd)
        for j in range(nq):
            for f in (F_PT, F_VT, F_AT):
                sim.set_joint(mid, f, -1, j, 0.0)
        for buf, v in ((BUF_POS_T, qt), (BUF_VEL_T, vt), (16, at)):
            sim.tensor(mid, buf).copy_(torch.as_tensor(v, device="cuda"))
        for e, r in refs.items():
            r.set_controller_period(0.001)
            r.load_computed_torque(kp, kd)
            for j in range(nq):
                r.set_position_target(j, qt[e, j]); r.set_velocity_target(j, vt[e, j]); r.set_acceleration_target(j, at[e, j])
    else:
        period = 0.001 if controller == "pid1" else 0.003
        sim.set_controller_period(mid, period)
        for j in range(nq):
            sim.set_pid(mid, j, *GAINS, DBL_MAX, -DBL_MAX, DBL_MAX, -DBL_MAX, 0.0)
            sim.set_control_mode(mid, j, MODE_POSITION)
        sim.tensor(mid, BUF_POS_T).copy_(torch.as_tensor(qt, device="cuda"))
        for e, r in refs.items():
            r.set_controller_period(period)
            for j in range(nq):
                r.set_pid(j, *GAINS, DBL_MAX, -DBL_MAX, DBL_MAX, -DBL_MAX, 0.0)
                r.set_control_mode(j, MODE_POSITION)
                r.set_position_target(j, qt[e, j])
    state = sim.tensor(mid, BUF_STATE)
    for run in range(20):
        sim.run()
        for r in refs.values():
            r.run(False)
    got = state.cpu().numpy()
    for e, r in refs.items():
        assert_state(got[e], oracle_state(r, nq), 1e-8, f"env {e}")
    moved = np.abs(got[:, :nq] - q).max()
    assert moved > 1e-3
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 5. external link wrenches
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4093, 20001])
@pytest.mark.parametrize("nq,topology", [(6, "random"), (12, "base_children")])
def test_link_wrenches_match_oracle(nq, topology, n, torch, oracle):
    """Link::applyWorldWrench on a link of a side branch (every env), on a link welded to a moving body (one env only), on a
    link welded to the base (a no-op) and one that expires after 7.5 ms of the 20 runs."""
    xml, t, model = make_tree(oracle, nq, topology, seed=600 + nq)
    envs = sample_envs(n, nq)
    rng = np.random.default_rng([nq, n])
    q, dq = random_state(rng, t, n)
    sim, mid = new_sim(torch, xml, n, q, dq)
    refs = {e: oracle_sim(oracle, model, q[e], dq[e]) for e in envs}
    for j in range(nq):
        sim.set_control_mode(mid, j, MODE_FORCE)
        for r in refs.values():
            r.set_control_mode(j, MODE_FORCE)
    tool, plate = welded_links(t)
    side = side_branch_link(t)
    one_env = envs[len(envs) // 2]
    wrenches = [(side, -1, [3.0, -2.0, 1.0, 0.2, 0.1, -0.3], 1.0), (tool, one_env, [-1.0, 2.0, 4.0, 0.0, 0.3, 0.1], 1.0),
                (plate, -1, [50.0, 50.0, 50.0, 5.0, 5.0, 5.0], 1.0), (tool, -1, [0.0, 0.0, 5.0, 0.1, 0.0, 0.0], 0.0075)]
    for link, env, w, dur in wrenches:
        sim.apply_link_wrench(mid, env, link, w, dur)
        b = int(t["link_body"][link])
        for e, r in refs.items():
            if b >= 0 and env in (-1, e):
                r.apply_link_wrench(b, t["link_p"][link], w, dur)
    state = sim.tensor(mid, BUF_STATE)
    for run in range(20):
        sim.run()
        for r in refs.values():
            r.run(False)
    got = state.cpu().numpy()
    for e, r in refs.items():
        assert_state(got[e], oracle_state(r, nq), 1e-8, f"env {e}")
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 6. reach task on generic trees
# ------------------------------------------------------------------------------------------------------------------
def _reach_case(oracle, case):
    if case == "g8":
        xml, t, model = make_tree(oracle, 5, "random", seed=701)
        ee = side_branch_link(t)
    elif case == "g10":
        xml, t, model = make_tree(oracle, 9, "random", seed=702)
        assert list(t["parent"][:9]) != [-1, 0, 1, 2, 3, 4, 5, 6, 6]
        ee = welded_links(t)[0]
    elif case == "panda":
        xml, t, model = make_tree(oracle, 9, "panda", seed=703)
        assert list(t["parent"][:9]) == [-1, 0, 1, 2, 3, 4, 5, 6, 6] and list(t["jtype"][:9]) == [1] * 7 + [2] * 2
        ee = next(l for l in range(len(t["link_names"])) if t["link_body"][l] == 8)   # a finger body
    else:   # the model's last link is welded to the base: the default end effector (no end_effector_frame)
        xml, t, model = make_tree(oracle, 6, "base_children", seed=704, last_link_on_world=True)
        ee = -1
    return xml, t, model, ee


@pytest.mark.parametrize("case", ["g8", "g10", "panda", "base_welded"])
def test_reach_task_on_generic_trees_matches_oracle(case, torch, oracle):
    """TASK_PANDA_REACH on a 5-joint tree (k_task_panda_lanes<T, 8, 0>), a 9-joint non-Panda tree (<T, 10, 0>), the Panda's
    body structure with random axes and constants and the end effector on a finger body (the compile-time specialisation
    must assume only the structure), and a model whose default end effector is welded to the base. Lane kernel (4,095 or
    32,767 envs) and thread kernel (32,769 envs) from the same per-env states and targets: observation (q, dq, end-effector
    position and orientation, MIXED Jacobian), reward and the TimeLimit reset against the oracle, and the two kernels
    against each other."""
    import b2sim
    xml, t, model, ee = _reach_case(oracle, case)
    D = oracle.Dynamics(model)
    nq = int(t["nb"])
    ee_link = ee if ee >= 0 else len(t["link_names"]) - 1
    body, lp = int(t["link_body"][ee_link]), t["link_p"][ee_link]
    assert (body < 0) == (case == "base_welded")
    goal = np.array([0.3, -0.1, 0.6])
    rng = np.random.default_rng(len(case))
    q0 = rng.uniform(-0.3, 0.3, nq)
    n_lanes = 4095 if case in ("g8", "panda") else 32767
    sizes = (n_lanes, 32769)
    q, dq = random_state(rng, t, sizes[1])
    T, limit = 7, 5
    targets = q[None] + rng.uniform(-0.2, 0.2, (T, sizes[1], nq))
    obs_all = {}
    for n in sizes:
        sim = b2sim.Simulator(n, 0.001, 1)
        mid = sim.insert_model(xml, pose=POSE)
        sim.set_task(mid, TASK_PANDA_REACH, max_episode_steps=limit)
        sim.set_task_params(mid, goal, q0, ee)
        for j in range(nq):
            sim.set_pid(mid, j, *GAINS, DBL_MAX, -DBL_MAX, DBL_MAX, -DBL_MAX, 0.0)
        sim.task_reset_all(mid)
        sim.tensor(mid, BUF_STATE).copy_(torch.as_tensor(np.hstack([q[:n], dq[:n]]), device="cuda"))
        envs = sample_envs(n, nq)
        refs = {}

        def fresh(e, qe, dqe):
            r = oracle_sim(oracle, model, qe, dqe)
            r.set_controller_period(0.001)
            for j in range(nq):
                r.set_pid(j, *GAINS, DBL_MAX, -DBL_MAX, DBL_MAX, -DBL_MAX, 0.0)
                r.set_control_mode(j, MODE_POSITION)
            return r

        refs = {e: fresh(e, q[e], dq[e]) for e in envs}
        obs_steps = []
        for step in range(T):
            act = torch.as_tensor(targets[step, :n], device="cuda")
            sim.task_step(mid, act.data_ptr())
            obs = sim.tensor(mid, BUF_OBS).cpu().numpy()
            rew = sim.tensor(mid, BUF_REWARD).cpu().numpy()
            done = sim.tensor(mid, BUF_DONE).cpu().numpy()
            obs_steps.append((obs, rew, done))
            assert done.sum() == (n if step == limit - 1 else 0)
            for e, r in refs.items():
                for j in range(nq):
                    r.set_position_target(j, targets[step, e, j])
                r.run(False)
                qe = np.array([r.position(j) for j in range(nq)]); dqe = np.array([r.velocity(j) for j in range(nq)])
                msg = f"n {n} step {step} env {e}"
                o = obs[e]
                np.testing.assert_allclose(o[:nq], qe, rtol=1e-8, atol=1e-10, err_msg=msg)
                np.testing.assert_allclose(o[nq:2 * nq], dqe, rtol=1e-7, atol=1e-9, err_msg=msg)
                R, pe = link_world(t, D, qe, ee_link)
                np.testing.assert_allclose(o[2 * nq:2 * nq + 3], pe, rtol=1e-8, atol=1e-10, err_msg=msg)
                np.testing.assert_allclose(quat_R(o[2 * nq + 3:2 * nq + 7]), R, atol=1e-9, err_msg=msg)
                J = o[2 * nq + 7:].reshape(6, 6 + nq)
                Jq = D.point_jacobian(qe, body, lp) if body >= 0 else np.zeros((6, nq))
                np.testing.assert_allclose(J[:, 6:], Jq, rtol=1e-7, atol=1e-9, err_msg=msg)
                r_ = pe - t["base_p"]
                S = np.array([[0, -r_[2], r_[1]], [r_[2], 0, -r_[0]], [-r_[1], r_[0], 0]])
                np.testing.assert_allclose(J[:, :6], np.block([[np.eye(3), -S], [np.zeros((3, 3)), np.eye(3)]]), atol=1e-9,
                                           err_msg=msg)
                assert rew[e] == pytest.approx(-np.linalg.norm(pe - goal), rel=1e-8), msg
            if step == limit - 1:   # TimeLimit: every env back to q0, PID state cleared
                np.testing.assert_allclose(sim.tensor(mid, BUF_STATE).cpu().numpy(), np.tile(np.r_[q0, np.zeros(nq)], (n, 1)))
                refs = {e: fresh(e, q0, np.zeros(nq)) for e in envs}
        obs_all[n] = obs_steps
        sim.close()
    m = sizes[0]
    for (o1, r1, d1), (o2, r2, d2) in zip(obs_all[sizes[0]], obs_all[sizes[1]]):
        np.testing.assert_allclose(o1, o2[:m], rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(r1, r2[:m], rtol=1e-10, atol=1e-12)
        assert np.array_equal(d1, d2[:m])


# ------------------------------------------------------------------------------------------------------------------
# 7. fp32
# ------------------------------------------------------------------------------------------------------------------
def _fp32_tolerance(D, q, dq, ddq, nq):
    """Bound on |fp32 step - fp64 step| from the same (fp32-representable) state, with u = 2^-24:
    the forward dynamics solves M ddq = tau - h in fp32, so the acceleration carries a relative error of about
    c(nq) u cond(M) (c(nq) ~ nq for the O(nq) recursions and the LDL^T); one step moves it into dq through dt, and q picks
    up dt times that plus its own rounding. The factor 50 covers the constants of the recursions (sums of up to 2 nq
    products per entry)."""
    u = 2.0 ** -24
    k = np.linalg.cond(D.mass_matrix(q))
    err_ddq = 50 * nq * u * k * (1.0 + np.abs(ddq).max())
    tol_dq = 50 * u * (1.0 + np.abs(dq).max()) + 1e-3 * err_ddq
    tol_q = 50 * u * (1.0 + np.abs(q).max()) + 1e-3 * tol_dq
    return tol_q, tol_dq


@pytest.mark.parametrize("nq,topology", [(6, "random"), (10, "base_children"), (15, "random")])
def test_fp32_run_one_step_against_the_fp64_oracle(nq, topology, torch, oracle):
    """dtype float32, k_run_tree_lanes<float, G>: one step per env from the device's own fp32 state converted exactly to
    fp64, against the fp64 oracle, within the bound of _fp32_tolerance."""
    xml, t, model = make_tree(oracle, nq, topology, seed=800 + nq)
    D = oracle.Dynamics(model)
    n = 4093 if nq <= 8 else 4095
    rng = np.random.default_rng(nq)
    q, dq = random_state(rng, t, n)
    q, dq = q.astype(np.float32).astype(np.float64), dq.astype(np.float32).astype(np.float64)
    tau = rng.uniform(-2, 2, (n, nq)).astype(np.float32).astype(np.float64)
    sim, mid = new_sim(torch, xml, n, q.astype(np.float32), dq.astype(np.float32), dtype="float32")
    for j in range(nq):
        sim.set_control_mode(mid, j, MODE_FORCE)
    sim.tensor(mid, BUF_FCMD).copy_(torch.as_tensor(tau.astype(np.float32), device="cuda"))
    sim.run()
    got = sim.tensor(mid, BUF_STATE).cpu().numpy().astype(np.float64)
    for e in sample_envs(n, nq):
        r = oracle_sim(oracle, model, q[e], dq[e])
        for j in range(nq):
            r.set_control_mode(j, MODE_FORCE); r.set_force_target(j, tau[e, j])
        r.run(False)
        ref = oracle_state(r, nq)
        tol_q, tol_dq = _fp32_tolerance(D, q[e], dq[e], D.forward_dynamics(q[e], dq[e], tau[e], 1e-3), nq)
        np.testing.assert_allclose(got[e, :nq], ref[:nq], rtol=0, atol=tol_q, err_msg=f"env {e}")
        np.testing.assert_allclose(got[e, nq:], ref[nq:], rtol=0, atol=tol_dq, err_msg=f"env {e}")
    sim.close()


@pytest.mark.parametrize("case", ["g8", "panda"])
def test_fp32_reach_one_step_against_the_fp64_oracle(case, torch, oracle):
    """dtype float32 reach task (lane kernel): one step from the device's own fp32 state, against the fp64 oracle;
    joint state within the bound of _fp32_tolerance (the PID torque adds one fp32 rounding of tau), end-effector position
    within the joint error propagated through the Jacobian."""
    import b2sim
    xml, t, model, ee = _reach_case(oracle, case)
    D = oracle.Dynamics(model)
    nq = int(t["nb"])
    body, lp = int(t["link_body"][ee]), t["link_p"][ee]
    n = 4095
    sim = b2sim.Simulator(n, 0.001, 1, "float32")
    mid = sim.insert_model(xml, pose=POSE)
    sim.set_task(mid, TASK_PANDA_REACH, max_episode_steps=100)
    sim.set_task_params(mid, [0.3, -0.1, 0.6], None, ee)
    for j in range(nq):
        sim.set_pid(mid, j, *GAINS, DBL_MAX, -DBL_MAX, DBL_MAX, -DBL_MAX, 0.0)
    rng = np.random.default_rng(9)
    q, dq = random_state(rng, t, n)
    q, dq = q.astype(np.float32).astype(np.float64), dq.astype(np.float32).astype(np.float64)
    targets = (q + rng.uniform(-0.2, 0.2, (n, nq))).astype(np.float32).astype(np.float64)
    sim.tensor(mid, BUF_STATE).copy_(torch.as_tensor(np.hstack([q, dq]).astype(np.float32), device="cuda"))
    sim.task_step(mid, torch.as_tensor(targets.astype(np.float32), device="cuda").data_ptr())
    obs = sim.tensor(mid, BUF_OBS).cpu().numpy().astype(np.float64)
    for e in sample_envs(n, nq):
        r = oracle_sim(oracle, model, q[e], dq[e])
        r.set_controller_period(0.001)
        for j in range(nq):
            r.set_pid(j, *GAINS, DBL_MAX, -DBL_MAX, DBL_MAX, -DBL_MAX, 0.0)
            r.set_control_mode(j, MODE_POSITION)
            r.set_position_target(j, targets[e, j])
        r.run(False)
        ref = oracle_state(r, nq)
        tau = GAINS[0] * (targets[e] - q[e]) - GAINS[2] * dq[e]
        tol_q, tol_dq = _fp32_tolerance(D, q[e], dq[e], D.forward_dynamics(q[e], dq[e], tau, 1e-3), nq)
        np.testing.assert_allclose(obs[e, :nq], ref[:nq], rtol=0, atol=tol_q, err_msg=f"env {e}")
        np.testing.assert_allclose(obs[e, nq:2 * nq], ref[nq:], rtol=0, atol=tol_dq, err_msg=f"env {e}")
        _, pe = link_world(t, D, ref[:nq], ee)
        tol_p = np.abs(D.point_jacobian(ref[:nq], body, lp)[:3]).sum(axis=1).max() * tol_q + 50 * 2.0 ** -24 * (1 + np.abs(pe).max())
        np.testing.assert_allclose(obs[e, 2 * nq:2 * nq + 3], pe, rtol=0, atol=tol_p, err_msg=f"env {e}")
    sim.close()


# ------------------------------------------------------------------------------------------------------------------
# 8. refusals
# ------------------------------------------------------------------------------------------------------------------
def test_reach_task_on_ten_or_more_joints_is_refused(torch, oracle):
    """The reach observation holds up to 9 joints: a 10- or 16-joint tree is refused with B2Error (unsupported) at the
    first step, on either kernel's batch size, and nothing is written."""
    import b2sim
    from b2sim import _lib
    for nq in (10, 16):
        xml, _, _ = make_tree(oracle, nq, "random", seed=900 + nq)
        for n in (64, 32769):
            sim = b2sim.Simulator(n, 0.001, 1)
            mid = sim.insert_model(xml, pose=POSE)
            sim.set_task(mid, TASK_PANDA_REACH)
            before = sim.tensor(mid, BUF_STATE).clone()
            act = torch.zeros((n, nq), dtype=torch.float64, device="cuda")
            with pytest.raises(b2sim.B2Error) as err:
                sim.task_step(mid, act.data_ptr())
            assert err.value.code == _lib.ERR_UNSUPPORTED
            assert torch.equal(sim.tensor(mid, BUF_STATE), before)
            sim.close()


@pytest.mark.parametrize("n", [64, 20001])
def test_tree_with_more_than_four_branching_bodies_is_refused(n, torch, oracle):
    """The run path needs at most 4 branching bodies (tree_topology runs before the lane / thread choice): more is refused
    with B2Error (unsupported) on every batch size, and the state is left as it was."""
    import b2sim
    from b2sim import _lib
    xml, t, _ = make_tree(oracle, 12, "bushy", seed=950)
    assert tree_urdf.branching_bodies(list(t["parent"][:12])) > tree_urdf.MAX_BRANCH
    sim = b2sim.Simulator(n, 0.001, 1)
    mid = sim.insert_model(xml, pose=POSE)
    for j in range(12):
        sim.set_control_mode(mid, j, MODE_FORCE)
    before = sim.tensor(mid, BUF_STATE).clone()
    with pytest.raises(b2sim.B2Error) as err:
        sim.run()
    assert err.value.code == _lib.ERR_UNSUPPORTED
    assert torch.equal(sim.tensor(mid, BUF_STATE), before)
    sim.close()
