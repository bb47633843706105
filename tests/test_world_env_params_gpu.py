"""Per-env free-body inertia and contact friction on the B200 (b2sim_enable_free_body_params, b2sim_enable_shape_friction):
initial values, untouched rows against a twin simulator without rows, random rows against one oracle world per env on the
free-body and coupled pipelines, known answers (resting forces, sliding distances), the rows' lifecycle and fp32."""
import os
import subprocess
import sys

import numpy as np
import pytest

from test_coupled_cpu import BASE, EDGE as PICK_EDGE, Q0, pick_scene

pytestmark = pytest.mark.gpu

MASS, EDGE = 5.0, 0.2
I = 1 / 12 * MASS * (EDGE ** 2 + EDGE ** 2)
CUBE_URDF = f"""
    <robot name="cube_robot">
        <link name="cube">
            <inertial><origin rpy="0 0 0" xyz="0 0 0"/><mass value="{MASS}"/>
              <inertia ixx="{I}" ixy="0" ixz="0" iyy="{I}" iyz="0" izz="{I}"/></inertial>
            <collision><geometry><box size="{EDGE} {EDGE} {EDGE}"/></geometry><origin rpy="0 0 0" xyz="0 0 0"/></collision>
        </link>
    </robot>"""
TABLE_CENTRE, TABLE_SIZE = (0.6, 0.0, 0.05), (0.4, 0.4, 0.1)
TABLE_SDF = f"""<?xml version="1.0"?>
<sdf version="1.7"><model name="table"><static>true</static><link name="top">
  <collision name="c"><geometry><box><size>{TABLE_SIZE[0]} {TABLE_SIZE[1]} {TABLE_SIZE[2]}</size></box></geometry></collision>
</link></model></sdf>"""
BALL_URDF = """<robot name="ball"><link name="ball">
  <inertial><mass value="1.0"/><inertia ixx="0.01" ixy="0" ixz="0" iyy="0.01" iyz="0" izz="0.01"/></inertial>
</link></robot>"""
PICK_I = 0.1 / 12 * 2 * PICK_EDGE ** 2
PICK_CUBE_URDF = CUBE_URDF.replace(f'value="{MASS}"', 'value="0.1"').replace(f'"{I}"', f'"{PICK_I}"').replace(
    f"{EDGE} {EDGE} {EDGE}", f"{PICK_EDGE} {PICK_EDGE} {PICK_EDGE}")
PICK_TABLE_SDF = """<?xml version="1.0"?>
<sdf version="1.7"><model name="table"><static>true</static><link name="top">
  <collision name="c"><geometry><box><size>0.4 0.4 0.05</size></box></geometry></collision>
</link></model></sdf>"""
KP, KD = [100.0] * 7 + [10000.0] * 2, [17.5] * 7 + [100.0] * 2
G = 9.8


def sample_envs(n):
    """Envs of the first warp, a middle warp and the tail of the batch."""
    mid = (n // 64) * 32
    return sorted(set(list(range(0, 32, 3)) + list(range(mid, mid + 32, 3)) + list(range(n - 20, n, 2))))


def random_body_rows(rng, n, mass, inertia, com_max=0.005):
    """[n, 10] rows: mass in [0.5, 2] x nominal, centre of mass within com_max, nominal inertia scaled per axis and rotated."""
    rows = np.zeros((n, 10))
    rows[:, 0] = mass * rng.uniform(0.5, 2.0, n)
    d = rng.normal(size=(n, 3))
    rows[:, 1:4] = d / np.linalg.norm(d, axis=1, keepdims=True) * rng.uniform(0, com_max, (n, 1))
    for e in range(n):
        q = rng.normal(size=4); q /= np.linalg.norm(q)
        R = rotation(q)
        Ic = R @ np.diag(np.diag(inertia) * rng.uniform(0.7, 1.4, 3)) @ R.T
        rows[e, 4:] = Ic[[0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]]
    return rows


def rotation(q):
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def inertia_of(row):
    xx, xy, xz, yy, yz, zz = row[4:]
    return np.array([[xx, xy, xz], [xy, yy, yz], [xz, yz, zz]])


def put(view, values):
    import torch
    view.copy_(torch.as_tensor(np.asarray(values), device=view.device, dtype=view.dtype))


@pytest.fixture()
def tumbling_world(model_files):
    """Factory: two tumbling cubes (a over the ground, b over a table box), ground plane and table, the initial states of
    test_world_kernel_matches_oracle. Returns (sim, ground, table, a, b, X0)."""
    import b2sim
    sims = []

    def make(n, dtype="float64", seed=0):
        sim = b2sim.Simulator(n, 0.001, 1, dtype)
        sims.append(sim)
        ground = sim.insert_model_file(model_files["ground_plane"])
        table = sim.insert_model(TABLE_SDF, pose=list(TABLE_CENTRE) + [1.0, 0, 0, 0], name="table")
        a = sim.insert_model(CUBE_URDF, name="a")
        b = sim.insert_model(CUBE_URDF, name="b")
        rng = np.random.default_rng(seed)
        X0 = np.zeros((n, 2, 13))
        X0[:, :, 3] = 1.0
        X0[:, 0, :3] = np.c_[rng.uniform(-0.02, 0.02, (n, 2)), rng.uniform(0.12, 0.3, n)]
        X0[:, 1, :3] = np.c_[TABLE_CENTRE[0] + rng.uniform(-0.02, 0.02, n), rng.uniform(-0.02, 0.02, n),
                             rng.uniform(0.22, 0.4, n)]
        quat = rng.normal(size=(n, 2, 4)); quat /= np.linalg.norm(quat, axis=2, keepdims=True)
        X0[::2, :, 3:7] = quat[::2]
        X0[:, :, 7:13] = rng.uniform(-1, 1, (n, 2, 6))
        put(sim.tensor(a, 14), X0[:, 0])
        put(sim.tensor(b, 14), X0[:, 1])
        return sim, ground, table, a, b, X0

    yield make
    for sim in sims:
        sim.close()


def free_states(sim, ids):
    return np.stack([sim.tensor(m, 14).cpu().numpy() for m in ids], axis=1)


def test_initial_values(tumbling_world, model_files):
    """The views start from the loader's body_mass, body_com, body_Ic and shape_mu, in every env; enabling again returns
    the same rows without refilling them."""
    n = 200
    sim, ground, table, a, b, _ = tumbling_world(n)
    panda = sim.insert_model_file(model_files["panda"], pose=list(BASE) + [1.0, 0, 0, 0], name="panda")
    envs = sample_envs(n)
    for m in (a, b):
        t = sim.info(m).tables()
        rows = sim.enable_free_body_params(m)
        assert rows.shape == (n, 10) and rows.dtype.is_floating_point and rows.element_size() == 8
        want = np.r_[t["body_mass"], t["body_com"], t["body_Ic"][[0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]]]
        np.testing.assert_array_equal(rows.cpu().numpy()[envs], np.tile(want, (len(envs), 1)))
        assert want[0] == MASS and want[4] == pytest.approx(I)
    for m in (ground, table, a, panda):
        t = sim.info(m).tables()
        mu = sim.enable_shape_friction(m)
        assert mu.shape == (n, t["nshapes"]) and t["nshapes"] > 0
        np.testing.assert_array_equal(mu.cpu().numpy()[envs], np.tile(t["shape_mu"], (len(envs), 1)))
    mu = sim.enable_shape_friction(a)
    mu[:, 0] = 0.3
    again = sim.enable_shape_friction(a)
    assert again.data_ptr() == mu.data_ptr() and (again == 0.3).all()
    assert sim.enable_shape_friction(a, False) is None
    assert sim.enable_free_body_params(a, False) is None
    # the C entry point accepts a NULL view
    assert sim.lib.b2sim_enable_free_body_params(sim.handle, b, 1, None) == 0


def test_untouched_rows_track_the_twin(tumbling_world):
    """A world whose rows were never written tracks a twin simulator without rows: 1e-12 relative after one step, the
    tolerances of test_world_kernel_matches_oracle over 200 steps. After disabling every row, one step from a state copied
    into both is bit-identical."""
    n = 160
    sim, ground, table, a, b, _ = tumbling_world(n)
    twin, *_ = tumbling_world(n)
    for m in (a, b):
        sim.enable_free_body_params(m)
    for m in (ground, table, a, b):
        sim.enable_shape_friction(m)
    ids = (a, b)
    sim.run(); twin.run()
    got, want = free_states(sim, ids), free_states(twin, ids)
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    for _ in range(199):
        sim.run(); twin.run()
    got, want = free_states(sim, ids), free_states(twin, ids)
    close = np.abs(got - want).reshape(n, -1).max(axis=1)
    assert np.median(close) < 1e-8 and (close < 1e-5).mean() > 0.9, close
    counts = np.array([len(sim.contacts(e)) for e in range(n)])
    twin_counts = np.array([len(twin.contacts(e)) for e in range(n)])
    assert (counts == twin_counts).mean() > 0.9
    for m in (a, b):
        assert sim.enable_free_body_params(m, False) is None
    for m in (ground, table, a, b):
        assert sim.enable_shape_friction(m, False) is None
    for m in ids:
        sim.tensor(m, 14).copy_(twin.tensor(m, 14))
    sim.run(); twin.run()
    for m in ids:
        assert (sim.tensor(m, 14) == twin.tensor(m, 14)).all()


def test_random_free_body_rows_match_the_oracle(tumbling_world, oracle):
    """Two tumbling cubes over the ground and a table box: every env has its own masses, centres of mass (within 5 mm),
    rotated and scaled inertias and friction on every shape. Each sampled env against an oracle world built from its own
    rows, at the tolerances of test_world_kernel_matches_oracle (states and contact counts) over 400 steps."""
    n, T = 160, 400
    sim, ground, table, a, b, X0 = tumbling_world(n, seed=1)
    rng = np.random.default_rng(11)
    body = {m: random_body_rows(rng, n, MASS, np.eye(3) * I) for m in (a, b)}
    mu = {m: rng.uniform(0.2, 1.2, n) for m in (ground, table, a, b)}
    for m in (a, b):
        put(sim.enable_free_body_params(m), body[m])
    for m in (ground, table, a, b):
        put(sim.enable_shape_friction(m)[:, 0], mu[m])
    envs = sample_envs(n)
    worlds = []
    for e in envs:
        bodies = [oracle.make_box_body(body[m][e, 0], [EDGE] * 3, inertia=inertia_of(body[m][e]), com=body[m][e, 1:4],
                                       mu=mu[m][e]) for m in (a, b)]
        statics = [oracle.ground_plane(mu=mu[ground][e]), oracle.make_box_static(TABLE_SIZE, TABLE_CENTRE, mu=mu[table][e])]
        worlds.append(oracle.make_world(bodies, statics))
    ref = X0[envs].copy()
    counts = np.zeros(len(envs), int)
    for _ in range(T):
        sim.run()
        for k in range(len(envs)):
            counts[k] = len(oracle.world_step(worlds[k], ref[k]))
    got = free_states(sim, (a, b))[envs]
    close = np.abs(got - ref).reshape(len(envs), -1).max(axis=1)
    assert np.median(close) < 1e-8 and (close < 1e-5).mean() > 0.9, close
    gpu_counts = np.array([len(sim.contacts(e)) for e in envs])
    assert (gpu_counts == counts).mean() > 0.9 and counts.max() > 0
    assert got[:, 0, 2].min() > 0.09


@pytest.mark.parametrize("solver", ["warp", "thread"])
def test_both_contact_solvers_with_rows(solver):
    """The free-body comparisons above under each contact pipeline (k_world_prepare / k_world_finish, k_world_free), in a
    subprocess because the selection is read once per process."""
    env = dict(os.environ, B2_CONTACT_SOLVER=solver)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", os.path.abspath(__file__), "-k",
                        "test_random_free_body_rows_match_the_oracle or test_untouched_rows or test_stacked or test_sliding "
                        "or test_rewritten_row or test_rows_survive or test_friction_rows_before"],
                       env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


def stacked_cubes(model_files, n, masses):
    import b2sim
    sim = b2sim.Simulator(n, 0.001, 1)
    ground = sim.insert_model_file(model_files["ground_plane"])
    ids = []
    for k, z in enumerate((EDGE / 2, 1.5 * EDGE)):
        m = sim.insert_model(CUBE_URDF, pose=(0, 0, z, 1, 0, 0, 0), name=f"c{k}")
        put(sim.enable_free_body_params(m)[:, 0], masses[:, k])
        ids.append(m)
    return sim, ground, ids


def ground_force_z(sim, e, body, ground):
    return sum(c[7][2] for c in sim.contacts(e) if c[0] == body and c[2] == ground)


def test_stacked_cubes_rest_on_their_masses(model_files):
    """Two stacked cubes with per-env masses (the upper one 0.5 - 2 times the lower one): after 150 steps the normal forces
    of the bottom cube's ground contacts sum to (m1 + m2) g within 0.1 N, averaged over the next 50 steps (50 sweeps a step
    leave the stack's impulses unconverged by up to ~1 N in a single step; the impulse over a span balances the weight to
    the stack's change of momentum)."""
    n = 100
    rng = np.random.default_rng(2)
    masses = rng.uniform(2.0, 6.0, (n, 2))
    masses[:, 1] = masses[:, 0] * rng.uniform(0.5, 2.0, n)
    sim, ground, (lower, upper) = stacked_cubes(model_files, n, masses)
    for _ in range(150):
        sim.run()
    envs = sample_envs(n)
    force = np.zeros(len(envs))
    for _ in range(50):
        sim.run()
        force += [ground_force_z(sim, e, lower, ground) / 50 for e in envs]
    np.testing.assert_allclose(force, masses[envs].sum(axis=1) * G, atol=0.1)
    sim.close()


def sliding_cube(sim, cube, v0):
    import torch
    X = sim.tensor(cube, 14)
    X.zero_()
    X[:, 2] = EDGE / 2
    X[:, 3] = 1.0
    X[:, 7] = v0
    for _ in range(800):
        sim.run()
    torch.cuda.synchronize()
    return X[:, 0].cpu().numpy(), X[:, 7].cpu().numpy()


def test_sliding_cube_stops_after_its_friction_distance(model_files):
    """A cube launched across the ground at v0 stops after v0^2 / (2 mu g) within 2 %, mu = the smaller of the cube's and
    the ground's rows; each of the two is the smaller one in some envs."""
    import b2sim
    n, v0 = 96, 1.0
    sim = b2sim.Simulator(n, 0.001, 1)
    ground = sim.insert_model_file(model_files["ground_plane"])
    cube = sim.insert_model(CUBE_URDF, pose=(0, 0, EDGE / 2, 1, 0, 0, 0), name="cube")
    rng = np.random.default_rng(4)
    mu_cube, mu_ground = rng.uniform(0.25, 0.8, n), rng.uniform(0.25, 0.8, n)
    put(sim.enable_shape_friction(cube)[:, 0], mu_cube)
    put(sim.enable_shape_friction(ground)[:, 0], mu_ground)
    mu = np.minimum(mu_cube, mu_ground)
    assert (mu_cube < mu_ground).any() and (mu_ground < mu_cube).any()
    x, v = sliding_cube(sim, cube, v0)
    envs = sample_envs(n)
    np.testing.assert_allclose(x[envs], v0 ** 2 / (2 * mu[envs] * G), rtol=0.02)
    assert np.abs(v[envs]).max() < 1e-6
    sim.close()


def pick_rows(rng, n, mu_cols):
    body = random_body_rows(rng, n, 0.1, np.eye(3) * PICK_I)
    mu = {k: rng.uniform(0.6, 1.2, n) for k in mu_cols}
    return body, mu


def run_pick_scene(oracle, model_files, extra_cubes=0):
    """test_coupled_kernel_matches_oracle with random rows: the cube's mass, centre of mass and inertia, and the friction of
    the cube, the table and both finger pads in every env; each sampled env against an oracle simulator built from them."""
    import torch
    import b2sim
    from b2sim import _lib
    n = 96
    t, m, D, _, rs0, X0, table_centre = pick_scene(oracle, model_files)
    m.effort[7] = m.effort[8] = 500.0
    sim = b2sim.Simulator(n, 0.001, 1)
    ground = sim.insert_model_file(model_files["ground_plane"])
    panda = sim.insert_model_file(model_files["panda"], pose=list(BASE) + [1.0, 0, 0, 0], name="panda")
    table = sim.insert_model(PICK_TABLE_SDF, pose=table_centre + [1.0, 0, 0, 0], name="table")
    cube = sim.insert_model(PICK_CUBE_URDF, pose=list(X0[0, :3]) + [1.0, 0, 0, 0], name="cube")
    extra_X = [np.array([-0.5, 0.4 * (k - 1), PICK_EDGE / 2, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0.0]) for k in range(extra_cubes)]
    extras = [sim.insert_model(PICK_CUBE_URDF, pose=list(x[:7]), name=f"extra{k}") for k, x in enumerate(extra_X)]
    rng = np.random.default_rng(5)
    Xc = np.tile(X0[0], (n, 1))
    Xc[:, 0] += rng.uniform(-0.004, 0.004, n)
    Xc[:, 1] += rng.uniform(-0.01, 0.01, n)
    put(sim.tensor(cube, _lib.BUF_BASE_STATE), Xc)
    tb = sim.info(panda).tables()
    pads = [k for k in range(tb["nshapes"]) if tb["link_body"][tb["shape_link"][k]] >= 0 and tb["shape_type"][k] == 0]
    assert len(pads) == 2
    body, mu = pick_rows(rng, n, ["cube", "table"] + [f"pad{k}" for k in pads])
    put(sim.enable_free_body_params(cube), body)
    put(sim.enable_shape_friction(cube)[:, 0], mu["cube"])
    put(sim.enable_shape_friction(table)[:, 0], mu["table"])
    pad_view = sim.enable_shape_friction(panda)
    for k in pads:
        put(pad_view[:, k], mu[f"pad{k}"])
    state = sim.tensor(panda, _lib.BUF_STATE)
    state[:, :9] = torch.as_tensor(Q0, device="cuda")
    for j in (7, 8):
        assert sim.lib.b2sim_set_max_generalized_force(sim.handle, panda, j, 500.0) == 0
    sim.set_controller_period(panda, 0.001)
    sim.set_computed_torque(panda, KP, KD)
    pos_t = sim.tensor(panda, _lib.BUF_POS_TARGET)
    for j in range(9):
        sim.set_joint(panda, _lib.FIELD_POSITION_TARGET, -1, j, Q0[j])
        sim.set_joint(panda, _lib.FIELD_VELOCITY_TARGET, -1, j, 0.0)
        sim.set_joint(panda, _lib.FIELD_ACCELERATION_TARGET, -1, j, 0.0)
    envs = sample_envs(n)
    refs = []
    for e in envs:
        bodies = [oracle.make_box_body(body[e, 0], [PICK_EDGE] * 3, inertia=inertia_of(body[e]), com=body[e, 1:4],
                                       mu=mu["cube"][e])]
        bodies += [oracle.make_box_body(0.1, [PICK_EDGE] * 3) for _ in extras]
        world = oracle.make_world(bodies, [oracle.ground_plane(),
                                           oracle.make_box_static([0.4, 0.4, 0.05], table_centre, mu=mu["table"][e])])
        rs = oracle.RobotShapes.from_buffer_copy(rs0)
        for slot, k in enumerate(pads):
            rs.rshape[slot].mu = mu[f"pad{k}"][e]
        ref = oracle.Sim(m, 0.001, 1)
        assert oracle.sim_attach_world(ref, world, rs, np.array([Xc[e]] + extra_X))
        ref.set_controller_period(0.001)
        for j in range(9):
            ref.reset_position(j, Q0[j])
        ref.run(True)
        ref.load_computed_torque(KP, KD)
        for j in range(9):
            ref.set_position_target(j, Q0[j]); ref.set_velocity_target(j, 0.0); ref.set_acceleration_target(j, 0.0)
        refs.append(ref)
    lift = np.linalg.pinv(D.point_jacobian(np.r_[Q0[:7], 0.025, 0.025], 6)[:3, :7]) @ np.array([0.0, 0.0, 0.05])
    ids = [cube] + extras

    def compare(tag, tol_q, tol_x):
        got_q = state.cpu().numpy()[envs]
        got_x = free_states(sim, ids)[envs]
        want_q = np.array([[r.position(j) for j in range(9)] + [r.velocity(j) for j in range(9)] for r in refs])
        want_x = np.array([oracle.sim_world_state(r) for r in refs])
        err_q = np.abs(got_q - want_q).max(axis=1)
        err_x = np.abs(got_x - want_x).reshape(len(envs), -1).max(axis=1)
        assert np.median(err_q) < tol_q and np.median(err_x) < tol_x, (tag, err_q, err_x)
        assert (err_q < 1e3 * tol_q).mean() > 0.9 and (err_x < 1e3 * tol_x).mean() > 0.9, (tag, err_q, err_x)
        return got_x

    for phase, steps in (("open", 100), ("close", 300), ("lift", 600)):
        if phase == "close":
            pos_t[:, 7:] = 0.0
            for r in refs:
                r.set_position_target(7, 0.0); r.set_position_target(8, 0.0)
        if phase == "lift":
            pos_t[:, :7] += torch.as_tensor(lift, device="cuda")
            for r in refs:
                for j in range(7):
                    r.set_position_target(j, Q0[j] + lift[j])
        for _ in range(steps):
            sim.run()
            for r in refs:
                r.run(False)
        got_x = compare(phase, 1e-8, 1e-8)
        counts = np.array([len(sim.contacts(e)) for e in envs])
        want_counts = np.array([len(oracle.sim_contacts(r)) for r in refs])
        assert (counts == want_counts).mean() > 0.9, (phase, counts, want_counts)
    assert (got_x[:, 0, 2] - X0[0, 2] > 0.03).all()       # every env lifted its cube
    sim.close()


@pytest.mark.parametrize("path", ["forked", "single_prepare", "four_cubes"])
def test_pick_scene_rows_match_the_oracle(path, oracle, model_files, monkeypatch):
    """The pick scene with random rows through the coupled kernels: the forked lane pipeline (k_coupled_rows), one prepare
    kernel (B2_COUPLED_SPLIT=0: k_coupled_prepare), and the Panda with four cubes (33 generalized velocities: k_world_coupled).
    The thread dynamics (k_coupled_dynamics) run in the next test."""
    if path == "single_prepare":
        monkeypatch.setenv("B2_COUPLED_SPLIT", "0")
    run_pick_scene(oracle, model_files, extra_cubes=3 if path == "four_cubes" else 0)


def test_pick_scene_rows_with_thread_dynamics():
    """B2_RUN_KERNEL=thread (read once per process, hence the subprocess): the split pipeline's dynamics run in
    k_coupled_dynamics instead of the lane kernel."""
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", os.path.abspath(__file__), "-k",
                        "test_pick_scene_rows_match_the_oracle and forked"],
                       env=dict(os.environ, B2_RUN_KERNEL="thread"), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


def test_rewritten_row_changes_only_its_env(tumbling_world):
    """A row written between runs acts from the next run on, in its env only: the other envs stay bit-identical to a twin
    whose rows were not rewritten."""
    n, env = 160, 77
    sim, ground, table, a, b, _ = tumbling_world(n)
    twin, tground, _, ta, tb_, _ = tumbling_world(n)
    rows = [sim.enable_free_body_params(a), sim.enable_shape_friction(ground)]
    twin.enable_free_body_params(ta); twin.enable_shape_friction(tground)
    for _ in range(20):
        sim.run(); twin.run()
    rows[0][env, 0] *= 3.0
    rows[1][env, 0] = 0.2
    for _ in range(100):
        sim.run(); twin.run()
    got, want = free_states(sim, (a, b)), free_states(twin, (ta, tb_))
    others = np.arange(n) != env
    np.testing.assert_array_equal(got[others], want[others])
    assert np.abs(got[env] - want[env]).max() > 1e-6


def test_rows_survive_world_rebuilds(model_files):
    """Rows written on a cube resting on a table survive inserting a second cube and removing the table: the cube falls
    onto the ground and rests there on its per-env mass."""
    import b2sim
    import torch
    n = 64
    sim = b2sim.Simulator(n, 0.001, 1)
    ground = sim.insert_model_file(model_files["ground_plane"])
    table = sim.insert_model(TABLE_SDF, pose=list(TABLE_CENTRE) + [1.0, 0, 0, 0], name="table")
    cube = sim.insert_model(CUBE_URDF, pose=(TABLE_CENTRE[0], 0, TABLE_SIZE[2] + EDGE / 2, 1, 0, 0, 0), name="cube")
    masses = np.random.default_rng(6).uniform(1.0, 8.0, n)
    rows = sim.enable_free_body_params(cube)
    put(rows[:, 0], masses)
    mu = sim.enable_shape_friction(cube)
    mu[:, 0] = 0.7
    before = rows.clone()
    for _ in range(100):
        sim.run()
    other = sim.insert_model(CUBE_URDF, pose=(-1.0, 0, EDGE / 2, 1, 0, 0, 0), name="other")
    sim.remove_model(table)
    for _ in range(600):
        sim.run()
    torch.cuda.synchronize()
    assert torch.equal(sim.enable_free_body_params(cube), before) and (sim.enable_shape_friction(cube) == 0.7).all()
    for e in sample_envs(n):
        assert ground_force_z(sim, e, cube, ground) == pytest.approx(masses[e] * G, abs=0.1), e
    assert sim.base_state(other, 0)[2] == pytest.approx(EDGE / 2, abs=3e-3)
    sim.close()


def test_friction_rows_before_the_first_free_body(model_files):
    """Friction rows of the ground enabled while the world has no free body are read once a cube is inserted."""
    import b2sim
    n, v0 = 64, 1.0
    sim = b2sim.Simulator(n, 0.001, 1)
    ground = sim.insert_model_file(model_files["ground_plane"])
    mu = np.random.default_rng(7).uniform(0.3, 0.9, n)
    put(sim.enable_shape_friction(ground)[:, 0], mu)
    sim.run()
    cube = sim.insert_model(CUBE_URDF, pose=(0, 0, EDGE / 2, 1, 0, 0, 0), name="cube")
    x, _ = sliding_cube(sim, cube, v0)
    envs = sample_envs(n)
    np.testing.assert_allclose(x[envs], v0 ** 2 / (2 * mu[envs] * G), rtol=0.02)
    sim.close()


def test_refusals(model_files):
    """Free-body rows on a model that is not free-floating, friction rows on a model without collision shapes."""
    import b2sim
    from b2sim import _lib
    sim = b2sim.Simulator(8, 0.001, 1)
    ground = sim.insert_model_file(model_files["ground_plane"])
    panda = sim.insert_model_file(model_files["panda"], pose=list(BASE) + [1.0, 0, 0, 0], name="panda")
    ball = sim.insert_model(BALL_URDF, pose=(0, 0, 1, 1, 0, 0, 0), name="ball")
    assert sim.info(ball).kind == _lib.KIND_FREE
    for m in (ground, panda):
        with pytest.raises(b2sim.B2Error) as err:
            sim.enable_free_body_params(m)
        assert err.value.code == _lib.ERR_UNSUPPORTED
    with pytest.raises(b2sim.B2Error) as err:
        sim.enable_shape_friction(ball)
    assert err.value.code == _lib.ERR_UNSUPPORTED
    assert sim.enable_free_body_params(ball).shape == (8, 10)
    sim.close()


def test_fp32_untouched_rows_track_the_twin(tumbling_world):
    """fp32 simulator: untouched rows track the fp32 twin without rows to 1e-5 relative after one step."""
    n = 160
    sim, ground, table, a, b, _ = tumbling_world(n, "float32")
    twin, *_ = tumbling_world(n, "float32")
    for m in (a, b):
        assert sim.enable_free_body_params(m).element_size() == 4
    for m in (ground, table, a, b):
        sim.enable_shape_friction(m)
    sim.run(); twin.run()
    np.testing.assert_allclose(free_states(sim, (a, b)), free_states(twin, (a, b)), rtol=1e-5, atol=1e-6)
