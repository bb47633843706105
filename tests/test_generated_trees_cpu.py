"""Generated kinematic trees of 1-16 joints (tests/helpers/tree_urdf.py) through the engine's loader and its host-compiled
rigid-body templates, against the oracle's independent loader and arithmetic.

The bundled models are a 1-joint pendulum, a 2-joint chain and the 9-joint Panda; these trees add star and multi-branch
topologies, bodies numbered out of depth-first order, non-z and random joint axes, prismatic joints inside chains, links
welded to moving bodies and to the base, and rotated inertial frames. The GPU counterpart is test_generated_trees_gpu.py.
"""
import importlib.util
import os

import numpy as np
import pytest

import b2sim
from test_rbd_host import G, POSES, dp, rbd  # noqa: F401  (rbd: the host-compiled templates, a module fixture)

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("tree_urdf", os.path.join(HERE, "helpers", "tree_urdf.py"))
tree_urdf = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(tree_urdf)

TREES = tree_urdf.generated_set(120, seed=7)


def _id(tree):
    return f"{tree[1]}-{tree[0]}-{tree[2]}"


@pytest.mark.parametrize("tree", TREES[:60], ids=_id)
def test_generated_tables_match_the_independent_loader(tree, oracle):
    nq, _, _, xml = tree
    info = b2sim.ModelInfo.from_string(xml)
    t = info.tables()
    ref, _ = oracle.load_urdf(xml)
    assert info.joint_names == ref["joint_names"] and info.link_names == ref["link_names"]
    assert t["nq"] == ref["nb"] == nq == info.dofs
    assert np.array_equal(t["parent"], ref["parent"][:nq])
    assert np.array_equal(t["jtype"] - 1, ref["jtype"][:nq])
    for key in ("axis", "R", "p", "mass", "com", "Ic", "damping", "friction", "effort"):
        np.testing.assert_allclose(t[key], np.asarray(ref[key])[:nq], rtol=0, atol=1e-14, err_msg=key)
    for key in ("lower", "upper"):
        assert np.array_equal(t[key], np.asarray(ref[key])[:nq]), key
    nl = t["nlinks"]
    assert np.array_equal(t["link_body"], ref["link_body"][:nl])
    np.testing.assert_allclose(t["link_R"], ref["link_R"], atol=1e-14)
    np.testing.assert_allclose(t["link_p"], ref["link_p"], atol=1e-14)
    np.testing.assert_allclose(t["base_mass"], ref["base_mass"], atol=1e-14)
    np.testing.assert_allclose(t["base_mc"], ref["base_mc"], atol=1e-14)
    np.testing.assert_allclose(t["base_Io"], ref["base_Io"], atol=1e-14)


def test_generated_set_covers_the_shapes_it_is_for(oracle):
    """The set the tests draw from really has what the kernels have to handle: every joint count, bodies whose parent is
    not the previous index, several children of the base, non-z axes, prismatic joints with a parent and a child, trees the
    low-footprint path refuses, and links welded to the base and to moving bodies."""
    seen = dict(nq=set(), nonseq=0, base_kids=0, nonz=0, mid_prismatic=0, bushy=0, welded_base=0, welded_body=0)
    for nq, topo, _, xml in TREES:
        t, _ = oracle.load_urdf(xml)
        par = list(t["parent"][:nq])
        seen["nq"].add(nq)
        seen["nonseq"] += sum(p >= 0 and p != i - 1 for i, p in enumerate(par))
        seen["base_kids"] += par.count(-1) >= 2
        seen["nonz"] += sum(abs(a[2]) != 1.0 for a in t["axis"][:nq])
        seen["mid_prismatic"] += sum(t["jtype"][i] == 2 and par[i] >= 0 and i in par for i in range(nq))
        seen["bushy"] += tree_urdf.branching_bodies(par) > tree_urdf.MAX_BRANCH
        nb = t["link_body"]
        seen["welded_base"] += int(np.sum(nb < 0) > 0)
        seen["welded_body"] += int(len(nb) - np.sum(nb < 0) > nq)
    assert seen["nq"] == set(range(1, 17))
    assert min(v for k, v in seen.items() if k != "nq") >= 10, seen


def _padded(rng, nq, lo, hi):
    x = np.zeros(16)
    x[:nq] = rng.uniform(lo, hi, nq)
    return x


@pytest.mark.parametrize("pose", POSES, ids=["identity", "offset"])
def test_generated_host_dynamics_match_oracle(pose, rbd, oracle):  # noqa: F811
    """Forward dynamics (articulated-body algorithm and the low-footprint variant, dt 0 and 1e-3), inverse dynamics, mass
    matrix, forward kinematics, centroidal quantities and the momentum Jacobian of every generated tree, at the tolerances
    of test_rbd_host.py. The low-footprint path refuses (-2) exactly the trees with more than 4 branching bodies."""
    pose7 = np.array(list(pose[0]) + list(pose[1]))
    refused = 0
    for nq, topo, seed, xml in TREES:
        x = xml.encode()
        t, model = oracle.load_urdf(xml, base_position=pose[0], base_orientation_wxyz=pose[1])
        D = oracle.Dynamics(model)
        bushy = tree_urdf.branching_bodies(list(t["parent"][:nq])) > tree_urdf.MAX_BRANCH
        rng = np.random.default_rng(seed)
        msg = f"{topo} nq={nq} seed={seed}"
        for trial in range(2):
            q, dq = _padded(rng, nq, -2, 2), _padded(rng, nq, -3, 3)
            tau, ddq_in = _padded(rng, nq, -10, 10), _padded(rng, nq, -5, 5)
            for dt in (0.0, 1e-3):
                ref = D.forward_dynamics(q[:nq], dq[:nq], tau[:nq], dt)
                tol = dict(rtol=1e-9, atol=1e-9 * (1 + np.abs(ref).max()), err_msg=msg)
                out = np.zeros(16)
                assert rbd.rbd_forward_dynamics(x, dp(pose7), dp(G), dt, dp(q), dp(dq), dp(tau), dp(out)) == nq
                np.testing.assert_allclose(out[:nq], ref, **tol)
                fast = np.zeros(16)
                rc = rbd.rbd_forward_dynamics_fast(x, dp(pose7), dp(G), dt, dp(q), dp(dq), dp(tau), dp(fast))
                assert rc == (-2 if bushy else nq), msg
                if not bushy:
                    np.testing.assert_allclose(fast[:nq], ref, **tol)
            refused += bushy
            out = np.zeros(16)
            rbd.rbd_inverse_dynamics(x, dp(pose7), dp(G), dp(q), dp(dq), dp(ddq_in), 1, dp(out))
            np.testing.assert_allclose(out[:nq], D.inverse_dynamics(q[:nq], dq[:nq], ddq_in[:nq]), rtol=1e-10, atol=1e-10,
                                       err_msg=msg)
            M = np.full(256, np.nan)
            rbd.rbd_mass_matrix(x, dp(pose7), dp(G), dp(q), dp(M))
            np.testing.assert_allclose(M[:nq * nq].reshape(nq, nq), D.mass_matrix(q[:nq]), rtol=1e-10, atol=1e-12, err_msg=msg)
            R = np.zeros(16 * 9); p = np.zeros(16 * 3)
            rbd.rbd_forward_kinematics(x, dp(pose7), dp(G), dp(q), dp(R), dp(p))
            Rr, pr = D.forward_kinematics(q[:nq])
            np.testing.assert_allclose(R[:9 * nq].reshape(nq, 3, 3), Rr, atol=1e-12, err_msg=msg)
            np.testing.assert_allclose(p[:3 * nq].reshape(nq, 3), pr, atol=1e-12, err_msg=msg)
            com, vel, mom, jac = np.zeros(3), np.zeros(3), np.zeros(12), np.zeros(3 * nq)
            assert rbd.rbd_centroidal(x, dp(pose7), dp(G), dp(q), dp(dq), dp(com), dp(vel), dp(mom), dp(jac)) == nq
            rc, rv, rm, rg, rJ = D.centroidal(q[:nq], dq[:nq], t["base_mass"], t["base_mc"])
            np.testing.assert_allclose(com, rc, rtol=1e-12, atol=1e-13, err_msg=msg)
            np.testing.assert_allclose(vel, rv, rtol=1e-11, atol=1e-12, err_msg=msg)
            np.testing.assert_allclose(mom[:6], rm, rtol=1e-10, atol=1e-11, err_msg=msg)
            np.testing.assert_allclose(mom[6:], rg, rtol=1e-10, atol=1e-11, err_msg=msg)
            np.testing.assert_allclose(jac.reshape(3, nq), rJ, rtol=1e-11, atol=1e-12, err_msg=msg)
            jm, locked = np.zeros(6 * nq), np.zeros(10)
            assert rbd.rbd_momentum(x, dp(pose7), dp(G), dp(q), dp(jm), dp(locked)) == nq
            rJm, rl = D.momentum_jacobian(q[:nq], t["base_mass"], t["base_mc"], t["base_Io"])
            np.testing.assert_allclose(jm.reshape(6, nq), rJm, rtol=1e-10, atol=1e-11, err_msg=msg)
            np.testing.assert_allclose(locked, rl, rtol=1e-11, atol=1e-12, err_msg=msg)
    assert refused >= 10
