"""Seeded URDF generator for fixed-base kinematic trees of 1-16 one-DoF joints (test helper, not a conftest).

`generate(nq, topology, seed, ...)` returns URDF text that the engine's loader and the oracle's loader both accept: root
link `world`, revolute / continuous / prismatic joints with z, x / y or random unit axes, joint and inertial origins with
`rpy`, off-diagonal inertias, fixed joints interleaved, and joints written in shuffled file order so that the loaded body
indices are not depth-first (`parent != i - 1` is common).

Topologies:
    chain          every body on the previous one (a prismatic joint in the middle)
    star           every body a child of the base
    base_children  2-3 children of the base, each carrying a sub-chain
    random         a random tree with at most 4 branching bodies once loaded (kMaxBranch of the engine)
    panda          the Panda's body structure: a 7-chain of revolute joints plus two prismatic leaves on body 6, bodies in
                   that order; axes, origins and inertias are random
    bushy          more than 4 branching bodies once loaded (the engine refuses it)

A branching body is a body with a child that is not the next body index (b2_tree_fast.hpp, branch_slots). Both loaders
number bodies by scanning the joints in file order and taking the first one whose parent link is already placed, so the
count depends on the file order; `loaded_parents` restates that scan.
"""
import numpy as np

TOPOLOGIES = ("chain", "star", "base_children", "random", "panda", "bushy")
MAX_BRANCH = 4


def _f(x):
    return repr(float(x))


def _v(v):
    return " ".join(_f(x) for x in v)


def _rpy_R(rpy):
    r, p, y = rpy
    cr, sr, cp, sp, cy, sy = np.cos(r), np.sin(r), np.cos(p), np.sin(p), np.cos(y), np.sin(y)
    return (np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]]) @ np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]])
            @ np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]]))


def _tree_parents(nq, topology, rng):
    """Parent of each body in generation order (-1 = the base)."""
    if topology == "chain":
        return [i - 1 for i in range(nq)]
    if topology == "star":
        return [-1] * nq
    if topology == "base_children":
        k = min(nq, int(rng.integers(2, 4)))
        tails = list(range(k))
        par = [-1] * k
        for i in range(k, nq):
            c = int(rng.integers(0, k))
            par.append(tails[c])
            tails[c] = i
        return par
    if topology == "panda":
        assert nq == 9, "the Panda topology has 9 joints"
        return [-1, 0, 1, 2, 3, 4, 5, 6, 6]
    if topology in ("random", "bushy"):
        return [-1] + [int(rng.integers(-1, i)) for i in range(1, nq)]
    raise ValueError(topology)


def _joint_kinds(nq, topology, par, rng):
    if topology == "panda":
        return ["revolute"] * 7 + ["prismatic"] * 2
    kinds = [str(rng.choice(["revolute", "continuous", "prismatic"], p=[0.45, 0.25, 0.3])) for _ in range(nq)]
    # a prismatic joint in the middle of a chain: a body with a parent and a child
    mid = [i for i in range(nq) if par[i] >= 0 and i in par]
    if mid:
        kinds[mid[len(mid) // 2]] = "prismatic"
    return kinds


def _axis(rng, axes):
    pick = {"mixed": int(rng.integers(0, 3)), "z": 0, "xy": 1, "random": 2}[axes]
    if pick == 0:
        return np.array([0.0, 0.0, 1.0])
    if pick == 1:
        return np.array([1.0, 0.0, 0.0]) if rng.random() < 0.5 else np.array([0.0, 1.0, 0.0])
    a = rng.normal(size=3)
    return a / np.linalg.norm(a)


def _inertial(rng):
    """Mass 0.2-2 kg, a centre-of-mass offset, an inertial frame rotated by `rpy` and a principal inertia with eigenvalues in
    [0.02, 0.04] kg m^2 written in a second random frame: off-diagonal terms, smallest eigenvalue >= 0.02, and the triangle
    inequality of a physical body holds."""
    m = rng.uniform(0.2, 2.0)
    Q = _rpy_R(rng.uniform(-np.pi, np.pi, 3))
    I = Q @ np.diag(rng.uniform(0.02, 0.04, 3)) @ Q.T
    return (f"<inertial><origin xyz='{_v(rng.uniform(-0.1, 0.1, 3))}' rpy='{_v(rng.uniform(-np.pi, np.pi, 3))}'/>"
            f"<mass value='{_f(m)}'/><inertia ixx='{_f(I[0, 0])}' ixy='{_f(I[0, 1])}' ixz='{_f(I[0, 2])}' "
            f"iyy='{_f(I[1, 1])}' iyz='{_f(I[1, 2])}' izz='{_f(I[2, 2])}'/></inertial>")


def _origin(rng, scale=0.25):
    return f"<origin xyz='{_v(rng.uniform(-scale, scale, 3))}' rpy='{_v(rng.uniform(-np.pi, np.pi, 3))}'/>"


def loaded_parents(joints):
    """Body parents as both loaders number them. joints: [(name, type, parent_link, child_link)] in file order."""
    placed = {"world": -1}
    pending = list(joints)
    parents = []
    while pending:
        for j in pending:
            if j[2] in placed:
                break
        else:
            raise ValueError("disconnected joints")
        pending.remove(j)
        if j[1] == "fixed":
            placed[j[3]] = placed[j[2]]
        else:
            placed[j[3]] = len(parents)
            parents.append(placed[j[2]])
    return parents


def branching_bodies(parents):
    return len({p for c, p in enumerate(parents) if p >= 0 and p != c - 1})


def generate(nq, topology="random", seed=0, axes="mixed", fixed_links=True, last_link_on_world=False, damping=0.0,
             friction=0.0, name=None):
    """URDF text of a seeded random fixed-base tree with `nq` one-DoF joints.

    fixed_links: a link welded to `world` (some children of the base hang from it) and links welded to two moving bodies
        (with mass: they are lumped into their body; a child body may hang from one).
    last_link_on_world: the last <link> in file order is welded to `world` (the reach task's default end effector when the
        model has no `end_effector_frame`).
    damping / friction: <dynamics> on every joint (0: none written).
    Revolute and prismatic joints have position limits that include [-2, 2] rad / [-0.4, 0.4] m; continuous joints have none.
    """
    assert 1 <= nq <= 16 and topology in TOPOLOGIES
    rng = np.random.default_rng([seed, nq, TOPOLOGIES.index(topology)])
    for attempt in range(1000):
        par = _tree_parents(nq, topology, rng)
        kinds = _joint_kinds(nq, topology, par, rng)
        links, joints = [], []   # joints: (text, (name, type, parent link, child link))
        body_link = [f"b{i}" for i in range(nq)]
        attach = {i: body_link[i] for i in range(-1, nq)}   # the link children of body i hang from
        attach[-1] = "world"
        if fixed_links:
            links.append(f"<link name='plate'>{_inertial(rng)}</link>")
            joints.append((f"<joint name='plate_weld' type='fixed'><parent link='world'/><child link='plate'/>"
                           f"{_origin(rng)}</joint>", ("plate_weld", "fixed", "world", "plate")))
            for i in sorted(set(rng.choice(nq, size=min(2, nq), replace=False).tolist())):
                links.append(f"<link name='tool{i}'>{_inertial(rng)}</link>")
                joints.append((f"<joint name='tool{i}_weld' type='fixed'><parent link='{body_link[i]}'/>"
                               f"<child link='tool{i}'/>{_origin(rng)}</joint>", (f"tool{i}_weld", "fixed", body_link[i], f"tool{i}")))
                if rng.random() < 0.5:
                    attach[i] = f"tool{i}"
        for i in range(nq):
            links.append(f"<link name='{body_link[i]}'>{_inertial(rng)}</link>")
            p = par[i]
            plink = attach[p]
            if p < 0 and fixed_links and rng.random() < 0.5:
                plink = "plate"
            k = kinds[i]
            extra = ""
            if k == "revolute":
                lim = (rng.uniform(-2.8, -2.0), rng.uniform(2.0, 2.8))
                extra += f"<limit lower='{_f(lim[0])}' upper='{_f(lim[1])}' effort='1000' velocity='100'/>"
            elif k == "prismatic":
                lim = (rng.uniform(-0.6, -0.4), rng.uniform(0.4, 0.6))
                extra += f"<limit lower='{_f(lim[0])}' upper='{_f(lim[1])}' effort='1000' velocity='100'/>"
            elif rng.random() < 0.5:
                extra += "<limit effort='1000' velocity='100'/>"
            if damping or friction:
                extra += f"<dynamics damping='{_f(damping)}' friction='{_f(friction)}'/>"
            joints.append((f"<joint name='j{i}' type='{k}'><parent link='{plink}'/><child link='{body_link[i]}'/>"
                           f"{_origin(rng)}<axis xyz='{_v(_axis(rng, axes))}'/>{extra}</joint>",
                           (f"j{i}", k, plink, body_link[i])))
        if last_link_on_world:
            links.append(f"<link name='tip'>{_inertial(rng)}</link>")
            joints.append((f"<joint name='tip_weld' type='fixed'><parent link='world'/><child link='tip'/>{_origin(rng)}</joint>",
                           ("tip_weld", "fixed", "world", "tip")))
        if topology != "panda":
            order = rng.permutation(len(joints))
            joints = [joints[k] for k in order]
            if not last_link_on_world:
                links = [links[k] for k in rng.permutation(len(links))]
        nbr = branching_bodies(loaded_parents([j[1] for j in joints]))
        if (topology == "bushy") == (nbr > MAX_BRANCH) and (topology != "panda" or nbr == 1):
            break
    else:
        raise RuntimeError(f"no {topology} tree with {nq} joints found")
    body = "".join(links) + "".join(j[0] for j in joints)
    return f"<robot name='{name or f'gen_{topology}_{nq}_{seed}'}'><link name='world'/>{body}</robot>"


def generated_set(count=300, seed=0):
    """(nq, topology, seed, xml) for `count` trees of 1-16 joints over every topology that fits the joint count."""
    out = []
    rng = np.random.default_rng(seed)
    k = 0
    while len(out) < count:
        nq = int(rng.integers(1, 17))
        topo = TOPOLOGIES[k % len(TOPOLOGIES)]
        k += 1
        if (topo == "panda" and nq != 9) or (topo == "bushy" and nq < 10):
            continue
        out.append((nq, topo, k, generate(nq, topo, seed=k)))
    return out
