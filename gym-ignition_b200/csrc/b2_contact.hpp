// Free-floating rigid bodies with ground / box contacts: one world = a few free bodies + static shapes.
//
// What it replaces for these bodies: DART World::step as reached from
// cpp/scenario/plugins/Physics/Physics.cpp:1824-1835 (free-joint dynamics, collision detection, contact
// constraints) and the contact readback of Physics.cpp:2351-2540 / cpp/scenario/gazebo/src/Link.cpp:360-482.
// DART solves the contact LCP with Dantzig (PGS fallback) on ODE/FCL contact points; this is the "LCP-lite"
// the north star allows: box-corner / sphere contact points against planes and boxes, friction pyramid,
// projected Gauss-Seidel with a fixed iteration count, DART's error-reduction velocity for penetration.
// Contact configurations are compared on trajectory statistics (resting force, height, contact count), not on
// trajectories. Host+device templates: the CUDA kernel, the host test helper and nothing else use them.
#pragma once

#include "b2_rbd.hpp"

namespace b2 {

constexpr int kMaxFree = 8;
constexpr int kMaxStaticShapes = 16;
constexpr int kMaxBodyShapes = 2;
constexpr int kMaxContacts = 32;
constexpr int kContactRec = 10;  // position(3), normal(3), depth, force(3)

enum { kShapeBox = 0, kShapeSphere = 1, kShapeCylinder = 2, kShapePlane = 3 };

template <typename T>
struct ShapeDev {
    int type;
    int owner_model, owner_link;  // for reporting
    T size[3];                    // box: half extents; sphere: radius; plane: unit normal (world)
    T R[9];                       // body frame (free bodies) or world frame (static shapes)
    T p[3];
    T mu;
};

template <typename T>
struct FreeBodyDev {
    T mass;
    T Ic[9];      // about the COM, body axes
    T Ic_inv[9];
    T com[3];     // COM in the body (root link) frame
    int nshapes;
    ShapeDev<T> shape[kMaxBodyShapes];
};

constexpr int kMaxRobotShapes = 4;    // collision shapes on moving links of the articulated model of a world
constexpr int kMaxRobotContacts = 16; // contact points that involve such a shape
constexpr int kMaxJointRows = 16;     // joint limit / friction / servo rows solved together with the contacts
constexpr int kRobotSide = -1000;     // Contact::a / b = kRobotSide - k: shape k of the articulated model

template <typename T>
struct alignas(16) WorldDev {
    int nfree, nstatic, iterations;
    T dt, erp, max_erv;
    T g[3];
    FreeBodyDev<T> body[kMaxFree];
    ShapeDev<T> stat[kMaxStaticShapes];
    // shapes carried by moving links of the (single) articulated model of the world: pose in the body frame
    int nrobot, robot_model;
    int rbody[kMaxRobotShapes];
    ShapeDev<T> rshape[kMaxRobotShapes];
    // external wrench on free body i (Link::applyWorldWrench, Physics.cpp:1483-1532): world-frame force at the origin of
    // the body's root link and torque, for env ext_env[i] (-1: every env, -2: none). The host clears it on expiry.
    T ext[kMaxFree][6];
    long long ext_env[kMaxFree];
};

// Where the inertial data of the free bodies and the friction coefficients of the collision shapes come from (the world's
// counterpart of NominalParams / EnvParams, b2_rbd.hpp). WorldNominal: the shared world description.
template <typename T>
struct WorldNominal {
    B2_HD T mass(const FreeBodyDev<T>& fb, int) const { return fb.mass; }
    B2_HD V3<T> com(const FreeBodyDev<T>& fb, int) const { return ld3(fb.com); }
    B2_HD M3<T> Ic(const FreeBodyDev<T>& fb, int) const { return ld9(fb.Ic); }
    B2_HD M3<T> Ic_inv(const FreeBodyDev<T>& fb, int) const { return ld9(fb.Ic_inv); }
    // shape s of free body i, static shape k, shape r of the articulated model
    B2_HD T body_mu(const ShapeDev<T>& sh, int, int) const { return sh.mu; }
    B2_HD T stat_mu(const ShapeDev<T>& sh, int) const { return sh.mu; }
    B2_HD T robot_mu(const ShapeDev<T>& sh, int) const { return sh.mu; }
};

// Per-env rows of a world (b2sim_enable_free_body_params / b2sim_enable_shape_friction), resolved per slot by the host on
// every launch: env 0's row of free body i ([N][kFreeBodyCols]: mass, centre of mass xyz, inertia about it xx xy xz yy yz
// zz, root-link frame), and env 0's friction coefficient of every shape slot in its model's [N][nshapes] rows with that
// row's stride. Null: the slot reads the shared world description.
constexpr int kFreeBodyCols = 10;

template <typename T>
struct WorldRows {
    const T* body[kMaxFree];
    const T* body_mu[kMaxFree][kMaxBodyShapes];
    const T* stat_mu[kMaxStaticShapes];
    const T* robot_mu[kMaxRobotShapes];
    int body_mu_stride[kMaxFree];
    int stat_mu_stride[kMaxStaticShapes];
    int robot_mu_stride;
};

// WorldEnv: env e's rows wherever the slot has them, the shared value otherwise.
template <typename T>
struct WorldEnv {
    const WorldRows<T>& rows;
    long long e;
    B2_HD const T* row(int i) const { return rows.body[i] + e * kFreeBodyCols; }
    B2_HD T mass(const FreeBodyDev<T>& fb, int i) const { return rows.body[i] ? row(i)[0] : fb.mass; }
    B2_HD V3<T> com(const FreeBodyDev<T>& fb, int i) const { return rows.body[i] ? ld3(row(i) + 1) : ld3(fb.com); }
    B2_HD M3<T> Ic(const FreeBodyDev<T>& fb, int i) const
    {
        if (!rows.body[i]) return ld9(fb.Ic);
        const T* r = row(i);
        return M3<T>{{r[4], r[5], r[6], r[5], r[7], r[8], r[6], r[8], r[9]}};
    }
    // adjugate over determinant, as upload_world inverts the shared inertia on the host (b2_sim.cu)
    B2_HD M3<T> Ic_inv(const FreeBodyDev<T>& fb, int i) const
    {
        if (!rows.body[i]) return ld9(fb.Ic_inv);
        const M3<T> M = Ic(fb, i);
        const T* I = M.m;
        const T det = I[0] * (I[4] * I[8] - I[5] * I[7]) - I[1] * (I[3] * I[8] - I[5] * I[6]) + I[2] * (I[3] * I[7] - I[4] * I[6]);
        return M3<T>{{(I[4] * I[8] - I[5] * I[7]) / det, (I[2] * I[7] - I[1] * I[8]) / det, (I[1] * I[5] - I[2] * I[4]) / det,
                      (I[5] * I[6] - I[3] * I[8]) / det, (I[0] * I[8] - I[2] * I[6]) / det, (I[2] * I[3] - I[0] * I[5]) / det,
                      (I[3] * I[7] - I[4] * I[6]) / det, (I[1] * I[6] - I[0] * I[7]) / det, (I[0] * I[4] - I[1] * I[3]) / det}};
    }
    B2_HD T body_mu(const ShapeDev<T>& sh, int i, int s) const
    {
        const T* p = rows.body_mu[i][s];
        return p ? p[e * rows.body_mu_stride[i]] : sh.mu;
    }
    B2_HD T stat_mu(const ShapeDev<T>& sh, int k) const
    {
        const T* p = rows.stat_mu[k];
        return p ? p[e * rows.stat_mu_stride[k]] : sh.mu;
    }
    B2_HD T robot_mu(const ShapeDev<T>& sh, int r) const
    {
        const T* p = rows.robot_mu[r];
        return p ? p[e * rows.robot_mu_stride] : sh.mu;
    }
};

template <typename T> B2_HD M3<T> quat_to_rot(const T* q)
{
    const T w = q[0], x = q[1], y = q[2], z = q[3];
    return M3<T>{{T(1) - T(2) * (y * y + z * z), T(2) * (x * y - z * w), T(2) * (x * z + y * w),
                  T(2) * (x * y + z * w), T(1) - T(2) * (x * x + z * z), T(2) * (y * z - x * w),
                  T(2) * (x * z - y * w), T(2) * (y * z + x * w), T(1) - T(2) * (x * x + y * y)}};
}

template <typename T>
struct Contact {
    int a, b;          // side: free body index (>= 0), -1 - static shape index (b only), or kRobotSide - robot shape
    int shape_a;       // shape of body a that generated the point (reporting)
    int rslot;         // slot of the joint-space rows when one side is a link of the articulated model, else -1
    V3<T> pos, n;      // world; n points from b towards a
    T depth, mu;
    V3<T> t1, t2;
    T kn, kt1, kt2;    // effective masses along n, t1, t2
    T ln, lt1, lt2;    // accumulated impulses
    T bias;
};

// per-body working set during the solve
template <typename T>
struct BodyWork {
    V3<T> xc, vc, w;   // COM position, COM velocity, angular velocity (world)
    M3<T> R, Iinv;     // orientation, world inverse inertia
    T inv_mass;
};

template <typename T>
B2_HD void add_contact(Contact<T>* cs, int& nc, int a, int shape_a, int b, V3<T> pos, V3<T> n, T depth, T mu)
{
    if (nc >= kMaxContacts) return;
    Contact<T>& c = cs[nc++];
    c.a = a; c.b = b; c.shape_a = shape_a;
    c.rslot = -1;
    c.pos = pos; c.n = n; c.depth = depth; c.mu = mu;
    c.ln = c.lt1 = c.lt2 = T(0);
}

// Corners of `box` (half extents h, world pose Rb / pb) against the reference face of box B, or against a plane.
template <typename T>
B2_HD void box_vs_shape(Contact<T>* cs, int& nc, int a, int shape_a, int b, const M3<T>& Ra, V3<T> pa, const T* ha,
                        const ShapeDev<T>& sb, const M3<T>& Rb, V3<T> pb, T mu)
{
    if (sb.type == kShapePlane) {
        const V3<T> n = ld3(sb.size);
        for (int k = 0; k < 8; ++k) {
            const V3<T> cl = v3((k & 1) ? ha[0] : -ha[0], (k & 2) ? ha[1] : -ha[1], (k & 4) ? ha[2] : -ha[2]);
            const V3<T> x = pa + mul(Ra, cl);
            const T d = dot(n, x - pb);
            if (d <= T(0)) add_contact(cs, nc, a, shape_a, b, x, n, -d, mu);
        }
        return;
    }
    if (sb.type != kShapeBox) return;
    // reference face of B: the one A's centre is most outside of
    const V3<T> cb = mulT(Rb, pa - pb);
    const T ex[3] = {fabs(cb.x) - sb.size[0], fabs(cb.y) - sb.size[1], fabs(cb.z) - sb.size[2]};
    int axis = 0;
    if (ex[1] > ex[axis]) axis = 1;
    if (ex[2] > ex[axis]) axis = 2;
    const T cbv[3] = {cb.x, cb.y, cb.z};
    const T sgn = cbv[axis] >= T(0) ? T(1) : T(-1);
    const T margin = T(1e-6);
    for (int k = 0; k < 8; ++k) {
        const V3<T> cl = v3((k & 1) ? ha[0] : -ha[0], (k & 2) ? ha[1] : -ha[1], (k & 4) ? ha[2] : -ha[2]);
        const V3<T> x = pa + mul(Ra, cl);
        const V3<T> xl = mulT(Rb, x - pb);
        const T xv[3] = {xl.x, xl.y, xl.z};
        bool inside = true;
        for (int j = 0; j < 3; ++j)
            if (j != axis && fabs(xv[j]) > sb.size[j] + margin) inside = false;
        const T depth = sb.size[axis] - sgn * xv[axis];
        if (inside && depth >= T(0) && depth <= T(2) * sb.size[axis]) {
            const V3<T> nl = v3(axis == 0 ? sgn : T(0), axis == 1 ? sgn : T(0), axis == 2 ? sgn : T(0));
            add_contact(cs, nc, a, shape_a, b, x, mul(Rb, nl), depth, mu);
        }
    }
}

template <typename T>
B2_HD void sphere_vs_shape(Contact<T>* cs, int& nc, int a, int shape_a, int b, V3<T> ca, T r, const ShapeDev<T>& sb,
                           const M3<T>& Rb, V3<T> pb, T mu)
{
    if (sb.type == kShapePlane) {
        const V3<T> n = ld3(sb.size);
        const T d = dot(n, ca - pb) - r;
        if (d <= T(0)) add_contact(cs, nc, a, shape_a, b, ca - r * n, n, -d, mu);
    } else if (sb.type == kShapeBox) {
        const V3<T> cl = mulT(Rb, ca - pb);
        const T cv[3] = {cl.x, cl.y, cl.z};
        T q[3];
        bool inside = true;
        for (int j = 0; j < 3; ++j) {
            q[j] = cv[j] < -sb.size[j] ? -sb.size[j] : (cv[j] > sb.size[j] ? sb.size[j] : cv[j]);
            if (q[j] != cv[j]) inside = false;
        }
        if (inside) return;  // centre inside the box: not handled
        const V3<T> dl = v3(cv[0] - q[0], cv[1] - q[1], cv[2] - q[2]);
        const T dist = sqrt(dot(dl, dl));
        if (dist <= r) {
            const V3<T> n = mul(Rb, (T(1) / dist) * dl);
            add_contact(cs, nc, a, shape_a, b, pb + mul(Rb, v3(q[0], q[1], q[2])), n, r - dist, mu);
        }
    }
}

// Per-env working set of the articulated model inside a coupled world step (robot link shapes touching free bodies
// or static shapes). Joint rows and contact rows act on the same joint velocities dq through M^-1.
template <typename T>
struct RobotWork {
    int nq, nrc, nrows;
    T dq[kMaxDofs];
    T Minv[kMaxDofs * kMaxDofs];               // [i * nq + j]
    M3<T> Rw[kMaxDofs];                        // world pose of the body frames
    V3<T> pw[kMaxDofs];
    // contact rows: J = d (n, t1, t2) . (linear Jacobian of the contact point), Y = M^-1 J^T; [slot][3][nq]
    T J[kMaxRobotContacts * 3 * kMaxDofs];
    T Y[kMaxRobotContacts * 3 * kMaxDofs];
    // joint rows (limits, Coulomb friction, velocity servo): dq[rj] - rtarget in [.., ..] with impulse lambda in [lo, hi]
    int rj[kMaxJointRows];
    T rtarget[kMaxJointRows], rlo[kMaxJointRows], rhi[kMaxJointRows], rlam[kMaxJointRows];
};

B2_HD bool side_is_robot(int s) { return s <= kRobotSide; }

template <typename T> B2_HD V3<T> point_velocity(const BodyWork<T>& b, V3<T> r) { return b.vc + cross(b.w, r); }

// Velocity of side a minus velocity of side b at the contact point, along direction k (0: n, 1: t1, 2: t2).
template <bool ROBOT, typename T>
B2_HD T relative_velocity_along(const BodyWork<T>* bw, const RobotWork<T>* rw, const Contact<T>& c, int k, V3<T> d)
{
    V3<T> rel = v3(T(0), T(0), T(0));
    if (!ROBOT || c.a >= 0) rel = point_velocity(bw[c.a], c.pos - bw[c.a].xc);
    if (c.b >= 0) rel = rel - point_velocity(bw[c.b], c.pos - bw[c.b].xc);
    T v = dot(d, rel);
    if (ROBOT && c.rslot >= 0) {  // J already carries the sign of the robot's side
        const T* J = rw->J + (c.rslot * 3 + k) * rw->nq;
        for (int j = 0; j < rw->nq; ++j) v += J[j] * rw->dq[j];
    }
    return v;
}

template <typename T>
B2_HD T free_effective_mass(const BodyWork<T>& A, V3<T> pos, V3<T> d)
{
    const V3<T> ra = pos - A.xc;
    return A.inv_mass + dot(d, cross(mul(A.Iinv, cross(ra, d)), ra));
}

template <bool ROBOT, typename T>
B2_HD T effective_mass(const BodyWork<T>* bw, const RobotWork<T>* rw, const Contact<T>& c, int k, V3<T> d)
{
    T m = T(0);
    if (!ROBOT || c.a >= 0) m += free_effective_mass(bw[c.a], c.pos, d);
    if (c.b >= 0) m += free_effective_mass(bw[c.b], c.pos, d);
    if (ROBOT && c.rslot >= 0) {
        const T* J = rw->J + (c.rslot * 3 + k) * rw->nq;
        const T* Y = rw->Y + (c.rslot * 3 + k) * rw->nq;
        for (int j = 0; j < rw->nq; ++j) m += J[j] * Y[j];
    }
    return m;
}

// Impulse of magnitude `mag` along direction k (d) on side a, the opposite on side b.
template <bool ROBOT, typename T>
B2_HD void apply_impulse(BodyWork<T>* bw, RobotWork<T>* rw, const Contact<T>& c, int k, V3<T> d, T mag)
{
    const V3<T> P = mag * d;
    if (!ROBOT || c.a >= 0) {
        BodyWork<T>& A = bw[c.a];
        A.vc = A.vc + A.inv_mass * P;
        A.w = A.w + mul(A.Iinv, cross(c.pos - A.xc, P));
    }
    if (c.b >= 0) {
        BodyWork<T>& B = bw[c.b];
        B.vc = B.vc - B.inv_mass * P;
        B.w = B.w - mul(B.Iinv, cross(c.pos - B.xc, P));
    }
    if (ROBOT && c.rslot >= 0) {
        const T* Y = rw->Y + (c.rslot * 3 + k) * rw->nq;
        for (int j = 0; j < rw->nq; ++j) rw->dq[j] += Y[j] * mag;
    }
}

// Loads the free bodies of one world and applies the unconstrained velocity update (gravity, gyroscopic torque).
// P: where the inertial data and friction coefficients come from (WorldNominal / WorldEnv), here and below.
template <typename T, typename P = WorldNominal<T>>
B2_HD void bodies_begin(const WorldDev<T>& W, const T* X, BodyWork<T>* bw, long long env = -1, const P& prm = P())
{
    const T dt = W.dt;
    const V3<T> g = ld3(W.g);
    for (int i = 0; i < W.nfree; ++i) {
        const FreeBodyDev<T>& fb = W.body[i];
        const T* x = X + 13 * i;
        BodyWork<T>& b = bw[i];
        b.R = quat_to_rot(x + 3);
        const V3<T> rc = mul(b.R, prm.com(fb, i));
        b.xc = ld3(x) + rc;
        b.w = ld3(x + 10);
        b.vc = ld3(x + 7) + cross(b.w, rc);
        b.inv_mass = T(1) / prm.mass(fb, i);
        b.Iinv = mulBt(mul(b.R, prm.Ic_inv(fb, i)), b.R);
        const M3<T> Iw = mulBt(mul(b.R, prm.Ic(fb, i)), b.R);
        b.vc = b.vc + dt * g;
        b.w = b.w - dt * mul(b.Iinv, cross(b.w, mul(Iw, b.w)));
        if (W.ext_env[i] == -1 || (W.ext_env[i] >= 0 && W.ext_env[i] == env)) {
            const V3<T> f = ld3(W.ext[i]), mo = ld3(W.ext[i] + 3) + cross(ld3(x) - b.xc, f);
            b.vc = b.vc + (dt * b.inv_mass) * f;
            b.w = b.w + dt * mul(b.Iinv, mo);
        }
    }
}

// Contact points of the free bodies against static shapes and against each other.
template <typename T, typename P = WorldNominal<T>>
B2_HD void free_contacts(const WorldDev<T>& W, const BodyWork<T>* bw, Contact<T>* cs, int& nc, const P& prm = P())
{
    for (int i = 0; i < W.nfree; ++i) {
        const FreeBodyDev<T>& fb = W.body[i];
        for (int s = 0; s < fb.nshapes; ++s) {
            const ShapeDev<T>& sa = fb.shape[s];
            const M3<T> Ra = mul(bw[i].R, ld9(sa.R));
            const V3<T> pa = bw[i].xc + mul(bw[i].R, ld3(sa.p) - prm.com(fb, i));
            for (int k = 0; k < W.nstatic; ++k) {
                const ShapeDev<T>& sb = W.stat[k];
                const T mu = prm.body_mu(sa, i, s) < prm.stat_mu(sb, k) ? prm.body_mu(sa, i, s) : prm.stat_mu(sb, k);
                if (sa.type == kShapeBox) box_vs_shape(cs, nc, i, s, -1 - k, Ra, pa, sa.size, sb, ld9(sb.R), ld3(sb.p), mu);
                else if (sa.type == kShapeSphere) sphere_vs_shape(cs, nc, i, s, -1 - k, pa, sa.size[0], sb, ld9(sb.R), ld3(sb.p), mu);
            }
            for (int j = 0; j < W.nfree; ++j) {
                if (j == i) continue;
                const FreeBodyDev<T>& fj = W.body[j];
                for (int u = 0; u < fj.nshapes; ++u) {
                    const ShapeDev<T>& sb = fj.shape[u];
                    if (sb.type != kShapeBox) continue;
                    const M3<T> Rb = mul(bw[j].R, ld9(sb.R));
                    const V3<T> pb = bw[j].xc + mul(bw[j].R, ld3(sb.p) - prm.com(fj, j));
                    const T mu = prm.body_mu(sa, i, s) < prm.body_mu(sb, j, u) ? prm.body_mu(sa, i, s) : prm.body_mu(sb, j, u);
                    if (sa.type == kShapeBox) box_vs_shape(cs, nc, i, s, j, Ra, pa, sa.size, sb, Rb, pb, mu);
                    else if (sa.type == kShapeSphere) sphere_vs_shape(cs, nc, i, s, j, pa, sa.size[0], sb, Rb, pb, mu);
                }
            }
        }
    }
}

// Contact points of the articulated model's link shapes against static shapes and free bodies (both directions
// for box pairs: corners of either box against the reference face of the other). Self-collisions are disabled by
// the reference on insertion (cpp/scenario/gazebo/src/Model.cpp:175-178).
template <typename T, typename P = WorldNominal<T>>
B2_HD void robot_contacts(const WorldDev<T>& W, const BodyWork<T>* bw, const RobotWork<T>& rw, Contact<T>* cs, int& nc,
                          const P& prm = P())
{
    for (int r = 0; r < W.nrobot; ++r) {
        const ShapeDev<T>& sr = W.rshape[r];
        const int body = W.rbody[r];
        const M3<T> Rr = mul(rw.Rw[body], ld9(sr.R));
        const V3<T> pr = rw.pw[body] + mul(rw.Rw[body], ld3(sr.p));
        const int side = kRobotSide - r;
        for (int k = 0; k < W.nstatic; ++k) {
            const ShapeDev<T>& sb = W.stat[k];
            const T mu = prm.robot_mu(sr, r) < prm.stat_mu(sb, k) ? prm.robot_mu(sr, r) : prm.stat_mu(sb, k);
            if (sr.type == kShapeBox) box_vs_shape(cs, nc, side, r, -1 - k, Rr, pr, sr.size, sb, ld9(sb.R), ld3(sb.p), mu);
            else if (sr.type == kShapeSphere) sphere_vs_shape(cs, nc, side, r, -1 - k, pr, sr.size[0], sb, ld9(sb.R), ld3(sb.p), mu);
        }
        for (int j = 0; j < W.nfree; ++j) {
            const FreeBodyDev<T>& fj = W.body[j];
            for (int u = 0; u < fj.nshapes; ++u) {
                const ShapeDev<T>& sb = fj.shape[u];
                const M3<T> Rb = mul(bw[j].R, ld9(sb.R));
                const V3<T> pb = bw[j].xc + mul(bw[j].R, ld3(sb.p) - prm.com(fj, j));
                const T mu = prm.robot_mu(sr, r) < prm.body_mu(sb, j, u) ? prm.robot_mu(sr, r) : prm.body_mu(sb, j, u);
                if (sb.type == kShapeBox) {  // robot shape against the free box
                    if (sr.type == kShapeBox) box_vs_shape(cs, nc, side, r, j, Rr, pr, sr.size, sb, Rb, pb, mu);
                    else if (sr.type == kShapeSphere) sphere_vs_shape(cs, nc, side, r, j, pr, sr.size[0], sb, Rb, pb, mu);
                }
                if (sr.type == kShapeBox) {  // free shape against the robot box
                    if (sb.type == kShapeBox) box_vs_shape(cs, nc, j, u, side, Rb, pb, sb.size, sr, Rr, pr, mu);
                    else if (sb.type == kShapeSphere) sphere_vs_shape(cs, nc, j, u, side, pb, sb.size[0], sr, Rr, pr, mu);
                }
            }
        }
    }
}

// Joint-space rows of the robot-side contacts: J (along n, t1, t2, signed by the robot's side) and Y = M^-1 J^T.
// Contacts beyond kMaxRobotContacts are dropped (compacted out of the list).
template <typename T>
B2_HD void robot_contact_rows(const WorldDev<T>& W, const ModelDev<T>& m, RobotWork<T>& rw, Contact<T>* cs, int& nc)
{
    const int nq = rw.nq;
    int keep = 0;
    rw.nrc = 0;
    for (int k = 0; k < nc; ++k) {
        Contact<T> c = cs[k];
        const bool ra = side_is_robot(c.a), rb = side_is_robot(c.b);
        if (ra || rb) {
            if (rw.nrc >= kMaxRobotContacts) continue;
            c.rslot = rw.nrc++;
            const int body = W.rbody[kRobotSide - (ra ? c.a : c.b)];
            const T sign = ra ? T(1) : T(-1);
            const V3<T> dir[3] = {c.n, c.t1, c.t2};
            T* J = rw.J + c.rslot * 3 * nq;
            T* Y = rw.Y + c.rslot * 3 * nq;
            for (int e = 0; e < 3 * nq; ++e) J[e] = T(0);
            for (int i = body; i >= 0; i = m.parent[i]) {
                const V3<T> aw = mul(rw.Rw[i], ld3(m.axis[i]));
                const V3<T> lin = m.jtype[i] == kRevolute ? cross(aw, c.pos - rw.pw[i]) : aw;
                for (int d = 0; d < 3; ++d) J[d * nq + i] = sign * dot(dir[d], lin);
            }
            for (int d = 0; d < 3; ++d)
                for (int i = 0; i < nq; ++i) {
                    T y = T(0);
                    for (int j = 0; j < nq; ++j) y += rw.Minv[i * nq + j] * J[d * nq + j];
                    Y[d * nq + i] = y;
                }
        }
        cs[keep++] = c;
    }
    nc = keep;
}

// Tangent frame, effective masses and the error-reduction velocity of every contact.
template <typename T>
B2_HD void contact_frames(Contact<T>* cs, int nc)
{
    for (int k = 0; k < nc; ++k) {
        Contact<T>& c = cs[k];
        const V3<T> seed = fabs(c.n.x) < T(0.9) ? v3(T(1), T(0), T(0)) : v3(T(0), T(1), T(0));
        V3<T> t1 = cross(c.n, seed);
        t1 = (T(1) / sqrt(dot(t1, t1))) * t1;
        c.t1 = t1;
        c.t2 = cross(c.n, t1);
    }
}

template <bool ROBOT, typename T>
B2_HD void contact_rows(const WorldDev<T>& W, const BodyWork<T>* bw, const RobotWork<T>* rw, Contact<T>* cs, int nc)
{
    for (int k = 0; k < nc; ++k) {
        Contact<T>& c = cs[k];
        c.kn = effective_mass<ROBOT>(bw, rw, c, 0, c.n);
        c.kt1 = effective_mass<ROBOT>(bw, rw, c, 1, c.t1);
        c.kt2 = effective_mass<ROBOT>(bw, rw, c, 2, c.t2);
        T erv = c.depth * W.erp / W.dt;  // DART: penetration * ERP / dt, capped
        c.bias = erv > W.max_erv ? W.max_erv : erv;
    }
}

// One projected Gauss-Seidel sweep over the contacts.
template <bool ROBOT, typename T>
B2_HD void contact_sweep(BodyWork<T>* bw, RobotWork<T>* rw, Contact<T>* cs, int nc)
{
    for (int k = 0; k < nc; ++k) {
        Contact<T>& c = cs[k];
        const T ln = c.ln + (c.bias - relative_velocity_along<ROBOT>(bw, rw, c, 0, c.n)) / c.kn;
        const T ln_new = ln > T(0) ? ln : T(0);
        apply_impulse<ROBOT>(bw, rw, c, 0, c.n, ln_new - c.ln);
        c.ln = ln_new;
        const T lim = c.mu * c.ln;
        T l1 = c.lt1 - relative_velocity_along<ROBOT>(bw, rw, c, 1, c.t1) / c.kt1;
        l1 = l1 < -lim ? -lim : (l1 > lim ? lim : l1);
        apply_impulse<ROBOT>(bw, rw, c, 1, c.t1, l1 - c.lt1);
        c.lt1 = l1;
        T l2 = c.lt2 - relative_velocity_along<ROBOT>(bw, rw, c, 2, c.t2) / c.kt2;
        l2 = l2 < -lim ? -lim : (l2 > lim ? lim : l2);
        apply_impulse<ROBOT>(bw, rw, c, 2, c.t2, l2 - c.lt2);
        c.lt2 = l2;
    }
}

// One projected Gauss-Seidel sweep over the joint rows (DART's JointLimit / JointCoulombFriction / ServoMotor
// constraints): the row impulse acts on every joint velocity through column rj of M^-1.
template <typename T>
B2_HD void joint_row_sweep(RobotWork<T>& rw)
{
    const int nq = rw.nq;
    for (int a = 0; a < rw.nrows; ++a) {
        const int j = rw.rj[a];
        const T w = rw.dq[j] - rw.rtarget[a];
        T nl = rw.rlam[a] - w / rw.Minv[j * nq + j];
        nl = nl < rw.rlo[a] ? rw.rlo[a] : (nl > rw.rhi[a] ? rw.rhi[a] : nl);
        const T dl = nl - rw.rlam[a];
        rw.rlam[a] = nl;
        for (int i = 0; i < nq; ++i) rw.dq[i] += rw.Minv[i * nq + j] * dl;
    }
}

// Integrates the poses of the free bodies (rotation by the exponential map) and stores them back.
template <typename T, typename P = WorldNominal<T>>
B2_HD void body_end(const WorldDev<T>& W, int i, T* x /* the body's 13 state values */, BodyWork<T>& b, const P& prm = P())
{
    const T dt = W.dt;
    {
        const FreeBodyDev<T>& fb = W.body[i];
        const T wn = sqrt(dot(b.w, b.w));
        T q[4] = {x[3], x[4], x[5], x[6]};
        if (wn > T(0)) {
            T s, c;
            sincos_t(T(0.5) * wn * dt, &s, &c);
            const V3<T> ax = (s / wn) * b.w;
            const T d[4] = {c, ax.x, ax.y, ax.z};
            const T r0 = d[0] * q[0] - d[1] * q[1] - d[2] * q[2] - d[3] * q[3];
            const T r1 = d[0] * q[1] + d[1] * q[0] + d[2] * q[3] - d[3] * q[2];
            const T r2 = d[0] * q[2] - d[1] * q[3] + d[2] * q[0] + d[3] * q[1];
            const T r3 = d[0] * q[3] + d[1] * q[2] - d[2] * q[1] + d[3] * q[0];
            const T nrm = T(1) / sqrt(r0 * r0 + r1 * r1 + r2 * r2 + r3 * r3);
            q[0] = r0 * nrm; q[1] = r1 * nrm; q[2] = r2 * nrm; q[3] = r3 * nrm;
        }
        b.xc = b.xc + dt * b.vc;
        const M3<T> Rn = quat_to_rot(q);
        const V3<T> rc = mul(Rn, prm.com(fb, i));
        const V3<T> p = b.xc - rc, v = b.vc - cross(b.w, rc);
        x[0] = p.x; x[1] = p.y; x[2] = p.z;
        x[3] = q[0]; x[4] = q[1]; x[5] = q[2]; x[6] = q[3];
        x[7] = v.x; x[8] = v.y; x[9] = v.z;
        x[10] = b.w.x; x[11] = b.w.y; x[12] = b.w.z;
    }
}
template <typename T, typename P = WorldNominal<T>>
B2_HD void bodies_end(const WorldDev<T>& W, T* X, BodyWork<T>* bw, const P& prm = P())
{
    for (int i = 0; i < W.nfree; ++i) body_end(W, i, X + 13 * i, bw[i], prm);
}

// One step of every free body of one world. X: nfree x 13 (position, quaternion wxyz, linear and angular velocity
// of the body frame, world coordinates). cs: caller-provided contact workspace (kMaxContacts). Returns the number
// of contacts; their impulses divided by dt are the contact forces on body a.
template <typename T, typename P = WorldNominal<T>>
B2_HD int world_step(const WorldDev<T>& W, T* X, Contact<T>* cs, long long env = -1, const P& prm = P())
{
    BodyWork<T> bw[kMaxFree];
    bodies_begin(W, X, bw, env, prm);
    int nc = 0;
    free_contacts(W, bw, cs, nc, prm);
    contact_frames(cs, nc);
    contact_rows<false>(W, bw, (const RobotWork<T>*)nullptr, cs, nc);
    for (int it = 0; it < W.iterations; ++it) contact_sweep<false>(bw, (RobotWork<T>*)nullptr, cs, nc);
    bodies_end(W, X, bw, prm);
    return nc;
}

// Cholesky inverse of the joint-space mass matrix (in place: M is overwritten by its factor). Divisions are replaced
// by the reciprocals of the factor's diagonal, the unit right-hand sides skip their leading zeros, and only the
// lower triangle of the (symmetric) inverse is solved for.
template <typename T>
B2_HD void spd_inverse(int n, T* M, T* Minv)
{
    T rd[kMaxDofs];
    for (int j = 0; j < n; ++j) {
        T s = M[j * n + j];
        for (int k = 0; k < j; ++k) s -= M[j * n + k] * M[j * n + k];
        const T d = sqrt(s);
        M[j * n + j] = d;
        rd[j] = T(1) / d;
        for (int i = j + 1; i < n; ++i) {
            T t = M[i * n + j];
            for (int k = 0; k < j; ++k) t -= M[i * n + k] * M[j * n + k];
            M[i * n + j] = t * rd[j];
        }
    }
    for (int c = 0; c < n; ++c) {
        T y[kMaxDofs];
        y[c] = rd[c];
        for (int i = c + 1; i < n; ++i) {
            T t = T(0);
            for (int k = c; k < i; ++k) t -= M[i * n + k] * y[k];
            y[i] = t * rd[i];
        }
        for (int i = n - 1; i >= c; --i) {
            T t = y[i];
            for (int k = i + 1; k < n; ++k) t -= M[k * n + i] * Minv[k * n + c];
            const T x = t * rd[i];
            Minv[i * n + c] = x;
            Minv[c * n + i] = x;
        }
    }
}

// One step of a world that couples an articulated model with free bodies through contacts: DART's constraint
// stage (ConstraintSolver::solve behind Physics.cpp:1824-1835) sees the joint rows of the skeleton and every contact
// in one LCP. On entry q holds the joint positions and dq the joint velocities after the unconstrained update
// (dq += ddq dt); on return dq holds the constrained velocities. Positions are integrated by the caller.
// servo_bits / servo_target: joints under a velocity servo. Returns the number of contacts.
template <typename T, typename P = WorldNominal<T>>
B2_HD int coupled_step(const WorldDev<T>& W, const ModelDev<T>& m, const T* q, T* dq, unsigned servo_bits,
                       const T* servo_target, T* X, Contact<T>* cs, RobotWork<T>& rw, long long env = -1, const P& prm = P());

// ---------------------------------------------------------------------------------------------------------
// Dense-row form of the same constraint problem, for the warp-cooperative solver (b2_kernels.cuh k_pgs_solve):
// generalized velocity v = [dq (nq), (vc, w) of free body 0, (vc, w) of free body 1, ...] padded to nvp lanes,
// one row per joint constraint and three per contact (normal, t1, t2): J, Y = M^-1 J^T, and
// par = [c, -, lo | mu, hi] with the row update  lambda <- clamp(lambda + (c - J v) / k),  v += Y dlambda.
// ---------------------------------------------------------------------------------------------------------
constexpr int kMaxPgsRows = kMaxJointRows + 3 * kMaxContacts;

template <typename T>
struct PgsEnv {
    T* v;      // [nvp]
    T* J;      // [rows][nvp]
    T* par;    // [rows][4]: c, (reciprocal effective mass, filled by the solver), lo | mu, hi
    T* aux;    // M^-1 of the articulated model [nq][nq], then per free body: 1 / mass, world inverse inertia [9]
    int* cnt;  // nrows, joint rows
    int nvp;
};

B2_HD int pgs_aux_size(int nq, int nfree) { return nq * nq + 10 * nfree; }

// Writes the rows of one env: the Jacobians only, Y = M^-1 J^T and the effective masses are computed by the
// lanes of the solver from `aux`. nq = 0 / rw = nullptr: a world without an articulated model. Contacts that involve
// the articulated model beyond kMaxRobotContacts are dropped from the list (as in robot_contact_rows).
template <typename T>
B2_HD void write_dense_rows(const WorldDev<T>& W, const ModelDev<T>* m, int nq, const RobotWork<T>* rw,
                            const BodyWork<T>* bw, Contact<T>* cs, int& nc, const PgsEnv<T>& o, bool robot_state = true)
{
    // robot_state = false (split pipeline): the unconstrained joint velocities and M^-1 are written by the kernels
    // that run next to this one (k_coupled_dynamics, k_coupled_minv)
    const int nvp = o.nvp;
    for (int j = robot_state ? 0 : nq; j < nvp; ++j) o.v[j] = T(0);
    if (robot_state)
        for (int j = 0; j < nq; ++j) o.v[j] = rw->dq[j];
    for (int i = 0; i < W.nfree; ++i) {
        T* v = o.v + nq + 6 * i;
        v[0] = bw[i].vc.x; v[1] = bw[i].vc.y; v[2] = bw[i].vc.z;
        v[3] = bw[i].w.x; v[4] = bw[i].w.y; v[5] = bw[i].w.z;
        T* a = o.aux + nq * nq + 10 * i;
        a[0] = bw[i].inv_mass;
        for (int k = 0; k < 9; ++k) a[1 + k] = bw[i].Iinv.m[k];
    }
    int r = 0;
    const int njr = nq > 0 ? rw->nrows : 0;
    if (robot_state && nq > 0 && (njr > 0 || rw->nrc > 0))
        for (int k = 0; k < nq * nq; ++k) o.aux[k] = rw->Minv[k];
    for (int a = 0; a < njr; ++a, ++r) {
        T* J = o.J + r * nvp;
        for (int i = 0; i < nvp; ++i) J[i] = T(0);
        J[rw->rj[a]] = T(1);
        T* p = o.par + 4 * r;
        p[0] = rw->rtarget[a]; p[1] = T(0); p[2] = rw->rlo[a]; p[3] = rw->rhi[a];
    }
    V3<T> axis_w[kMaxDofs];  // world joint axes, once per env (every robot contact needs its chain's)
    for (int i = 0; i < nq; ++i) axis_w[i] = mul(rw->Rw[i], ld3(m->axis[i]));
    // joints between the base and each robot shape, as bit masks: the rows are then written joint by joint without walking
    // parent pointers (independent loads, no separate zero fill)
    unsigned chain_of[kMaxRobotShapes];
    for (int sidx = 0; sidx < W.nrobot; ++sidx) {
        unsigned bits = 0u;
        for (int i = W.rbody[sidx]; i >= 0; i = m->parent[i]) bits |= 1u << i;
        chain_of[sidx] = bits;
    }
    const int nv_used = nq + 6 * W.nfree;
    int keep = 0, nrc = 0;
    for (int k = 0; k < nc; ++k) {
        const Contact<T> c = cs[k];
        const bool ra = side_is_robot(c.a), rb = side_is_robot(c.b);
        if (ra || rb) {
            if (nrc >= kMaxRobotContacts) continue;
            ++nrc;
        }
        const V3<T> dir[3] = {c.n, c.t1, c.t2};
        T* J = o.J + r * nvp;
        {   // joint columns: sign * dir . (axis x (pos - origin)) for the revolute joints of the shape's chain, else zero
            const unsigned chain = (ra || rb) ? chain_of[kRobotSide - (ra ? c.a : c.b)] : 0u;
            const T sign = ra ? T(1) : T(-1);
            for (int i = 0; i < nq; ++i) {
                T v0 = T(0), v1 = T(0), v2 = T(0);
                if ((chain >> i) & 1u) {
                    const V3<T> aw = axis_w[i];
                    const V3<T> lin = m->jtype[i] == kRevolute ? cross(aw, c.pos - rw->pw[i]) : aw;
                    v0 = sign * dot(dir[0], lin); v1 = sign * dot(dir[1], lin); v2 = sign * dot(dir[2], lin);
                }
                J[i] = v0; J[nvp + i] = v1; J[2 * nvp + i] = v2;
            }
        }
        for (int b = 0; b < W.nfree; ++b) {  // free-body columns: +/- [dir, arm x dir] for the contact's sides, else zero
            const T sign = b == c.a ? T(1) : (b == c.b ? T(-1) : T(0));
            const V3<T> arm = c.pos - bw[b].xc;
            for (int d = 0; d < 3; ++d) {
                const V3<T> lin = sign * dir[d], ang = sign * cross(arm, dir[d]);
                T* Jb = J + d * nvp + nq + 6 * b;
                Jb[0] = lin.x; Jb[1] = lin.y; Jb[2] = lin.z; Jb[3] = ang.x; Jb[4] = ang.y; Jb[5] = ang.z;
            }
        }
        for (int d = 0; d < 3; ++d)
            for (int i = nv_used; i < nvp; ++i) J[d * nvp + i] = T(0);
        T erv = c.depth * W.erp / W.dt;  // DART: penetration * ERP / dt, capped
        erv = erv > W.max_erv ? W.max_erv : erv;
        for (int d = 0; d < 3; ++d) {
            T* p = o.par + 4 * (r + d);
            p[0] = d == 0 ? erv : T(0);
            p[1] = T(0);
            p[2] = d == 0 ? T(0) : c.mu;
            p[3] = T(INFINITY);
        }
        r += 3;
        cs[keep++] = c;
    }
    nc = keep;
    o.cnt[0] = r;
    o.cnt[1] = njr;
}

// Everything of a coupled step before the solve: kinematics, unconstrained free-body velocities, contact points,
// joint rows, M^-1, the robot-side contact rows and effective masses. Same sequence as coupled_step.
template <typename T, typename P = WorldNominal<T>>
B2_HD int coupled_prepare(const WorldDev<T>& W, const ModelDev<T>& m, const T* q, const T* dq, unsigned servo_bits,
                          const T* servo_target, const T* X, BodyWork<T>* bw, Contact<T>* cs, RobotWork<T>& rw, long long env = -1,
                          const P& prm = P())
{
    const int nq = m.nq;
    const T dt = W.dt, inf = T(INFINITY);
    rw.nq = nq;
    rw.nrc = 0;
    for (int j = 0; j < nq; ++j) rw.dq[j] = dq[j];
    forward_kinematics<T, kMaxDofs>(m, q, rw.Rw, rw.pw);
    bodies_begin(W, X, bw, env, prm);
    int nc = 0;
    free_contacts(W, bw, cs, nc, prm);
    robot_contacts(W, bw, rw, cs, nc, prm);
    int nr = 0;
    for (int j = 0; j < nq; ++j) {
        if ((servo_bits >> j) & 1u) {
            if (nr < kMaxJointRows) { rw.rj[nr] = j; rw.rtarget[nr] = servo_target[j]; rw.rlo[nr] = -m.effort[j] * dt; rw.rhi[nr] = m.effort[j] * dt; ++nr; }
            continue;
        }
        if (m.friction[j] != T(0) && nr < kMaxJointRows) { rw.rj[nr] = j; rw.rtarget[nr] = T(0); rw.rlo[nr] = -m.friction[j] * dt; rw.rhi[nr] = m.friction[j] * dt; ++nr; }
        if (q[j] <= m.lower[j] && nr < kMaxJointRows) { rw.rj[nr] = j; rw.rtarget[nr] = T(0); rw.rlo[nr] = T(0); rw.rhi[nr] = inf; ++nr; }
        if (q[j] >= m.upper[j] && nr < kMaxJointRows) { rw.rj[nr] = j; rw.rtarget[nr] = T(0); rw.rlo[nr] = -inf; rw.rhi[nr] = T(0); ++nr; }
    }
    rw.nrows = nr;
    for (int a = 0; a < nr; ++a) rw.rlam[a] = T(0);
    bool robot_touched = false;
    for (int k = 0; k < nc; ++k) robot_touched = robot_touched || side_is_robot(cs[k].a) || side_is_robot(cs[k].b);
    contact_frames(cs, nc);
    if (nr > 0 || robot_touched) {
        T M[kMaxDofs * kMaxDofs];
        mass_matrix<T, kMaxDofs>(m, q, M);
        spd_inverse(nq, M, rw.Minv);
        robot_contact_rows(W, m, rw, cs, nc);
    }
    contact_rows<true>(W, bw, &rw, cs, nc);
    return nc;
}

// What the three-launch pipeline needs of a coupled step before its solver: kinematics, unconstrained free-body
// velocities, contact points and tangents, joint rows and M^-1 (only when a joint row or a robot contact exists).
// M_known: the joint-space mass matrix at q when the caller already has it (the computed-torque controller), or null.
template <typename T, typename P = WorldNominal<T>>
B2_HD int coupled_prepare_rows(const WorldDev<T>& W, const ModelDev<T>& m, const T* q, const T* dq, unsigned servo_bits,
                               const T* servo_target, const T* X, const T* M_known, BodyWork<T>* bw, Contact<T>* cs,
                               RobotWork<T>& rw, bool with_minv = true, long long env = -1, const P& prm = P())
{
    const int nq = m.nq;
    const T dt = W.dt, inf = T(INFINITY);
    rw.nq = nq;
    for (int j = 0; j < nq; ++j) rw.dq[j] = dq[j];
    forward_kinematics<T, kMaxDofs>(m, q, rw.Rw, rw.pw);
    bodies_begin(W, X, bw, env, prm);
    int nc = 0;
    free_contacts(W, bw, cs, nc, prm);
    robot_contacts(W, bw, rw, cs, nc, prm);
    int nr = 0;
    for (int j = 0; j < nq; ++j) {
        if ((servo_bits >> j) & 1u) {
            if (nr < kMaxJointRows) { rw.rj[nr] = j; rw.rtarget[nr] = servo_target[j]; rw.rlo[nr] = -m.effort[j] * dt; rw.rhi[nr] = m.effort[j] * dt; ++nr; }
            continue;
        }
        if (m.friction[j] != T(0) && nr < kMaxJointRows) { rw.rj[nr] = j; rw.rtarget[nr] = T(0); rw.rlo[nr] = -m.friction[j] * dt; rw.rhi[nr] = m.friction[j] * dt; ++nr; }
        if (q[j] <= m.lower[j] && nr < kMaxJointRows) { rw.rj[nr] = j; rw.rtarget[nr] = T(0); rw.rlo[nr] = T(0); rw.rhi[nr] = inf; ++nr; }
        if (q[j] >= m.upper[j] && nr < kMaxJointRows) { rw.rj[nr] = j; rw.rtarget[nr] = T(0); rw.rlo[nr] = -inf; rw.rhi[nr] = T(0); ++nr; }
    }
    rw.nrows = nr;
    int nrc = 0;
    for (int k = 0; k < nc; ++k) nrc += (side_is_robot(cs[k].a) || side_is_robot(cs[k].b)) ? 1 : 0;
    rw.nrc = nrc;
    contact_frames(cs, nc);
    if (with_minv && (nr > 0 || nrc > 0)) {  // split pipeline: k_coupled_minv computes M^-1 concurrently
        T M[kMaxDofs * kMaxDofs];
        if (M_known) for (int k = 0; k < nq * nq; ++k) M[k] = M_known[k];
        else mass_matrix<T, kMaxDofs>(m, q, M);
        spd_inverse(nq, M, rw.Minv);
    }
    return nc;
}

// Pose part of bodies_begin only (no velocity update): what the finishing kernel needs to integrate the bodies.
template <typename T, typename P = WorldNominal<T>>
B2_HD void body_pose(const WorldDev<T>& W, int i, const T* x, BodyWork<T>& b, const P& prm = P())
{
    b.R = quat_to_rot(x + 3);
    b.xc = ld3(x) + mul(b.R, prm.com(W.body[i], i));
}
template <typename T, typename P = WorldNominal<T>>
B2_HD void bodies_pose(const WorldDev<T>& W, const T* X, BodyWork<T>* bw, const P& prm = P())
{
    for (int i = 0; i < W.nfree; ++i) body_pose(W, i, X + 13 * i, bw[i], prm);
}

// One step of a world that couples an articulated model with free bodies through contacts, solved by one thread
// (host tests, worlds too large for the warp-cooperative solver).
template <typename T, typename P>
B2_HD int coupled_step(const WorldDev<T>& W, const ModelDev<T>& m, const T* q, T* dq, unsigned servo_bits,
                       const T* servo_target, T* X, Contact<T>* cs, RobotWork<T>& rw, long long env, const P& prm)
{
    BodyWork<T> bw[kMaxFree];
    const int nc = coupled_prepare(W, m, q, dq, servo_bits, servo_target, X, bw, cs, rw, env, prm);
    for (int it = 0; it < W.iterations; ++it) {
        joint_row_sweep(rw);
        contact_sweep<true>(bw, &rw, cs, nc);
    }
    for (int j = 0; j < m.nq; ++j) dq[j] = rw.dq[j];
    bodies_end(W, X, bw, prm);
    return nc;
}

// Force on body a transmitted through contact c (world frame).
template <typename T> B2_HD V3<T> contact_force(const Contact<T>& c, T dt)
{
    return (T(1) / dt) * (c.ln * c.n + c.lt1 * c.t1 + c.lt2 * c.t2);
}

}  // namespace b2
