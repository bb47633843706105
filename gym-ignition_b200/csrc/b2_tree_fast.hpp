// Low-footprint articulated-body step for fixed-base trees (the Panda path).
//
// Same dynamics as b2_rbd.hpp::forward_dynamics (DART's ABA with implicit joint damping/spring; reference:
// cpp/scenario/plugins/Physics/Physics.cpp:1824-1835 -> dartsim World::step), reorganised for one-thread-per-env
// execution on the GPU:
//   * what crosses the three passes lives in a per-thread scratch column (shared memory on the device, a plain
//     array on the host): 19 scalars per body + 33 per branching body, instead of ~60 per body;
//   * joint transforms, velocity-product accelerations and bias forces are recomputed from (sin q, cos q, V)
//     instead of stored;
//   * articulated inertias are carried in registers down a chain and only parked in scratch at branching
//     bodies; their rotational / mass blocks are kept symmetric (21 scalars);
//   * gravity enters as a fictitious base acceleration, so no per-body gravity vector is kept.
// Host+device: tests/helpers/rbd_host.cpp runs it on the CPU against the oracle.
#pragma once

#include "b2_rbd.hpp"

namespace b2 {

// Strided view of one thread's scratch: element k lives at base[k * stride]. STRIDE > 0 fixes the stride at
// compile time (1 = a private array), STRIDE = 0 takes it from the `stride` member (shared-memory columns).
template <typename T, int STRIDE = 0>
struct Scratch {
    T* base;
    int stride;
    B2_HD T& operator[](int k) const { return STRIDE > 0 ? base[k * STRIDE] : base[k * stride]; }
};

constexpr int kSlotsPerBody = 19;   // s, c, V(6), U(6), psi, u, q, dq, tau
constexpr int kSlotsPerBranch = 27; // parked articulated inertia (21) + bias force (6)
constexpr int kMaxBranch = 4;

enum { SL_S = 0, SL_C = 1, SL_V = 2, SL_U = 8, SL_PSI = 14, SL_UU = 15, SL_Q = 16, SL_DQ = 17, SL_TAU = 18 };

B2_HD int scratch_slots(int nq, int nbranch) { return kSlotsPerBody * nq + kSlotsPerBranch * nbranch; }

// Which bodies need a parking slot: a body with a child that is not the next index (index order is
// parents-first, so a pure chain never parks). Returns the number of branch bodies, or -1 if too many.
inline int branch_slots(int nq, const int* parent, int* slot_of_body)
{
    int n = 0;
    for (int i = 0; i < nq; ++i) slot_of_body[i] = -1;
    for (int c = 0; c < nq; ++c) {
        const int p = parent[c];
        if (p >= 0 && p != c - 1 && slot_of_body[p] < 0) {
            if (n >= kMaxBranch) return -1;
            slot_of_body[p] = n++;
        }
    }
    return n;
}

template <typename T>
struct Sym3 {
    T xx, xy, xz, yy, yz, zz;
};
template <typename T> B2_HD V3<T> mul(const Sym3<T>& S, V3<T> v)
{
    return {S.xx * v.x + S.xy * v.y + S.xz * v.z, S.xy * v.x + S.yy * v.y + S.yz * v.z,
            S.xz * v.x + S.yz * v.y + S.zz * v.z};
}
// R S R^T for symmetric S
template <typename T> B2_HD Sym3<T> rot_sym(const M3<T>& R, const Sym3<T>& S)
{
    T t[9];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < 3; ++i) {
        const T r0 = R.m[3 * i], r1 = R.m[3 * i + 1], r2 = R.m[3 * i + 2];
        t[3 * i + 0] = r0 * S.xx + r1 * S.xy + r2 * S.xz;
        t[3 * i + 1] = r0 * S.xy + r1 * S.yy + r2 * S.yz;
        t[3 * i + 2] = r0 * S.xz + r1 * S.yz + r2 * S.zz;
    }
    Sym3<T> o;
    o.xx = t[0] * R.m[0] + t[1] * R.m[1] + t[2] * R.m[2];
    o.xy = t[0] * R.m[3] + t[1] * R.m[4] + t[2] * R.m[5];
    o.xz = t[0] * R.m[6] + t[1] * R.m[7] + t[2] * R.m[8];
    o.yy = t[3] * R.m[3] + t[4] * R.m[4] + t[5] * R.m[5];
    o.yz = t[3] * R.m[6] + t[4] * R.m[7] + t[5] * R.m[8];
    o.zz = t[6] * R.m[6] + t[7] * R.m[7] + t[8] * R.m[8];
    return o;
}

// Articulated inertia with symmetric diagonal blocks: [[A, B], [B^T, C]].
template <typename T>
struct AiS {
    Sym3<T> A, C;
    M3<T> B;
};

template <typename T> B2_HD V3<T> row(const M3<T>& M, int i) { return {M.m[3 * i], M.m[3 * i + 1], M.m[3 * i + 2]}; }
template <typename T> B2_HD V3<T> col(const M3<T>& M, int j) { return {M.m[j], M.m[3 + j], M.m[6 + j]}; }

// Joint placement from the stored sine / cosine (revolute) or the joint position (prismatic).
template <typename T>
B2_HD void joint_pose_sc(const ModelDev<T>& m, int i, T s, T c, T q, M3<T>& R, V3<T>& p)
{
    const V3<T> a = ld3(m.axis[i]);
    const M3<T> R0 = ld9(m.R[i]);
    const V3<T> p0 = ld3(m.p[i]);
    if (m.jtype[i] == kRevolute) {
        if (a.z == T(1)) {
            // rotation about the joint z axis (every Panda arm joint): the first two columns of R0 mix
            R = M3<T>{{c * R0.m[0] + s * R0.m[1], c * R0.m[1] - s * R0.m[0], R0.m[2],
                       c * R0.m[3] + s * R0.m[4], c * R0.m[4] - s * R0.m[3], R0.m[5],
                       c * R0.m[6] + s * R0.m[7], c * R0.m[7] - s * R0.m[6], R0.m[8]}};
        } else {
            const T t = T(1) - c;
            const M3<T> Rq{{c + t * a.x * a.x, t * a.x * a.y - s * a.z, t * a.x * a.z + s * a.y,
                            t * a.x * a.y + s * a.z, c + t * a.y * a.y, t * a.y * a.z - s * a.x,
                            t * a.x * a.z - s * a.y, t * a.y * a.z + s * a.x, c + t * a.z * a.z}};
            R = mul(R0, Rq);
        }
        p = p0;
    } else {
        R = R0;
        p = p0 + mul(R0, q * a);
    }
}

// Forward dynamics (implicit damping/spring). On entry the SL_Q / SL_DQ / SL_TAU slots of every body hold
// q, dq and the applied joint force, and the parking slots are zero (clear_parking). On return SL_TAU holds
// the joint acceleration of the body; SL_Q / SL_DQ are untouched. P: where inertias, damping and gravity come from
// (NominalParams: the model's tables, EnvParams: one env's rows).
template <typename T, typename W, typename P = NominalParams<T>>
B2_HD void forward_dynamics_fast(const ModelDev<T>& m, const int* branch_slot, T dt, const W& w, const P& prm = P())
{
    const int nq = m.nq;
    const int park0 = kSlotsPerBody * nq;

    // ---- pass 1: velocities, root to leaves ---------------------------------------------------------
    for (int i = 0; i < nq; ++i) {
        const int o = kSlotsPerBody * i, par = m.parent[i];
        const bool rev = m.jtype[i] == kRevolute;
        const T q = w[o + SL_Q], dq = w[o + SL_DQ];
        T s = T(0), c = T(1);
        if (rev) sincos_t(q, &s, &c);
        w[o + SL_S] = s;
        w[o + SL_C] = c;
        M3<T> R;
        V3<T> p;
        joint_pose_sc(m, i, s, c, q, R, p);
        Sv<T> Vp = sv_zero<T>();
        if (par >= 0) {
            const int op = kSlotsPerBody * par + SL_V;
            Vp = {{w[op], w[op + 1], w[op + 2]}, {w[op + 3], w[op + 4], w[op + 5]}};
        }
        Sv<T> V = {mulT(R, Vp.a), mulT(R, Vp.l + cross(Vp.a, p))};
        const V3<T> sd = dq * ld3(m.axis[i]);
        if (rev) V.a = V.a + sd;
        else V.l = V.l + sd;
        w[o + SL_V + 0] = V.a.x; w[o + SL_V + 1] = V.a.y; w[o + SL_V + 2] = V.a.z;
        w[o + SL_V + 3] = V.l.x; w[o + SL_V + 4] = V.l.y; w[o + SL_V + 5] = V.l.z;
    }

    // ---- pass 2: articulated inertias and bias forces, leaves to root ----------------------------------
    AiS<T> carry;
    Sv<T> carry_p;
    bool have_carry = false;
    for (int i = nq - 1; i >= 0; --i) {
        const int o = kSlotsPerBody * i, par = m.parent[i];
        const bool rev = m.jtype[i] == kRevolute;
        const V3<T> a = ld3(m.axis[i]);
        const T q = w[o + SL_Q], dq = w[o + SL_DQ];
        const Sv<T> V = {{w[o + SL_V], w[o + SL_V + 1], w[o + SL_V + 2]},
                         {w[o + SL_V + 3], w[o + SL_V + 4], w[o + SL_V + 5]}};
        // rigid-body part
        const T mass = prm.mass(m, i);
        const V3<T> mc = prm.mc(m, i);
        AiS<T> IA;
        {
            const M3<T> Io = prm.Io(m, i);
            IA.A = {Io.m[0], Io.m[1], Io.m[2], Io.m[4], Io.m[5], Io.m[8]};
        }
        IA.B = skew(mc);
        IA.C = {mass, T(0), T(0), mass, T(0), mass};
        Sv<T> pA;
        {
            const V3<T> n = mul(IA.A, V.a) + cross(mc, V.l);
            const V3<T> f = mass * V.l - cross(mc, V.a);
            pA.a = cross(V.a, n) + cross(V.l, f);
            pA.l = cross(V.a, f);
        }
        if (have_carry) {
            IA.A.xx += carry.A.xx; IA.A.xy += carry.A.xy; IA.A.xz += carry.A.xz;
            IA.A.yy += carry.A.yy; IA.A.yz += carry.A.yz; IA.A.zz += carry.A.zz;
            IA.C.xx += carry.C.xx; IA.C.xy += carry.C.xy; IA.C.xz += carry.C.xz;
            IA.C.yy += carry.C.yy; IA.C.yz += carry.C.yz; IA.C.zz += carry.C.zz;
            IA.B = IA.B + carry.B;
            pA = pA + carry_p;
        }
        if (branch_slot[i] >= 0) {
            const int k = park0 + kSlotsPerBranch * branch_slot[i];
            IA.A.xx += w[k + 0]; IA.A.xy += w[k + 1]; IA.A.xz += w[k + 2];
            IA.A.yy += w[k + 3]; IA.A.yz += w[k + 4]; IA.A.zz += w[k + 5];
            IA.C.xx += w[k + 6]; IA.C.xy += w[k + 7]; IA.C.xz += w[k + 8];
            IA.C.yy += w[k + 9]; IA.C.yz += w[k + 10]; IA.C.zz += w[k + 11];
            for (int e = 0; e < 9; ++e) IA.B.m[e] += w[k + 12 + e];
            pA.a.x += w[k + 21]; pA.a.y += w[k + 22]; pA.a.z += w[k + 23];
            pA.l.x += w[k + 24]; pA.l.y += w[k + 25]; pA.l.z += w[k + 26];
        }
        // velocity-product acceleration eta = V x (S dq)
        const V3<T> sd = dq * a;
        Sv<T> eta;
        if (rev) eta = {cross(V.a, sd), cross(V.l, sd)};
        else eta = {v3(T(0), T(0), T(0)), cross(V.a, sd)};
        // U = IA S, psi, u
        Sv<T> U;
        T d;
        if (rev) {
            U = {mul(IA.A, a), mulT(IA.B, a)};
            d = dot(a, U.a);
        } else {
            U = {mul(IA.B, a), mul(IA.C, a)};
            d = dot(a, U.l);
        }
        const T damping = prm.damping(m, i);
        d += dt * damping + dt * dt * m.stiffness[i];
        const T psi = T(1) / d;
        const Sv<T> pa = {mul(IA.A, eta.a) + mul(IA.B, eta.l) + pA.a, mulT(IA.B, eta.a) + mul(IA.C, eta.l) + pA.l};
        const T u = w[o + SL_TAU] - damping * dq - m.stiffness[i] * (q - m.rest[i] + dt * dq) -
                    (rev ? dot(a, pa.a) : dot(a, pa.l));
        w[o + SL_U + 0] = U.a.x; w[o + SL_U + 1] = U.a.y; w[o + SL_U + 2] = U.a.z;
        w[o + SL_U + 3] = U.l.x; w[o + SL_U + 4] = U.l.y; w[o + SL_U + 5] = U.l.z;
        w[o + SL_PSI] = psi;
        w[o + SL_UU] = u;
        have_carry = false;
        if (par >= 0) {
            // Pi = IA - U psi U^T ; beta = pa + U psi u
            const V3<T> Ua = psi * U.a, Ul = psi * U.l;
            AiS<T> Pi;
            Pi.A = {IA.A.xx - Ua.x * U.a.x, IA.A.xy - Ua.x * U.a.y, IA.A.xz - Ua.x * U.a.z,
                    IA.A.yy - Ua.y * U.a.y, IA.A.yz - Ua.y * U.a.z, IA.A.zz - Ua.z * U.a.z};
            Pi.C = {IA.C.xx - Ul.x * U.l.x, IA.C.xy - Ul.x * U.l.y, IA.C.xz - Ul.x * U.l.z,
                    IA.C.yy - Ul.y * U.l.y, IA.C.yz - Ul.y * U.l.z, IA.C.zz - Ul.z * U.l.z};
            Pi.B = IA.B - outer(Ua, U.l);
            const T su = psi * u;
            const Sv<T> beta = {pa.a + su * U.a, pa.l + su * U.l};
            // express in the parent frame: rotate by R, then move the reference point by p
            M3<T> R;
            V3<T> p;
            joint_pose_sc(m, i, w[o + SL_S], w[o + SL_C], q, R, p);
            const Sym3<T> A1 = rot_sym(R, Pi.A), C1 = rot_sym(R, Pi.C);
            const M3<T> B1 = mulBt(mul(R, Pi.B), R);
            // P C1 (columns p x col_j(C1)); C1 symmetric
            const V3<T> c0 = cross(p, v3(C1.xx, C1.xy, C1.xz)), c1 = cross(p, v3(C1.xy, C1.yy, C1.yz)),
                        c2 = cross(p, v3(C1.xz, C1.yz, C1.zz));
            const M3<T> PC{{c0.x, c1.x, c2.x, c0.y, c1.y, c2.y, c0.z, c1.z, c2.z}};
            const M3<T> TR = B1 + PC;
            // W = P B1^T : column j = p x row_j(B1)
            const V3<T> w0 = cross(p, row(B1, 0)), w1 = cross(p, row(B1, 1)), w2 = cross(p, row(B1, 2));
            // (P C1) P : row i = row_i(PC) x p
            const V3<T> g0 = cross(row(PC, 0), p), g1 = cross(row(PC, 1), p), g2 = cross(row(PC, 2), p);
            AiS<T> Tp;
            Tp.A = {A1.xx + (w0.x + w0.x) - g0.x, A1.xy + (w1.x + w0.y) - g0.y, A1.xz + (w2.x + w0.z) - g0.z,
                    A1.yy + (w1.y + w1.y) - g1.y, A1.yz + (w2.y + w1.z) - g1.z, A1.zz + (w2.z + w2.z) - g2.z};
            Tp.B = TR;
            Tp.C = C1;
            const V3<T> fl = mul(R, beta.l);
            const Sv<T> Tb = {mul(R, beta.a) + cross(p, fl), fl};
            if (par == i - 1) {
                carry = Tp;
                carry_p = Tb;
                have_carry = true;
            } else {
                const int k = park0 + kSlotsPerBranch * branch_slot[par];
                w[k + 0] += Tp.A.xx; w[k + 1] += Tp.A.xy; w[k + 2] += Tp.A.xz;
                w[k + 3] += Tp.A.yy; w[k + 4] += Tp.A.yz; w[k + 5] += Tp.A.zz;
                w[k + 6] += Tp.C.xx; w[k + 7] += Tp.C.xy; w[k + 8] += Tp.C.xz;
                w[k + 9] += Tp.C.yy; w[k + 10] += Tp.C.yz; w[k + 11] += Tp.C.zz;
                for (int e = 0; e < 9; ++e) w[k + 12 + e] += Tp.B.m[e];
                w[k + 21] += Tb.a.x; w[k + 22] += Tb.a.y; w[k + 23] += Tb.a.z;
                w[k + 24] += Tb.l.x; w[k + 25] += Tb.l.y; w[k + 26] += Tb.l.z;
            }
        }
    }

    // ---- pass 3: accelerations, root to leaves (the V slots are overwritten by spatial accelerations) ----
    const V3<T> g_base = mulT(ld9(m.baseR), prm.g(m));
    for (int i = 0; i < nq; ++i) {
        const int o = kSlotsPerBody * i, par = m.parent[i];
        const bool rev = m.jtype[i] == kRevolute;
        const V3<T> a = ld3(m.axis[i]);
        const T q = w[o + SL_Q], dq = w[o + SL_DQ];
        M3<T> R;
        V3<T> p;
        joint_pose_sc(m, i, w[o + SL_S], w[o + SL_C], q, R, p);
        Sv<T> Ap = {v3(T(0), T(0), T(0)), T(-1) * g_base};  // fictitious base acceleration -g
        if (par >= 0) {
            const int op = kSlotsPerBody * par + SL_V;
            Ap = {{w[op], w[op + 1], w[op + 2]}, {w[op + 3], w[op + 4], w[op + 5]}};
        }
        const Sv<T> ap = {mulT(R, Ap.a), mulT(R, Ap.l + cross(Ap.a, p))};
        const Sv<T> V = {{w[o + SL_V], w[o + SL_V + 1], w[o + SL_V + 2]},
                         {w[o + SL_V + 3], w[o + SL_V + 4], w[o + SL_V + 5]}};
        const V3<T> sd = dq * a;
        Sv<T> acc = ap;
        if (rev) {
            acc.a = acc.a + cross(V.a, sd);
            acc.l = acc.l + cross(V.l, sd);
        } else {
            acc.l = acc.l + cross(V.a, sd);
        }
        const V3<T> Ua = {w[o + SL_U], w[o + SL_U + 1], w[o + SL_U + 2]};
        const V3<T> Ul = {w[o + SL_U + 3], w[o + SL_U + 4], w[o + SL_U + 5]};
        const T ddq = w[o + SL_PSI] * (w[o + SL_UU] - dot(Ua, ap.a) - dot(Ul, ap.l));
        if (rev) acc.a = acc.a + ddq * a;
        else acc.l = acc.l + ddq * a;
        w[o + SL_V + 0] = acc.a.x; w[o + SL_V + 1] = acc.a.y; w[o + SL_V + 2] = acc.a.z;
        w[o + SL_V + 3] = acc.l.x; w[o + SL_V + 4] = acc.l.y; w[o + SL_V + 5] = acc.l.z;
        w[o + SL_TAU] = ddq;
    }
}

// ---------------------------------------------------------------------------------------------------------
// Joint-space constraint stage on the quantities forward_dynamics_fast left in scratch.
//
// DART's ConstraintSolver (not in the reference tree) treats joint limits, joint Coulomb friction and velocity
// servos as 1-D rows on joint velocities and solves a boxed LCP  w = A lambda + b  with A = rows/cols of M^-1,
// obtained by applying unit impulses through the articulated-body recursion (computeImpulseForwardDynamics).
// The same recursion is used here: the U / psi of every body are still in scratch, so one impulse response
// costs two light sweeps over the tree. It uses the articulated inertias WITHOUT the implicit damping / spring
// terms, which equal the stored ones only when every joint has zero damping and stiffness: callers must use
// the dense M^-1 path (b2_kernels.cuh joint_constraints) otherwise, or when more than kMaxRows rows are active.
constexpr int kMaxRows = 4;

// Solves M dv = Lambda for an impulse vector that is non-zero on at most kMaxRows joints. On return the joint
// velocity changes are in the SL_UU slots. Uses the V slots as workspace (they hold nothing needed any more).
template <typename T, typename W>
B2_HD void impulse_response(const ModelDev<T>& m, const W& w, int nr, const int* row_joint, const T* lambda)
{
    const int nq = m.nq;
    for (int i = 0; i < nq; ++i)
        for (int k = 0; k < 6; ++k) w[kSlotsPerBody * i + SL_V + k] = T(0);
    // leaves to root: bias impulses
    for (int i = nq - 1; i >= 0; --i) {
        const int o = kSlotsPerBody * i, par = m.parent[i];
        const bool rev = m.jtype[i] == kRevolute;
        const V3<T> a = ld3(m.axis[i]);
        const Sv<T> P = {{w[o + SL_V], w[o + SL_V + 1], w[o + SL_V + 2]}, {w[o + SL_V + 3], w[o + SL_V + 4], w[o + SL_V + 5]}};
        T L = T(0);
        for (int r = 0; r < kMaxRows; ++r)
            if (r < nr && row_joint[r] == i) L += lambda[r];
        const T u = L - (rev ? dot(a, P.a) : dot(a, P.l));
        w[o + SL_UU] = u;
        if (par >= 0) {
            const T su = w[o + SL_PSI] * u;
            const Sv<T> Q = {P.a + su * v3(w[o + SL_U], w[o + SL_U + 1], w[o + SL_U + 2]),
                             P.l + su * v3(w[o + SL_U + 3], w[o + SL_U + 4], w[o + SL_U + 5])};
            M3<T> R;
            V3<T> p;
            joint_pose_sc(m, i, w[o + SL_S], w[o + SL_C], w[o + SL_Q], R, p);
            const V3<T> fl = mul(R, Q.l);
            const V3<T> na = mul(R, Q.a) + cross(p, fl);
            const int op = kSlotsPerBody * par + SL_V;
            w[op + 0] += na.x; w[op + 1] += na.y; w[op + 2] += na.z;
            w[op + 3] += fl.x; w[op + 4] += fl.y; w[op + 5] += fl.z;
        }
    }
    // root to leaves: velocity changes
    for (int i = 0; i < nq; ++i) {
        const int o = kSlotsPerBody * i, par = m.parent[i];
        const bool rev = m.jtype[i] == kRevolute;
        const V3<T> a = ld3(m.axis[i]);
        Sv<T> dv = sv_zero<T>();
        if (par >= 0) {
            const int op = kSlotsPerBody * par + SL_V;
            const Sv<T> D = {{w[op], w[op + 1], w[op + 2]}, {w[op + 3], w[op + 4], w[op + 5]}};
            M3<T> R;
            V3<T> p;
            joint_pose_sc(m, i, w[o + SL_S], w[o + SL_C], w[o + SL_Q], R, p);
            dv = {mulT(R, D.a), mulT(R, D.l + cross(D.a, p))};
        }
        const T ddv = w[o + SL_PSI] * (w[o + SL_UU] - dot(v3(w[o + SL_U], w[o + SL_U + 1], w[o + SL_U + 2]), dv.a) -
                                        dot(v3(w[o + SL_U + 3], w[o + SL_U + 4], w[o + SL_U + 5]), dv.l));
        if (rev) dv.a = dv.a + ddv * a;
        else dv.l = dv.l + ddv * a;
        w[o + SL_V + 0] = dv.a.x; w[o + SL_V + 1] = dv.a.y; w[o + SL_V + 2] = dv.a.z;
        w[o + SL_V + 3] = dv.l.x; w[o + SL_V + 4] = dv.l.y; w[o + SL_V + 5] = dv.l.z;
        w[o + SL_UU] = ddv;
    }
}

// Collects the active rows (joint, b, lo, hi). Returns the row count, or -1 when more than kMaxRows are active.
// servo_bits: joints under a velocity servo (VelocityFollowerDart), servo_target: their target velocities.
template <typename T, typename W, typename P = NominalParams<T>>
B2_HD int collect_rows(const ModelDev<T>& m, T dt, const W& w, unsigned servo_bits, const T* servo_target,
                       int* rj, T* rb, T* rlo, T* rhi, const P& prm = P())
{
    int nr = 0;
    const T inf = T(INFINITY);
    for (int j = 0; j < m.nq; ++j) {
        const T q = w[kSlotsPerBody * j + SL_Q], dq = w[kSlotsPerBody * j + SL_DQ];
        if ((servo_bits >> j) & 1u) {
            if (nr >= kMaxRows) return -1;
            rj[nr] = j; rb[nr] = dq - servo_target[j]; rlo[nr] = -m.effort[j] * dt; rhi[nr] = m.effort[j] * dt; ++nr;
            continue;
        }
        const T friction = prm.friction(m, j);
        if (friction != T(0)) {
            if (nr >= kMaxRows) return -1;
            rj[nr] = j; rb[nr] = dq; rlo[nr] = -friction * dt; rhi[nr] = friction * dt; ++nr;
        }
        if (q <= m.lower[j]) {
            if (nr >= kMaxRows) return -1;
            rj[nr] = j; rb[nr] = dq; rlo[nr] = T(0); rhi[nr] = inf; ++nr;
        }
        if (q >= m.upper[j]) {
            if (nr >= kMaxRows) return -1;
            rj[nr] = j; rb[nr] = dq; rlo[nr] = -inf; rhi[nr] = T(0); ++nr;
        }
    }
    return nr;
}

// Boxed LCP on the collected rows by projected Gauss-Seidel, then the velocity correction. dq (SL_DQ) and the
// joint accelerations (SL_TAU) are updated in place.
template <typename T, typename W>
B2_HD void constraints_fast(const ModelDev<T>& m, T dt, const W& w, int nr, const int* rj, const T* rb,
                            const T* rlo, const T* rhi)
{
    T A[kMaxRows * kMaxRows], lam[kMaxRows], unit[kMaxRows];
    for (int a = 0; a < kMaxRows; ++a) lam[a] = T(0);
    for (int a = 0; a < nr; ++a) {
        for (int r = 0; r < kMaxRows; ++r) unit[r] = r == a ? T(1) : T(0);
        impulse_response(m, w, nr, rj, unit);
        for (int c = 0; c < nr; ++c) A[c * kMaxRows + a] = w[kSlotsPerBody * rj[c] + SL_UU];
    }
    for (int it = 0; it < (nr == 1 ? 1 : 200); ++it) {  // a single row is solved exactly by one projection
        T change = T(0);
        for (int a = 0; a < nr; ++a) {
            T r = rb[a];
            for (int c = 0; c < nr; ++c) r += A[a * kMaxRows + c] * lam[c];
            T nl = lam[a] - r / A[a * kMaxRows + a];
            nl = nl < rlo[a] ? rlo[a] : (nl > rhi[a] ? rhi[a] : nl);
            change += fabs(nl - lam[a]);
            lam[a] = nl;
        }
        if (change < T(1e-18)) break;
    }
    impulse_response(m, w, nr, rj, lam);
    for (int j = 0; j < m.nq; ++j) {
        const int o = kSlotsPerBody * j;
        const T dv = w[o + SL_UU];
        w[o + SL_DQ] += dv;
        w[o + SL_TAU] += dv / dt;
    }
}

// Zero the parking slots (call before forward_dynamics_fast).
template <typename T, typename W>
B2_HD void clear_parking_t(int nq, int nbranch, const W& w)
{
    const int park0 = kSlotsPerBody * nq;
    for (int k = 0; k < kSlotsPerBranch * nbranch; ++k) w[park0 + k] = T(0);
}
template <typename T, int S>
B2_HD void clear_parking(int nq, int nbranch, const Scratch<T, S>& w) { clear_parking_t<T>(nq, nbranch, w); }

}  // namespace b2
