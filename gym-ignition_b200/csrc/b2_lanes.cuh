// Lane-parallel rigid-body step for fixed-base trees of 1-DoF joints: G lanes of a warp share one env.
//
// What it replaces: the same reference arithmetic as b2_tree_fast.hpp (cpp/scenario/plugins/Physics/Physics.cpp:1824-1835
// -> dartsim World::step; JointController.cpp:289-331 for the PID), organised for small batches (BASELINE configs 4 and 5:
// 16,384 / 4,096 envs per GPU) where one thread per env leaves most schedulers with one warp and the step time is one
// env's dependent instruction chain. Here an env's step is spread over G lanes (G = 8, 10 or 16 >= number of bodies;
// 10 for the 9-DoF Panda: three envs per warp):
//
//   * every quantity is expressed in ONE frame (world orientation, origin at the model's base), so nothing has to be
//     transformed between bodies: velocities, velocity-product accelerations, composite inertias and forces are plain
//     prefix / suffix sums over the tree;
//   * lane = body for everything that is local to a body (sine / cosine, joint placement, world-frame inertia, bias
//     force, the body's row of the mass matrix, PID); lane = row of the rotation for the forward kinematics; lane =
//     component (6 spatial components, 10 inertia parameters) for the sums over the tree;
//   * forward dynamics = composite-rigid-body mass matrix + bias forces (recursive Newton-Euler in the common frame) +
//     an LDL^T factorisation with lane = row kept in registers and one published column per elimination step;
//     DART's implicit joint damping / spring enters as (M + dt D + dt^2 K) ddq = tau - h - D dq - K (q - q0 + dt dq),
//     which is what the articulated-body recursion with psi = (S'AS + dt D + dt^2 K)^-1 solves;
//   * lanes exchange data through a per-env strip of shared memory (< 2 KB) and warp shuffles; the only block-level
//     barrier follows the staging of the model constants.
//
// A rigid body's (and a rigid sub-tree's) spatial inertia about the common origin has 10 parameters
// (rotational inertia about the origin: 6, first moment m c: 3, mass: 1) and is additive over bodies.
//
// Loops over bodies are unrolled over the lane count with a uniform `i < nq` guard: body indices, parents (4 bits each
// in two kernel-parameter words) and shared-memory offsets are then compile-time or uniform values.
#pragma once

#include "b2_kernels.cuh"

// -DB2_LANES_MARKERS puts a PMTRIG instruction at every phase boundary, so that an ncu source-page dump can be cut into
// phases (scripts/ncu_phases.py); off in the shipped build.
#if defined(B2_LANES_MARKERS)
#define B2_MARK(n) asm volatile("pmevent %0;" ::"n"(n))
#else
#define B2_MARK(n)
#endif

namespace b2 {

// Tree structure in kernel parameters: parent + 1 of body i in 4 bits (0 = child of the base), joint types as a bit mask.
struct TreeBits {
    unsigned p_lo, p_hi;   // bodies 0-7, 8-15
    unsigned rev_mask;
    int nq;
    unsigned short anc[16];  // bit j of anc[i]: body j is i or one of its ancestors (filled by make_tree_bits)
};
__host__ __device__ __forceinline__ int tb_parent(const TreeBits& t, int i)
{
    return (int)(((i < 8 ? t.p_lo : t.p_hi) >> (4 * (i & 7))) & 15u) - 1;
}

inline TreeBits make_tree_bits(int nq, const int* parent, const int* jtype)
{
    TreeBits t{0u, 0u, 0u, nq, {0}};
    for (int i = 0; i < nq; ++i) {
        (i < 8 ? t.p_lo : t.p_hi) |= (unsigned)(parent[i] + 1) << (4 * (i & 7));
        if (jtype[i] == kRevolute) t.rev_mask |= 1u << i;
        for (int j = i; j >= 0; j = parent[j]) t.anc[i] |= (unsigned short)(1u << j);
    }
    return t;
}

constexpr int cmax(int a, int b) { return a > b ? a : b; }

// Shared-memory strip of one env, in scalars. Regions are reused phase by phase:
//   P1: joint placements [NB][12] -> body / composite inertias [NB][10] -> LDL^T exchange (two published columns + L^T)
//       -> observation row
//   S : joint motion subspaces [NB][6]            } together: world placements [NB][12] while the forward kinematics runs
//   V : velocities -> accelerations -> forces [NB][6] }
template <int G>
struct LaneLayout {
    static constexpr int NB = G;
    static constexpr int envs_per_warp = 32 / G;
    // placements take 12 scalars per body at a stride of 14, records of the model constants 32 at a stride of 34: a lane
    // stride of 24 (or 64) 4-byte words would put the lanes of an env on 4 (or 1) bank groups; 28 and 68 spread them over 8
    static constexpr int PL = 14;
    static constexpr int REC = LT_SIZE + 2;
    static constexpr int p1_size = cmax(cmax(NB * PL, NB * NB + 2 * NB), 2 * ((kPandaObs + 2) / 2));
    static constexpr int oP1 = 0;
    static constexpr int oS = p1_size;
    static constexpr int oV = oS + NB * 7;
    static constexpr int oEnd = oV + NB * 7;
    // stride = 6 (mod 16) scalars: the envs of a warp start in different banks; even, so 16-byte accesses stay aligned
    static constexpr int stride = oEnd + ((6 - oEnd % 16) + 16) % 16;
    static constexpr int oCol = 0;             // two published columns [2][NB]
    static constexpr int oLT = 2 * NB;         // L^T [NB][NB]: LT[k][i] = l_ik
    static constexpr int table = NB * REC;     // per-block copy of the packed model constants
};

template <typename T> struct Pair;
template <> struct Pair<double> { using type = double2; };
template <> struct Pair<float> { using type = float2; };

template <typename T> __device__ __forceinline__ void ld2(const T* p, T& a, T& b)
{
    const typename Pair<T>::type v = *reinterpret_cast<const typename Pair<T>::type*>(p);
    a = v.x; b = v.y;
}
template <typename T> __device__ __forceinline__ void st2(T* p, T a, T b)
{
    typename Pair<T>::type v;
    v.x = a; v.y = b;
    *reinterpret_cast<typename Pair<T>::type*>(p) = v;
}
template <typename T> __device__ __forceinline__ void ld6(const T* p, T* o)
{
    ld2(p, o[0], o[1]); ld2(p + 2, o[2], o[3]); ld2(p + 4, o[4], o[5]);
}
template <typename T> __device__ __forceinline__ void st6(T* p, const T* o)
{
    st2(p, o[0], o[1]); st2(p + 2, o[2], o[3]); st2(p + 4, o[4], o[5]);
}
template <typename T> __device__ __forceinline__ T dot6(const T* a, const T* b)
{
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3] + a[4] * b[4] + a[5] * b[5];
}

// Spatial inertia about the common origin, 10 parameters: A (xx, xy, xz, yy, yz, zz), m c (x, y, z), m.
// y = I x for a motion vector x = (w, v): moment n = A w + mc x v, force f = m v - mc x w.
template <typename T> __device__ __forceinline__ void inertia_mul(const T* I, const T* x, T* y)
{
    const V3<T> w = v3(x[0], x[1], x[2]), v = v3(x[3], x[4], x[5]), mc = v3(I[6], I[7], I[8]);
    const V3<T> n = v3(I[0] * w.x + I[1] * w.y + I[2] * w.z, I[1] * w.x + I[3] * w.y + I[4] * w.z,
                       I[2] * w.x + I[4] * w.y + I[5] * w.z) + cross(mc, v);
    const V3<T> f = I[9] * v - cross(mc, w);
    y[0] = n.x; y[1] = n.y; y[2] = n.z; y[3] = f.x; y[4] = f.y; y[5] = f.z;
}

// Per-lane context of the lane-parallel routines (always inlined: it must stay in registers).
template <typename T, int G>
struct LaneCtx {
    T* sm;          // the env's strip
    const T* tab;   // the lane's record of the packed model constants (shared memory)
    int slot;       // env slot inside the warp
    int l;          // lane inside the env (>= G on the idle lanes of a warp when 32 % G != 0)
    int nq;
    bool body;      // the lane owns body / joint l of a live env
    bool live;      // the env exists
    TreeBits tb;
    unsigned anc;   // bit j: body j is l or one of its ancestors
};

struct NoStaging {
    __device__ void operator()() const {}
};

// Stages the packed model constants into shared memory (all threads of the block), then waits for the previous grid on
// the stream. `also`: further staging by the block's threads, published with the table by the same block barrier.
// Programmatic dependent launch (the launcher sets the stream-serialization attribute): the next step's blocks are
// scheduled while this grid drains and stage the model constants (written at set-up, never by a step) before they wait
// for the previous step's state. Without the attribute both griddepcontrol instructions are no-ops.
template <typename T, int G, typename Also = NoStaging>
__device__ __forceinline__ void lanes_stage_table_then_wait(const LaneTable<T>* __restrict__ lane_table, T* table,
                                                            Also also = Also())
{
    asm volatile("griddepcontrol.launch_dependents;");
    also();
    using V = typename Pair<T>::type;
    const V* src = reinterpret_cast<const V*>(lane_table);
    V* dst = reinterpret_cast<V*>(table);
    for (int k = threadIdx.x; k < G * LT_SIZE / 2; k += blockDim.x)
        dst[(k / (LT_SIZE / 2)) * (LaneLayout<G>::REC / 2) + (k % (LT_SIZE / 2))] = __ldg(src + k);
    __syncthreads();
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ---- phase A: sine / cosine and joint placement of the lane's joint -> P1[l][12] -------------------------------------
template <typename T, int G>
__device__ __forceinline__ void lanes_joint_placement(const LaneCtx<T, G>& c, T q)
{
    using L = LaneLayout<G>;
    if (c.body) {
        const T* t = c.tab;
        T R0[9], p0[3], ax[3];
#pragma unroll
        for (int k = 0; k < 8; k += 2) ld2(t + LT_R + k, R0[k], R0[k + 1]);
        ld2(t + LT_R + 8, R0[8], p0[0]);
        ld2(t + LT_P + 1, p0[1], p0[2]);
        ld2(t + LT_AXIS, ax[0], ax[1]);
        ax[2] = t[LT_AXIS + 2];
        T* jt = c.sm + L::oP1 + L::PL * c.l;
        if ((c.tb.rev_mask >> c.l) & 1u) {
            T s, co;
            sincos_t(q, &s, &co);
            T R[9];
            if (ax[2] == T(1)) {  // rotation about the joint z axis (every Panda arm joint): the first two columns of R0 mix
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    R[3 * r] = co * R0[3 * r] + s * R0[3 * r + 1];
                    R[3 * r + 1] = co * R0[3 * r + 1] - s * R0[3 * r];
                    R[3 * r + 2] = R0[3 * r + 2];
                }
            } else {
                const T v = T(1) - co;
                const T Rq[9] = {co + v * ax[0] * ax[0], v * ax[0] * ax[1] - s * ax[2], v * ax[0] * ax[2] + s * ax[1],
                                 v * ax[0] * ax[1] + s * ax[2], co + v * ax[1] * ax[1], v * ax[1] * ax[2] - s * ax[0],
                                 v * ax[0] * ax[2] - s * ax[1], v * ax[1] * ax[2] + s * ax[0], co + v * ax[2] * ax[2]};
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int k = 0; k < 3; ++k)
                        R[3 * r + k] = R0[3 * r] * Rq[k] + R0[3 * r + 1] * Rq[3 + k] + R0[3 * r + 2] * Rq[6 + k];
            }
            st2(jt + 0, R[0], R[1]); st2(jt + 2, R[2], R[3]); st2(jt + 4, R[4], R[5]);
            st2(jt + 6, R[6], R[7]); st2(jt + 8, R[8], p0[0]); st2(jt + 10, p0[1], p0[2]);
        } else {
            const T d0 = q * ax[0], d1 = q * ax[1], d2 = q * ax[2];
            st2(jt + 0, R0[0], R0[1]); st2(jt + 2, R0[2], R0[3]); st2(jt + 4, R0[4], R0[5]);
            st2(jt + 6, R0[6], R0[7]);
            st2(jt + 8, R0[8], p0[0] + R0[0] * d0 + R0[1] * d1 + R0[2] * d2);
            st2(jt + 10, p0[1] + R0[3] * d0 + R0[4] * d1 + R0[5] * d2, p0[2] + R0[6] * d0 + R0[7] * d1 + R0[8] * d2);
        }
    }
    __syncwarp();
}

// ---- phase B: forward kinematics, one lane per row of the orientations (and component of the origins) ------------------
// The 3 * EPW lowest lanes of the warp do it (lane f: env slot f / 3, row f % 3), not lanes 0-2 of each env: they then sit
// in one half-warp and their 16-byte broadcast loads cost one shared-memory wavefront instead of two.
// In: P1[i][12] joint placements. Out: (S|V)[i][4 r + c] = R_i[r][c] (c < 3), origin_i[r] (c = 3); origin relative to the base.
template <typename T, int G>
__device__ __forceinline__ void lanes_forward_kinematics(const LaneCtx<T, G>& c, const ModelDev<T>& m, T* warp_strips, int live_envs,
                                                         int nbodies = kMaxDofs)
{
    using L = LaneLayout<G>;
    const int f = threadIdx.x & 31, fs = f / 3, r = f - 3 * fs;
    if (fs < live_envs) {
        T* const sm = warp_strips + fs * L::stride;
        const T b0 = m.baseR[3 * r], b1 = m.baseR[3 * r + 1], b2 = m.baseR[3 * r + 2];
        T r0 = b0, r1 = b1, r2 = b2, pp = T(0);
        T* const out = sm + L::oS + 4 * r;
        const T* const jt0 = sm + L::oP1;
#pragma unroll
        for (int i = 0; i < G; ++i) {
            if (i < c.nq && i < nbodies) {
                const int par = tb_parent(c.tb, i);
                if (par != i - 1) {
                    if (par < 0) { r0 = b0; r1 = b1; r2 = b2; pp = T(0); }
                    else { ld2(out + L::PL * par, r0, r1); ld2(out + L::PL * par + 2, r2, pp); }
                }
                const T* jt = jt0 + L::PL * i;
                T a[12];
                ld2(jt, a[0], a[1]); ld2(jt + 2, a[2], a[3]); ld2(jt + 4, a[4], a[5]);
                ld2(jt + 6, a[6], a[7]); ld2(jt + 8, a[8], a[9]); ld2(jt + 10, a[10], a[11]);
                const T n0 = r0 * a[0] + r1 * a[3] + r2 * a[6];
                const T n1 = r0 * a[1] + r1 * a[4] + r2 * a[7];
                const T n2 = r0 * a[2] + r1 * a[5] + r2 * a[8];
                pp = pp + r0 * a[9] + r1 * a[10] + r2 * a[11];
                r0 = n0; r1 = n1; r2 = n2;
                st2(out + L::PL * i, r0, r1);
                st2(out + L::PL * i + 2, r2, pp);
            }
        }
    }
    __syncwarp();
}

// The lane's world placement from the forward-kinematics output.
template <typename T, int G>
__device__ __forceinline__ void lanes_load_placement(const LaneCtx<T, G>& c, T* R, V3<T>& p)
{
    using L = LaneLayout<G>;
    const T* rp = c.sm + L::oS + L::PL * c.l;
    ld2(rp + 0, R[0], R[1]); ld2(rp + 2, R[2], p.x);
    ld2(rp + 4, R[3], R[4]); ld2(rp + 6, R[5], p.y);
    ld2(rp + 8, R[6], R[7]); ld2(rp + 10, R[8], p.z);
}

// World axis of the lane's joint, R axis, from its body's world orientation R.
template <typename T, int G>
__device__ __forceinline__ V3<T> lanes_joint_axis(const LaneCtx<T, G>& c, const T* R)
{
    const T* t = c.tab;
    return v3(R[0] * t[LT_AXIS] + R[1] * t[LT_AXIS + 1] + R[2] * t[LT_AXIS + 2],
              R[3] * t[LT_AXIS] + R[4] * t[LT_AXIS + 1] + R[5] * t[LT_AXIS + 2],
              R[6] * t[LT_AXIS] + R[7] * t[LT_AXIS + 1] + R[8] * t[LT_AXIS + 2]);
}

// A point given at x in a body's frame, placed from the body's world placement (R, p): p + R x.
template <typename T>
__device__ __forceinline__ V3<T> place_point(const T* R, const V3<T>& p, const T* x)
{
    return v3(p.x + R[0] * x[0] + R[1] * x[1] + R[2] * x[2], p.y + R[3] * x[0] + R[4] * x[1] + R[5] * x[2],
              p.z + R[6] * x[0] + R[7] * x[1] + R[8] * x[2]);
}

// Sum over the tree towards the leaves (lane = component): x_i += x_parent(i), roots start from `root`.
// `mine` points at the lane's component of body 0; PER scalars per body.
template <typename T, int G, int PER>
__device__ __forceinline__ void lanes_prefix(const TreeBits& tb, T* mine, T root)
{
    T run = T(0);
#pragma unroll
    for (int i = 0; i < G; ++i) {
        if (i < tb.nq) {
            const int par = tb_parent(tb, i);
            T up = run;
            if (par < 0) up = root;
            else if (par != i - 1) up = mine[PER * par];
            run = up + mine[PER * i];
            mine[PER * i] = run;
        }
    }
}
// Sum over the tree towards the root (lane = component): x_parent(i) += x_i.
template <typename T, int G, int PER>
__device__ __forceinline__ void lanes_suffix(const TreeBits& tb, T* mine)
{
    T carry = T(0);
    bool have = false;
#pragma unroll
    for (int i = G - 1; i >= 0; --i) {
        if (i < tb.nq) {
            const int par = tb_parent(tb, i);
            T tot = mine[PER * i];
            if (have) {
                tot += carry;
                mine[PER * i] = tot;
            }
            have = par == i - 1 && par >= 0;
            carry = tot;
            if (!have && par >= 0) mine[PER * par] += tot;
        }
    }
}

// The lane's share of its env's rows of per-env parameters (k_run_tree_lanes<ENV>, EnvRows in b2_kernels.cuh): its body's
// inertia record (mass, com, inertia about the com: 10 scalars, 16-byte aligned in fp64), its joint's damping and Coulomb
// friction, the env's gravity.
template <typename T>
struct LaneRows {
    const T* body = nullptr;
    const T* joint = nullptr;
    const T* g = nullptr;
};

// ---- forward dynamics of one env on its G lanes ----------------------------------------------------------------------
// In: q, dq, tau of the lane's joint; (S|V) = world placements (lanes_forward_kinematics). Returns ddq of the lane's joint.
// ENV: inertia, damping and gravity come from `env` instead of the packed model constants.
template <typename T, int G, bool ENV = false>
__device__ __forceinline__ T lanes_forward_dynamics(const LaneCtx<T, G>& c, const ModelDev<T>& m, T dt, T q, T dq, T tau,
                                                    T* inv_d_out = nullptr, const LaneRows<T>& env = LaneRows<T>())
{
    using L = LaneLayout<G>;
    constexpr int NB = G;
    T* const P1 = c.sm + L::oP1;
    T* const PS = c.sm + L::oS;
    T* const PV = c.sm + L::oV;
    T* const myS = PS + 6 * c.l;
    T* const myV = PV + 6 * c.l;
    T* const myI = P1 + 10 * c.l;
    const bool rev = (c.tb.rev_mask >> c.l) & 1u;
    T S[6], I[10], Sdq[6];
    // ---- C: motion subspace and spatial inertia of the lane's body in the common frame ----
    if (c.body) {
        const T* t = c.tab;
        T R[9];
        V3<T> p;
        lanes_load_placement(c, R, p);
        T ax0, ax1, ax2, mass, ic[6], cm[3];
        ld2(t + LT_AXIS, ax0, ax1);
        if constexpr (ENV) {  // mass, com (3), inertia about the com (6)
            const T* r = env.body;
            ax2 = t[LT_AXIS + 2];
            ld2(r, mass, cm[0]); ld2(r + 2, cm[1], cm[2]);
            ld2(r + 4, ic[0], ic[1]); ld2(r + 6, ic[2], ic[3]); ld2(r + 8, ic[4], ic[5]);
        } else {
            ld2(t + LT_AXIS + 2, ax2, mass);
            ld2(t + LT_ICOM, ic[0], ic[1]); ld2(t + LT_ICOM + 2, ic[2], ic[3]); ld2(t + LT_ICOM + 4, ic[4], ic[5]);
            ld2(t + LT_COM, cm[0], cm[1]);
            cm[2] = t[LT_COM + 2];
        }
        const V3<T> aw = v3(R[0] * ax0 + R[1] * ax1 + R[2] * ax2, R[3] * ax0 + R[4] * ax1 + R[5] * ax2,
                            R[6] * ax0 + R[7] * ax1 + R[8] * ax2);
        if (rev) {
            const V3<T> lin = cross(p, aw);
            S[0] = aw.x; S[1] = aw.y; S[2] = aw.z; S[3] = lin.x; S[4] = lin.y; S[5] = lin.z;
        } else {
            S[0] = S[1] = S[2] = T(0); S[3] = aw.x; S[4] = aw.y; S[5] = aw.z;
        }
        const V3<T> cw = place_point(R, p, cm);
        const Sym3<T> Iw = rot_sym(M3<T>{{R[0], R[1], R[2], R[3], R[4], R[5], R[6], R[7], R[8]}},
                                   Sym3<T>{ic[0], ic[1], ic[2], ic[3], ic[4], ic[5]});
        const T cc = dot(cw, cw);
        I[0] = Iw.xx + mass * (cc - cw.x * cw.x);
        I[1] = Iw.xy - mass * (cw.x * cw.y);
        I[2] = Iw.xz - mass * (cw.x * cw.z);
        I[3] = Iw.yy + mass * (cc - cw.y * cw.y);
        I[4] = Iw.yz - mass * (cw.y * cw.z);
        I[5] = Iw.zz + mass * (cc - cw.z * cw.z);
        I[6] = mass * cw.x; I[7] = mass * cw.y; I[8] = mass * cw.z;
        I[9] = mass;
#pragma unroll
        for (int k = 0; k < 6; ++k) Sdq[k] = S[k] * dq;
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) S[k] = Sdq[k] = T(0);
#pragma unroll
        for (int k = 0; k < 10; ++k) I[k] = T(0);
    }
    __syncwarp();  // every lane has read its placement: S and V may be overwritten
    if (c.body) {
        st6(myS, S);
        st6(myV, Sdq);
        st2(myI, I[0], I[1]); st2(myI + 2, I[2], I[3]); st2(myI + 4, I[4], I[5]);
        st2(myI + 6, I[6], I[7]); st2(myI + 8, I[8], I[9]);
    }
    __syncwarp();
    B2_MARK(4);
    // ---- D: velocities V_i = V_parent + S_i dq_i; composite inertias Ic_i = I_i + sum over children ----
    if (c.live && c.l < 6) lanes_prefix<T, G, 6>(c.tb, PV + c.l, T(0));
    if (c.live && c.l < 10) lanes_suffix<T, G, 10>(c.tb, P1 + c.l);
    if (G < 10 && c.live && c.l < 10 - G) lanes_suffix<T, G, 10>(c.tb, P1 + c.l + G);  // 8 lanes: two of them take a second parameter
    __syncwarp();
    B2_MARK(5);
    // ---- E: velocity-product acceleration (V_i x S_i dq_i); force across the joint for a unit acceleration F = Ic S ----
    T V[6], F[6];
    if (c.body) {
        ld6(myV, V);
        const V3<T> w = v3(V[0], V[1], V[2]), v = v3(V[3], V[4], V[5]);
        const V3<T> sw = v3(Sdq[0], Sdq[1], Sdq[2]), sv = v3(Sdq[3], Sdq[4], Sdq[5]);
        const V3<T> ca = cross(w, sw), cl = cross(w, sv) + cross(v, sw);
        const T cd[6] = {ca.x, ca.y, ca.z, cl.x, cl.y, cl.z};
        st6(myV, cd);
        T Ic[10];
        ld2(myI, Ic[0], Ic[1]); ld2(myI + 2, Ic[2], Ic[3]); ld2(myI + 4, Ic[4], Ic[5]);
        ld2(myI + 6, Ic[6], Ic[7]); ld2(myI + 8, Ic[8], Ic[9]);
        inertia_mul(Ic, S, F);
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) V[k] = F[k] = T(0);
    }
    __syncwarp();
    B2_MARK(6);
    // ---- F: accelerations without the joint accelerations, a_i = a_parent + c_i, gravity as base acceleration -g ----
    if (c.live && c.l < 6) lanes_prefix<T, G, 6>(c.tb, PV + c.l, c.l >= 3 ? -(ENV ? env.g[c.l - 3] : m.g[c.l - 3]) : T(0));
    __syncwarp();
    B2_MARK(7);
    // ---- G: net force on the body f = I a + V x* (I V); the lane's row of the mass matrix M[l][j] = F_l . S_j ----
    T D = T(0), K = T(0), rest = T(0);
    if (c.body) {
        T a[6], Ia[6], IV[6];
        ld6(myV, a);
        inertia_mul(I, a, Ia);
        inertia_mul(I, V, IV);
        const V3<T> w = v3(V[0], V[1], V[2]), v = v3(V[3], V[4], V[5]);
        const V3<T> n = v3(IV[0], IV[1], IV[2]), f = v3(IV[3], IV[4], IV[5]);
        const V3<T> bn = cross(w, n) + cross(v, f), bf = cross(w, f);
        const T fo[6] = {Ia[0] + bn.x, Ia[1] + bn.y, Ia[2] + bn.z, Ia[3] + bf.x, Ia[4] + bf.y, Ia[5] + bf.z};
        st6(myV, fo);
        D = ENV ? env.joint[0] : c.tab[LT_DAMPING];
        ld2(c.tab + LT_STIFFNESS, K, rest);
    }
    T row[NB];
    const T diag = dt * D + dt * dt * K;
#pragma unroll
    for (int j = 0; j < NB; ++j) {
        row[j] = T(0);
        if (j < c.nq) {
            T Sj[6];
            ld6(PS + 6 * j, Sj);
            T v = dot6(F, Sj);
            if (j == c.l) v += diag;
            row[j] = ((c.anc >> j) & 1u) ? v : T(0);
        }
    }
    __syncwarp();
    B2_MARK(8);
    // ---- H: forces summed towards the root; bias force of the lane's joint h = S . f ----
    if (c.live && c.l < 6) lanes_suffix<T, G, 6>(c.tb, PV + c.l);
    __syncwarp();
    T rhs = T(0);
    if (c.body) {
        T fs[6];
        ld6(myV, fs);
        rhs = tau - dot6(S, fs) - D * dq - K * (q - rest + dt * dq);
    }
    B2_MARK(9);
    // ---- J: LDL^T with lane = row; column k is published before it is eliminated. Entries right of a lane's diagonal
    // are never read, so the elimination runs unpredicated on them. ----
    T* const col = P1 + L::oCol;
    T* const LT = P1 + L::oLT;
    T inv_d = T(0);
    const int lc = c.l < NB ? c.l : 0;  // idle lanes publish into slot 0 of nothing they own: guarded below
#pragma unroll
    for (int k = 0; k < NB; ++k) {
        if (k < c.nq) {
            T* ck = col + (k & 1) * NB;
            if (c.body) ck[lc] = row[k];
            __syncwarp();
            // the published column, two entries per load (NB is even; entries left of k are never used)
            T cv[NB];
#pragma unroll
            for (int j = k & ~1; j < NB; j += 2) ld2(ck + j, cv[j], cv[j + 1]);
            const T invd = T(1) / cv[k];
            if (c.l == k) inv_d = invd;
            const T lik = row[k] * invd;
#pragma unroll
            for (int j = k + 1; j < NB; ++j) row[j] -= lik * cv[j];
            row[k] = lik;
            if (c.body && c.l > k) LT[k * NB + c.l] = lik;
        }
    }
    B2_MARK(10);
    // forward substitution L y = rhs, diagonal scaling, back substitution L^T x = z
#pragma unroll
    for (int k = 0; k < NB; ++k) {
        if (k < c.nq) {
            const T yk = __shfl_sync(0xffffffffu, rhs, c.slot * G + k);
            if (c.l > k) rhs -= row[k] * yk;
        }
    }
    T z = rhs * inv_d;
    if (inv_d_out) *inv_d_out = inv_d;
    __syncwarp();  // L^T complete
#pragma unroll
    for (int k = NB - 1; k >= 1; --k) {
        if (k < c.nq) {
            const T xk = __shfl_sync(0xffffffffu, z, c.slot * G + k);
            if (c.body && c.l < k) z -= LT[c.l * NB + k] * xk;
        }
    }
    return z;
}

// ---- inverse dynamics of one env on its G lanes (recursive Newton-Euler in the common frame) -------------------------
// tau = M(q) acc + h(q, dq) under gravity `g`: what ComputedTorqueFixedBase::step evaluates with the controller's own
// gravity (cpp/scenario/controllers/src/ComputedTorqueFixedBase.cpp:312-327). Runs its own joint placement and forward
// kinematics (the controller of the first iteration sees the state BEFORE pending resets are applied, the physics the
// state after them) and leaves the strip's regions free for the forward dynamics that follows.
template <typename T, int G>
__device__ __forceinline__ T lanes_inverse_dynamics(const LaneCtx<T, G>& c, const ModelDev<T>& m, T* warp_strips, int live_envs,
                                                    T q, T dq, T acc, const T* g)
{
    using L = LaneLayout<G>;
    T* const PV = c.sm + L::oV;
    T* const myV = PV + 6 * c.l;
    lanes_joint_placement(c, q);
    lanes_forward_kinematics(c, m, warp_strips, live_envs);
    const bool rev = (c.tb.rev_mask >> c.l) & 1u;
    T S[6], I[10], Sdq[6];
    if (c.body) {
        const T* t = c.tab;
        T R[9];
        V3<T> p;
        lanes_load_placement(c, R, p);
        T ax0, ax1, ax2, mass, ic[6], cm[3];
        ld2(t + LT_AXIS, ax0, ax1);
        ld2(t + LT_AXIS + 2, ax2, mass);
        ld2(t + LT_ICOM, ic[0], ic[1]); ld2(t + LT_ICOM + 2, ic[2], ic[3]); ld2(t + LT_ICOM + 4, ic[4], ic[5]);
        ld2(t + LT_COM, cm[0], cm[1]);
        cm[2] = t[LT_COM + 2];
        const V3<T> aw = v3(R[0] * ax0 + R[1] * ax1 + R[2] * ax2, R[3] * ax0 + R[4] * ax1 + R[5] * ax2,
                            R[6] * ax0 + R[7] * ax1 + R[8] * ax2);
        if (rev) {
            const V3<T> lin = cross(p, aw);
            S[0] = aw.x; S[1] = aw.y; S[2] = aw.z; S[3] = lin.x; S[4] = lin.y; S[5] = lin.z;
        } else {
            S[0] = S[1] = S[2] = T(0); S[3] = aw.x; S[4] = aw.y; S[5] = aw.z;
        }
        const V3<T> cw = place_point(R, p, cm);
        const Sym3<T> Iw = rot_sym(M3<T>{{R[0], R[1], R[2], R[3], R[4], R[5], R[6], R[7], R[8]}},
                                   Sym3<T>{ic[0], ic[1], ic[2], ic[3], ic[4], ic[5]});
        const T cc = dot(cw, cw);
        I[0] = Iw.xx + mass * (cc - cw.x * cw.x);
        I[1] = Iw.xy - mass * (cw.x * cw.y);
        I[2] = Iw.xz - mass * (cw.x * cw.z);
        I[3] = Iw.yy + mass * (cc - cw.y * cw.y);
        I[4] = Iw.yz - mass * (cw.y * cw.z);
        I[5] = Iw.zz + mass * (cc - cw.z * cw.z);
        I[6] = mass * cw.x; I[7] = mass * cw.y; I[8] = mass * cw.z;
        I[9] = mass;
#pragma unroll
        for (int k = 0; k < 6; ++k) Sdq[k] = S[k] * dq;
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) S[k] = Sdq[k] = T(0);
#pragma unroll
        for (int k = 0; k < 10; ++k) I[k] = T(0);
    }
    __syncwarp();  // every lane has read its placement: the V region may be overwritten
    if (c.body) st6(myV, Sdq);
    __syncwarp();
    if (c.live && c.l < 6) lanes_prefix<T, G, 6>(c.tb, PV + c.l, T(0));  // V_i = V_parent + S_i dq_i
    __syncwarp();
    T V[6];
    if (c.body) {
        ld6(myV, V);
        const V3<T> w = v3(V[0], V[1], V[2]), v = v3(V[3], V[4], V[5]);
        const V3<T> sw = v3(Sdq[0], Sdq[1], Sdq[2]), sv = v3(Sdq[3], Sdq[4], Sdq[5]);
        const V3<T> ca = cross(w, sw), cl = cross(w, sv) + cross(v, sw);
        // a_i - a_parent = V_i x S_i dq_i + S_i acc_i
        const T da[6] = {ca.x + S[0] * acc, ca.y + S[1] * acc, ca.z + S[2] * acc, cl.x + S[3] * acc, cl.y + S[4] * acc,
                         cl.z + S[5] * acc};
        st6(myV, da);
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) V[k] = T(0);
    }
    __syncwarp();
    if (c.live && c.l < 6) lanes_prefix<T, G, 6>(c.tb, PV + c.l, c.l >= 3 ? -g[c.l - 3] : T(0));  // gravity as base acceleration
    __syncwarp();
    if (c.body) {
        T a[6], Ia[6], IV[6];
        ld6(myV, a);
        inertia_mul(I, a, Ia);
        inertia_mul(I, V, IV);
        const V3<T> w = v3(V[0], V[1], V[2]), v = v3(V[3], V[4], V[5]);
        const V3<T> n = v3(IV[0], IV[1], IV[2]), f = v3(IV[3], IV[4], IV[5]);
        const V3<T> bn = cross(w, n) + cross(v, f), bf = cross(w, f);
        const T fo[6] = {Ia[0] + bn.x, Ia[1] + bn.y, Ia[2] + bn.z, Ia[3] + bf.x, Ia[4] + bf.y, Ia[5] + bf.z};
        st6(myV, fo);
    }
    __syncwarp();
    if (c.live && c.l < 6) lanes_suffix<T, G, 6>(c.tb, PV + c.l);
    __syncwarp();
    T tau = T(0);
    if (c.body) {
        T fs[6];
        ld6(myV, fs);
        tau = dot6(S, fs);
    }
    __syncwarp();  // the strip is free again
    return tau;
}

// Solves (L D L^T) x = rhs with the factor lanes_forward_dynamics left behind: L^T in the env's strip (LT[k][i] = l_ik),
// the reciprocal of the lane's pivot in `inv_d`. Lane = row; every lane of the warp takes part (shuffles).
template <typename T, int G>
__device__ __forceinline__ T lanes_ldl_solve(const T* LT, T inv_d, int slot, int l, int nq, bool body, T rhs)
{
    constexpr int NB = G;
    const int lc = l < NB ? l : 0;
#pragma unroll
    for (int k = 0; k < NB; ++k) {
        if (k < nq) {
            const T yk = __shfl_sync(0xffffffffu, rhs, slot * G + k);
            if (body && l > k) rhs -= LT[k * NB + lc] * yk;
        }
    }
    T z = rhs * inv_d;
#pragma unroll
    for (int k = NB - 1; k >= 1; --k) {
        if (k < nq) {
            const T xk = __shfl_sync(0xffffffffu, z, slot * G + k);
            if (body && l < k) z -= LT[lc * NB + k] * xk;
        }
    }
    return z;
}

// Constraint stage on lanes (joint limits, Coulomb friction, velocity servo: DART's JointLimit / JointCoulombFriction /
// ServoMotor constraints; same rows, order and projected Gauss-Seidel as joint_constraints / constraints_fast of the thread
// kernels). A gripper resting on its lower limit makes this the common case, so it must not serialise on one lane: the
// rows' columns of M^-1 come from the LDL^T factor of the forward dynamics (one lane-parallel solve per row), the <= 4 x 4
// system is gathered with shuffles and every lane of the env runs the tiny sweep redundantly. Valid when no joint has
// damping or stiffness (the factor is then M's own) and every env of the warp has at most 4 rows; returns false
// (warp-uniform, nothing changed) otherwise and the caller falls back to the dense solve on lane 0.
// flags: f0 = servo or friction row, f1 = lower-limit row, f2 = upper-limit row of the lane's joint.
template <typename T, int G>
__device__ __noinline__ bool lanes_constraints_fast(const T* LT, T inv_d, int slot, int l, int nq, bool body, T dt, bool f0, bool f1,
                                                    bool f2, bool servo, T servo_target, T bound0, bool dk, T* dq_io, T* ddq_io)
{
    constexpr int EPW = 32 / G;
    const unsigned full = 0xffffffffu, env_bits = (1u << G) - 1u;
    if (__ballot_sync(full, dk)) return false;
    const unsigned B0 = __ballot_sync(full, f0), B1 = __ballot_sync(full, f1), B2 = __ballot_sync(full, f2);
    int nrw = 0;
#pragma unroll
    for (int s = 0; s < EPW; ++s) {
        const int n = __popc((B0 >> (s * G)) & env_bits) + __popc((B1 >> (s * G)) & env_bits) + __popc((B2 >> (s * G)) & env_bits);
        nrw = max(nrw, n);
    }
    if (nrw > 4) return false;
    const unsigned b0 = (B0 >> (slot * G)) & env_bits, b1 = (B1 >> (slot * G)) & env_bits, b2 = (B2 >> (slot * G)) & env_bits;
    // the env's rows in the order of joint_constraints: joint by joint, (servo | friction), lower, upper; 8 bits per row
    unsigned packed = 0u;
    int nr = 0;
#pragma unroll
    for (int j = 0; j < G; ++j) {
        if ((b0 >> j) & 1u) { packed |= (unsigned)(j | (0 << 4)) << (8 * nr); ++nr; }
        if ((b1 >> j) & 1u) { packed |= (unsigned)(j | (1 << 4)) << (8 * nr); ++nr; }
        if ((b2 >> j) & 1u) { packed |= (unsigned)(j | (2 << 4)) << (8 * nr); ++nr; }
    }
    T dq = *dq_io, ddq = *ddq_io;
    const T v0 = servo ? dq - servo_target : dq;
    const T inf = T(INFINITY);
    T X[4], A[16], rb[4], rlo[4], rhi[4], lam[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        X[a] = rb[a] = rlo[a] = rhi[a] = lam[a] = T(0);
        if (a < nrw) {  // uniform
            const bool on = a < nr;
            const int j = (packed >> (8 * a)) & 15u, kind = (packed >> (8 * a + 4)) & 3u, src = slot * G + j;
            X[a] = lanes_ldl_solve<T, G>(LT, inv_d, slot, l, nq, body, (on && l == j) ? T(1) : T(0));
            const T rv0 = __shfl_sync(full, v0, src), rdq = __shfl_sync(full, dq, src), rbd = __shfl_sync(full, bound0, src);
            if (on) {
                rb[a] = kind == 0 ? rv0 : rdq;
                rlo[a] = kind == 0 ? -rbd * dt : (kind == 1 ? T(0) : -inf);
                rhi[a] = kind == 0 ? rbd * dt : (kind == 1 ? inf : T(0));
            }
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            A[4 * a + cc] = T(0);
            if (a < nrw && cc < nrw) {  // A[a][c] = (M^-1 e_{j_c})[j_a]
                const T v = __shfl_sync(full, X[cc], slot * G + (int)((packed >> (8 * a)) & 15u));
                if (a < nr && cc < nr) A[4 * a + cc] = v;
            }
        }
    if (nr > 0) {
        // reciprocal effective masses once: an fp64 division costs as much as the rest of a row's update
        T rA[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) rA[a] = a < nr ? T(1) / A[4 * a + a] : T(0);
        for (int it = 0; it < (nr == 1 ? 1 : 200); ++it) {  // a single row is solved exactly by one projection
            T change = T(0);
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                if (a < nr) {
                    T r = rb[a];
#pragma unroll
                    for (int cc = 0; cc < 4; ++cc)
                        if (cc < nr) r += A[4 * a + cc] * lam[cc];
                    T nl = lam[a] - r * rA[a];
                    nl = nl < rlo[a] ? rlo[a] : (nl > rhi[a] ? rhi[a] : nl);
                    change += fabs(nl - lam[a]);
                    lam[a] = nl;
                }
            }
            if (change < T(1e-18)) break;
        }
        T dv = T(0);
#pragma unroll
        for (int a = 0; a < 4; ++a)
            if (a < nr) dv += X[a] * lam[a];
        if (body) {
            *dq_io = dq + dv;
            *ddq_io = ddq + dv / dt;
        }
    }
    return true;
}

// Rare path of the constraint stage: some joint of some env of the warp sits on a limit, has Coulomb friction or is under a
// velocity servo (servo_bits: the env's joints, servo_target: the lane's velocity target). Lane 0
// of each such env runs the dense boxed LCP of the one-thread-per-env kernels on its env (b2_kernels.cuh joint_constraints).
// Everything is passed by value: a reference to the lane context would force it (and the shared-memory pointer in it)
// into local memory for the whole kernel.
// `prm`: the env's EnvParams (k_run_tree_lanes<ENV>), or nothing for the model's tables.
template <typename T, int G, typename... P>
__device__ __noinline__ void lanes_joint_constraints(T* x /* [4][G] exchange strip */, int l, int nq, bool body, bool solve,
                                                     const ModelDev<T>* m, T dt, T q, T* dq_io, T* ddq_io,
                                                     unsigned servo_bits = 0u, T servo_target = T(0), P... prm)
{
    T dq = *dq_io, ddq = *ddq_io;
    __syncwarp();
    if (body) { x[l] = q; x[G + l] = dq; x[2 * G + l] = ddq; x[3 * G + l] = servo_target; }
    __syncwarp();
    if (solve) {
        T qa[kMaxDofs], dqa[kMaxDofs], ddqa[kMaxDofs], target[kMaxDofs];
        uint8_t servo[kMaxDofs];
        for (int j = 0; j < nq; ++j) {
            qa[j] = x[j]; dqa[j] = x[G + j]; ddqa[j] = x[2 * G + j];
            servo[j] = (servo_bits >> j) & 1u;
            target[j] = servo[j] ? x[3 * G + j] : T(0);
        }
        joint_constraints<T, kMaxDofs>(*m, dt, qa, dqa, servo, target, ddqa, prm...);
        for (int j = 0; j < nq; ++j) { x[G + j] = dqa[j]; x[2 * G + j] = ddqa[j]; }
    }
    __syncwarp();
    if (body) { *dq_io = x[G + l]; *ddq_io = x[2 * G + l]; }
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------------------
// Fused Panda task on lanes (BASELINE config 4); same contract as k_task_panda (b2_kernels.cuh): position PID at the
// physics rate -> physics step -> observation [q, dq, end-effector position + quaternion, MIXED Jacobian 6 x (6 + nq)],
// reward, TimeLimit, reset. blockDim.x = 32 * warps, each warp steps 32 / G envs; dynamic shared memory =
// LaneLayout<G>::table + warps * (32 / G) * LaneLayout<G>::stride scalars.
// ---------------------------------------------------------------------------------------------------------------------
// The register allocation is sized for 4 blocks of 128 threads per SM (127 registers, no spills): measured best at 4,096
// and 16,384 envs among budgets of 3 - 6 blocks (5: 96 registers, 6: 80 with ~200 bytes of spills).
// NQ > 0: the tree (joint count NQ, parents P_LO / P_HI, joint types REV, encoded like TreeBits) is a compile-time
// constant: the launcher instantiates the Panda's and dispatches on a match with the loaded model. Every `i < nq` guard,
// parent lookup and chain / branch decision of the unrolled body loops then folds away (about a third of the kernel's
// instructions). NQ = 0 reads the tree from the arguments.
// ENV: the physics reads every env's own inertias, damping, Coulomb friction and gravity from `env_rows`
// (b2sim_enable_env_params), as k_run_tree_lanes<ENV> does; the observation is kinematic and reads none of them.
template <typename T, int G, int NQ, unsigned P_LO, unsigned P_HI, unsigned REV, bool ENV = false>
__global__ void __launch_bounds__(128, 4) k_task_panda_lanes(const ModelDev<T>* __restrict__ tables,
                                                       const LaneTable<T>* __restrict__ lane_table, const PandaArgs<T> a,
                                                       const TreeBits tb_arg, const EnvRows<T> env_rows)
{
    const TreeBits tb = NQ > 0 ? TreeBits{P_LO, P_HI, REV, NQ, {0}} : tb_arg;  // the ancestor masks are read from tb_arg
    using L = LaneLayout<G>;
    constexpr int EPW = L::envs_per_warp;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* const table = reinterpret_cast<T*>(smem_raw);
    T* const strips = table + L::table + 12;
    const ModelDev<T>& m = *tables;
    // the end-effector frame in its body (12 scalars) rides behind the per-body records
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    LaneCtx<T, G> c;
    c.slot = min(lane / G, EPW - 1);
    c.l = lane - c.slot * G;  // lanes past EPW * G (32 % G != 0) idle with l >= G
    c.nq = NQ > 0 ? NQ : a.nq;
    c.tb = tb;
    c.tb.nq = c.nq;
    const int ee_body = a.ee_body;
    const int64_t env0 = ((int64_t)blockIdx.x * warps + warp) * EPW;  // first env of the warp
    const int64_t e = env0 + c.slot;
    c.live = e < a.n;
    c.body = c.live && c.l < c.nq;
    T* const warp_strips = strips + (size_t)(warp * EPW) * L::stride;
    const int live_envs = (int)max((int64_t)0, min((int64_t)EPW, a.n - env0));
    c.sm = warp_strips + c.slot * L::stride;
    const int nq = c.nq, jl = min(c.l, nq - 1);
    c.tab = table + L::REC * jl;
    c.anc = c.l < c.nq ? tb_arg.anc[c.l] : 0u;
    const int nobs = panda_obs_size(nq);
    LaneRows<T> env;
    if constexpr (ENV) {  // pointers only: lanes without a body never dereference theirs
        env.body = env_rows.inertia + (e * nq + jl) * kEnvInertiaCols;
        env.joint = env_rows.dyn + (e * nq + jl) * kEnvJointCols;
        env.g = env_rows.grav + 3 * e;
    }

    lanes_stage_table_then_wait<T, G>(lane_table, table, [&] {
        if (threadIdx.x < 9) table[L::table + threadIdx.x] = m.link_R[a.ee_link][threadIdx.x];
        else if (threadIdx.x < 12) table[L::table + threadIdx.x] = m.link_p[a.ee_link][threadIdx.x - 9];
    });
    T q = T(0), dq = T(0), target = T(0), st[3] = {T(0), T(0), T(0)};
    unsigned el = 0;
    if (c.live && c.l == 0) el = a.elapsed[e];  // needed at the very end: in flight with the state loads
    if (c.body) {
        q = __ldcs(a.state + e * 2 * nq + c.l);
        dq = __ldcs(a.state + e * 2 * nq + nq + c.l);
        target = __ldg(a.targets + e * nq + c.l);
#pragma unroll
        for (int k = 0; k < 3; ++k) st[k] = __ldcs(a.pid_state + e * 3 * nq + 3 * c.l + k);
    }
    B2_MARK(0);
    for (int it = 0; it < a.iterations; ++it) {
        // JointController::PreUpdate: error = current - reference, force = pid.Update(error, dt)
        T tau = T(0);
        if (c.body) tau = pid_update(a.pid[jl], st, q - target, a.dt);
        B2_MARK(1);
        lanes_joint_placement(c, q);
        B2_MARK(2);
        lanes_forward_kinematics(c, m, warp_strips, live_envs);
        B2_MARK(3);
        T inv_d;
        T ddq = lanes_forward_dynamics<T, G, ENV>(c, m, a.dt, q, dq, tau, &inv_d, env);
        dq += ddq * a.dt;
        T env_friction = T(0), env_damping = T(0);  // ENV: the joint's row (read once, used below)
        if (ENV && c.body) { env_damping = env.joint[0]; env_friction = env.joint[1]; }
        const bool f0 = c.body && (ENV ? env_friction : c.tab[LT_FRICTION]) != T(0), f1 = c.body && q <= c.tab[LT_LOWER],
                   f2 = c.body && q >= c.tab[LT_UPPER];
        const unsigned rows = __ballot_sync(0xffffffffu, f0 || f1 || f2);
        if (rows) {
            T dq_io = dq, ddq_io = ddq;  // copies: the out-of-line calls must not pin the kernel's registers to memory
            const bool dk = c.body && ((ENV ? env_damping : c.tab[LT_DAMPING]) != T(0) || c.tab[LT_STIFFNESS] != T(0));
            if (!lanes_constraints_fast<T, G>(c.sm + L::oP1 + L::oLT, inv_d, c.slot, c.l, nq, c.body, a.dt, f0, f1, f2, false, T(0),
                                              ENV ? env_friction : c.tab[LT_FRICTION], dk, &dq_io, &ddq_io)) {
                // ENV: lane 0 solves its env with the env's own inertias and friction (the pack holds its EnvParams)
                const auto dense = [&](auto... prm) {
                    lanes_joint_constraints<T, G>(c.sm + L::oV, c.l, nq, c.body,
                                                  c.l == 0 && ((rows >> (c.slot * G)) & ((1u << G) - 1u)) != 0u, tables, a.dt, q,
                                                  &dq_io, &ddq_io, 0u, T(0), prm...);
                };
                if constexpr (ENV) dense(env_rows.env(e, nq));
                else dense();
            }
            dq = dq_io;
            ddq = ddq_io;
        }
        q += dq * a.dt;
    }
    // ---- observation: kinematics at the new positions ----
    B2_MARK(11);
    {   // joints beyond the end-effector body (the fingers) are not on its chain
        LaneCtx<T, G> co = c;
        co.body = c.body && c.l <= ee_body;
        lanes_joint_placement(co, q);
    }
    B2_MARK(12);
    lanes_forward_kinematics(c, m, warp_strips, live_envs, ee_body + 1);
    B2_MARK(13);
    // an end effector welded to the base (ee_body = -1) has an empty chain: lane 0 places it from the base pose
    const int ee_lane = max(ee_body, 0);
    const unsigned on_chain = ee_body >= 0 ? tb_arg.anc[ee_body] : 0u;
    T* out = c.sm + L::oP1;  // the joint placements are dead once the forward kinematics has run
    V3<T> aw = v3(T(0), T(0), T(0)), po = aw, pe = aw;
    const T bx = m.basep[0], by = m.basep[1], bz = m.basep[2];
    const bool chain_lane = c.body && ((on_chain >> c.l) & 1u);
    if (chain_lane || (c.body && c.l == ee_lane)) {
        T R[9];
        if (chain_lane) {
            lanes_load_placement(c, R, po);
            aw = lanes_joint_axis(c, R);
        } else {
#pragma unroll
            for (int k = 0; k < 9; ++k) R[k] = m.baseR[k];
        }
        if (c.l == ee_lane) {
            const T* ee = table + L::table;  // link_R (9), link_p (3)
            pe = place_point(R, po, ee + 9);
            T E[9];
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int k = 0; k < 3; ++k) E[3 * r + k] = R[3 * r] * ee[k] + R[3 * r + 1] * ee[3 + k] + R[3 * r + 2] * ee[6 + k];
            const int k = 2 * nq;
            out[k + 0] = pe.x + bx; out[k + 1] = pe.y + by; out[k + 2] = pe.z + bz;
            // rotation -> unit quaternion with the branch selection of rot_to_quat (b2_rbd.hpp), one rsqrt instead of a
            // square root and three divisions: 1 + 2 R_kk - tr under the root for the k-major branches
            const T tr = E[0] + E[4] + E[8];
            const int br = tr > T(0) ? 0 : ((E[0] > E[4] && E[0] > E[8]) ? 1 : (E[4] > E[8] ? 2 : 3));
            const T S = T(1) + (br == 0 ? tr : T(2) * (br == 1 ? E[0] : (br == 2 ? E[4] : E[8])) - tr);
            const T ri = rsqrt(S), big = T(0.5) * (S * ri), f = T(0.5) * ri;
            const T d0 = (E[7] - E[5]) * f, d1 = (E[2] - E[6]) * f, d2 = (E[3] - E[1]) * f;
            const T sxy = (E[1] + E[3]) * f, sxz = (E[2] + E[6]) * f, syz = (E[5] + E[7]) * f;
            T qw = br == 0 ? big : (br == 1 ? d0 : (br == 2 ? d1 : d2));
            T qx = br == 0 ? d0 : (br == 1 ? big : (br == 2 ? sxy : sxz));
            T qy = br == 0 ? d1 : (br == 1 ? sxy : (br == 2 ? big : syz));
            T qz = br == 0 ? d2 : (br == 1 ? sxz : (br == 2 ? syz : big));
            if (qw < T(0)) { qw = -qw; qx = -qx; qy = -qy; qz = -qz; }
            out[k + 3] = qw; out[k + 4] = qx; out[k + 5] = qy; out[k + 6] = qz;
        }
    }
    const int src = c.slot * G + ee_lane;
    pe.x = __shfl_sync(0xffffffffu, pe.x, src);
    pe.y = __shfl_sync(0xffffffffu, pe.y, src);
    pe.z = __shfl_sync(0xffffffffu, pe.z, src);
    const int kj = 2 * nq + 7, ncol = 6 + nq;
    int done = 0;
    if (c.body) {
        out[c.l] = q;
        out[nq + c.l] = dq;
        V3<T> lin = v3(T(0), T(0), T(0)), ang = lin;
        if (chain_lane) {
            if ((tb.rev_mask >> c.l) & 1u) { lin = cross(aw, pe - po); ang = aw; }
            else lin = aw;
        }
        T* J = out + kj + 6 + c.l;
        J[0 * ncol] = lin.x; J[1 * ncol] = lin.y; J[2 * ncol] = lin.z;
        J[3 * ncol] = ang.x; J[4 * ncol] = ang.y; J[5 * ncol] = ang.z;
    }
    if (c.live && c.l < 6) {
        // base block of the MIXED Jacobian: [1, -S(p_ee - p_base); 0, 1], row l
        T* Jr = out + kj + c.l * ncol;
#pragma unroll
        for (int k = 0; k < 6; ++k) Jr[k] = k == c.l ? T(1) : T(0);
        if (c.l == 0) { Jr[4] = pe.z; Jr[5] = -pe.y; }
        if (c.l == 1) { Jr[3] = -pe.z; Jr[5] = pe.x; }
        if (c.l == 2) { Jr[3] = pe.y; Jr[4] = -pe.x; }
    }
    if (c.live && c.l == 0) {
        const V3<T> gd = v3(pe.x + bx - a.goal[0], pe.y + by - a.goal[1], pe.z + bz - a.goal[2]);
        const T reward = -sqrt(dot(gd, gd));
        a.reward[e] = reward;
        if (!a.observe_only) el += 1;
        done = !a.observe_only && (int)el >= a.max_episode_steps;  // gym TimeLimit; the task itself never terminates
        a.done[e] = done ? 1 : 0;
        if (a.ep_return && !a.observe_only) {  // episode statistics: one lane per env, plain atomics (b2_kernels.cuh)
            const bool finite = isfinite(reward);
            const T ret = a.ep_return[e] + (finite ? reward : T(0));
            a.ep_return[e] = done ? T(0) : ret;
            double* tot = a.ep_totals + 4 * (blockIdx.x % kStatStripes);
            if (done) { atomicAdd(tot + 0, (double)ret); atomicAdd(tot + 1, (double)el); atomicAdd(tot + 2, 1.0); }
            if (!finite) atomicAdd(tot + 3, 1.0);
        }
        if (done) el = 0;
        a.elapsed[e] = (uint16_t)el;
    }
    done = __shfl_sync(0xffffffffu, done, c.slot * G);
    __syncwarp();
    B2_MARK(14);
    // the observation rows of the warp's envs are contiguous in global memory
    {
        const int nenv = live_envs;
        const T* src = warp_strips + L::oP1;
        T* dst = a.obs + env0 * nobs;
#pragma unroll
        for (int s = 0; s < EPW; ++s) {
            if (s < nenv) {
#pragma unroll 4
                for (int k = lane; k < nobs; k += 32) __stcs(dst + (s * nobs + k), src[s * L::stride + k]);
            }
        }
    }
    B2_MARK(15);
    if (!a.observe_only && c.body) {
        if (done) {  // Task.reset_task + paused run: models/panda.py initial configuration, PID reset
            q = a.q0[jl];
            dq = T(0);
            st[0] = st[1] = st[2] = T(0);
        }
        __stcs(a.state + e * 2 * nq + c.l, q);
        __stcs(a.state + e * 2 * nq + nq + c.l, dq);
#pragma unroll
        for (int k = 0; k < 3; ++k) __stcs(a.pid_state + e * 3 * nq + 3 * c.l + k, st[k]);
    }
}


// ---------------------------------------------------------------------------------------------------------------------
// GazeboSimulator::run on lanes: the generic step of a fixed-base tree (k_run_tree / run_tree_env in b2_kernels.cuh,
// cpp/scenario/gazebo/src/GazeboSimulator.cpp:202-251 -> JointController.cpp:114-331 + Physics.cpp:646-685) for the small
// batches the BASELINE configurations use: lane = joint for the ScenarI/O bookkeeping (PID with the rate gate, pending
// velocity / position resets, command selection, one-shot clearing, readbacks), the lane-parallel forward dynamics for
// the physics iteration, the dense boxed LCP of the thread kernels on lane 0 when a joint row is active (limit, Coulomb
// friction, velocity servo). External link wrenches enter as J^T F from the world placements the forward kinematics
// just produced. Template flags (below) add the computed-torque controller and the coupled-world variant.
// ---------------------------------------------------------------------------------------------------------------------
// CT: the computed-torque controller (ComputedTorqueFixedBase run by ControllerRunner) is active: the torque
//   M(q) (ddq_ref - kp (q - q_ref) - kd (dq - dq_ref)) + h(q, dq) is evaluated by a lane-parallel recursive Newton-Euler pass
//   on the iterations the controller fires on and held in the PID `cmd` slot in between (computed_torque, b2_kernels.cuh).
// COUPLED: the model belongs to a world with contacts (k_coupled_dynamics): the joint rows are solved together with the
//   contacts by k_pgs_solve, so this kernel stops after the unconstrained velocity update, hands dq to the solver (v0),
//   leaves the positions unintegrated and the pending-reset mask in place (k_world_finish integrates and clears it).
// ENV (not with COUPLED): the physics reads every env's own inertias, damping, Coulomb friction and gravity from `rows`
//   (b2sim_enable_env_params); the computed-torque controller keeps the packed nominal constants.
template <typename T, int G, bool CT, bool COUPLED, bool ENV = false>
__global__ void __launch_bounds__(128, 4) k_run_tree_lanes(const ModelDev<T>* __restrict__ tables,
                                                           const LaneTable<T>* __restrict__ lane_table, const RunCfg<T> cfg,
                                                           const RunBuffers<T> b, const TreeBits tb, T* __restrict__ v0, int nvp,
                                                           const EnvRows<T> env_rows)
{
    static_assert(!(ENV && COUPLED), "per-env parameters are not supported in a coupled world");
    using L = LaneLayout<G>;
    constexpr int EPW = L::envs_per_warp;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* const table = reinterpret_cast<T*>(smem_raw);
    T* const strips = table + L::table + 12;
    const ModelDev<T>& m = *tables;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    LaneCtx<T, G> c;
    c.slot = min(lane / G, EPW - 1);
    c.l = lane - c.slot * G;
    c.nq = cfg.nq;
    c.tb = tb;
    c.tb.nq = c.nq;
    const int64_t env0 = ((int64_t)blockIdx.x * warps + warp) * EPW;
    const int64_t e = env0 + c.slot;
    c.live = e < b.n;
    c.body = c.live && c.l < c.nq;
    T* const warp_strips = strips + (size_t)(warp * EPW) * L::stride;
    const int live_envs = (int)max((int64_t)0, min((int64_t)EPW, b.n - env0));
    c.sm = warp_strips + c.slot * L::stride;
    const int nq = c.nq, jl = min(c.l, nq - 1);
    c.tab = table + L::REC * jl;
    c.anc = c.l < c.nq ? tb.anc[c.l] : 0u;

    const int md = cfg.mode[jl];
    const bool pid_mode = md == B2_MODE_POSITION || md == B2_MODE_VELOCITY;
    const bool pid_joint = cfg.controller_loaded && pid_mode;
    const bool control = !cfg.paused && cfg.controller_loaded && pid_mode;
    const bool has_fc = cfg.has_force_cmd[jl] != 0;
    LaneRows<T> env;
    if constexpr (ENV) {  // pointers only: lanes without a body never dereference theirs
        env.body = env_rows.inertia + (e * nq + jl) * kEnvInertiaCols;
        env.joint = env_rows.dyn + (e * nq + jl) * kEnvJointCols;
        env.g = env_rows.grav + 3 * e;
    }
    lanes_stage_table_then_wait<T, G>(lane_table, table);
    T q = T(0), dq = T(0), fc = T(0), ref = T(0), vel_t = T(0), st[3] = {T(0), T(0), T(0)};
    T ct_pos = T(0), ct_vel = T(0), ct_acc = T(0), ct_tau = T(0);
    const bool ct = CT && !cfg.paused && cfg.ct_active;
    uint32_t mask = 0u;
    if (c.live) mask = b.reset_mask[e];
    if (c.body) {
        q = b.state[e * 2 * nq + c.l];
        dq = b.state[e * 2 * nq + nq + c.l];
        if (has_fc) fc = b.force_cmd[e * nq + c.l];
        if (CT && ct) {
            ct_pos = b.pos_target[e * nq + c.l];
            ct_vel = b.vel_target[e * nq + c.l];
            ct_acc = b.acc_target[e * nq + c.l];
            ct_tau = b.pid_state[e * 3 * nq + 3 * c.l + 2];  // the torque held since the controller last fired
        }
        if (pid_mode) {
            ref = md == B2_MODE_POSITION ? b.pos_target[e * nq + c.l] : b.vel_target[e * nq + c.l];
#pragma unroll
            for (int k = 0; k < 3; ++k) st[k] = b.pid_state[e * 3 * nq + 3 * c.l + k];
        }
        if (md == B2_MODE_VELOCITY_FOLLOWER_DART) vel_t = b.vel_target[e * nq + c.l];
    }
    // JointController::PreUpdate of the first iteration sees the last readback: the state before the pending resets
    if (control && c.body) {
        fc = st[2];
        if (cfg.compute_new_bits & 1u) fc = pid_update(cfg.pid[jl], st, (md == B2_MODE_POSITION ? q : dq) - ref, cfg.dt);
    }
    // the controller of the first iteration sees the readback too (ControllerRunner::PreUpdate runs before Physics::Update)
    if (CT && ct && (cfg.ct_compute_bits & 1u))
        ct_tau = lanes_inverse_dynamics(c, m, warp_strips, live_envs, q, dq,
                                        ct_acc - cfg.ct_kp[jl] * (q - ct_pos) - cfg.ct_kd[jl] * (dq - ct_vel), cfg.ct_gravity);
    // Physics::UpdatePhysics: velocity reset, then position reset (Physics.cpp:1330-1375)
    if (mask && c.body) {
        if (mask & (1u << (16 + c.l))) dq = b.reset_state[e * 2 * nq + nq + c.l];
        if (mask & (1u << c.l)) q = b.reset_state[e * 2 * nq + c.l];
    }
    __syncwarp();  // every lane of the env holds the mask before it is cleared
    if (!COUPLED && mask && c.live && c.l == 0) b.reset_mask[e] = 0u;
    bool stepped = false;
    T acc = T(0), tau_read = T(0);
    for (int it = 0; it < cfg.iterations; ++it) {
        if (it > 0 && control && c.body) {
            fc = st[2];
            if ((cfg.compute_new_bits >> it) & 1u) fc = pid_update(cfg.pid[jl], st, (md == B2_MODE_POSITION ? q : dq) - ref, cfg.dt);
        }
        if (CT && ct) {
            if (it > 0 && ((cfg.ct_compute_bits >> it) & 1u))
                ct_tau = lanes_inverse_dynamics(c, m, warp_strips, live_envs, q, dq,
                                                ct_acc - cfg.ct_kp[jl] * (q - ct_pos) - cfg.ct_kd[jl] * (dq - ct_vel), cfg.ct_gravity);
            fc = ct_tau;  // ControllerRunner re-applies the last torque every iteration (ControllerRunner.cpp:276-281)
        }
        T tau = T(0);
        bool servo = false;
        if (c.body) {
            if (has_fc || (CT && ct) || (pid_joint && !cfg.paused)) tau = fc;
            else if (md == B2_MODE_VELOCITY_FOLLOWER_DART && !cfg.paused && !(mask & (1u << (16 + c.l)))) servo = true;
        }
        // UpdateSim: one-shot commands are zeroed after every iteration (Physics.cpp:2250-2267)
        tau_read = cfg.paused ? tau : T(0);
        fc = T(0);
        if (!cfg.paused) {
            lanes_joint_placement(c, q);
            lanes_forward_kinematics(c, m, warp_strips, live_envs);
            for (int k = 0; k < cfg.nwrench; ++k) {  // Link::applyWorldWrench as J^T F (Physics.cpp:1483-1532)
                const int link = cfg.wrench_link[k], wb = m.link_body[link];
                if (wb < 0 || it >= cfg.wrench_iters[k]) continue;  // uniform
                const unsigned chain = tb.anc[wb];
                V3<T> aw = v3(T(0), T(0), T(0)), po = aw, pl = aw;
                if (c.body) {
                    T R[9];
                    lanes_load_placement(c, R, po);
                    aw = lanes_joint_axis(c, R);
                    if (c.l == wb) pl = place_point(R, po, m.link_p[link]);
                }
                const int src = c.slot * G + wb;
                pl.x = __shfl_sync(0xffffffffu, pl.x, src);
                pl.y = __shfl_sync(0xffffffffu, pl.y, src);
                pl.z = __shfl_sync(0xffffffffu, pl.z, src);
                if (c.body && ((chain >> c.l) & 1u) && (cfg.wrench_env[k] < 0 || cfg.wrench_env[k] == e)) {
                    const V3<T> f = v3(cfg.wrench[k][0], cfg.wrench[k][1], cfg.wrench[k][2]);
                    const V3<T> tq = v3(cfg.wrench[k][3], cfg.wrench[k][4], cfg.wrench[k][5]);
                    tau += ((tb.rev_mask >> c.l) & 1u) ? dot(cross(aw, pl - po), f) + dot(aw, tq) : dot(aw, f);
                }
            }
            T inv_d;
            T ddq = lanes_forward_dynamics<T, G, ENV>(c, m, cfg.dt, q, dq, tau, &inv_d, env);
            dq += ddq * cfg.dt;
            if (COUPLED) {  // the solver owns the constraint stage and k_world_finish the integration
                acc = ddq;
                stepped = true;
                continue;
            }
            // rows of joint_constraints: a servoed joint has its servo row only
            T env_friction = T(0), env_damping = T(0);  // ENV: the joint's row (read once, used below)
            if (ENV && c.body) { env_damping = env.joint[0]; env_friction = env.joint[1]; }
            const bool f0 = c.body && (servo || (ENV ? env_friction : c.tab[LT_FRICTION]) != T(0));
            const bool f1 = c.body && !servo && q <= c.tab[LT_LOWER], f2 = c.body && !servo && q >= c.tab[LT_UPPER];
            const unsigned rows = __ballot_sync(0xffffffffu, f0 || f1 || f2);
            if (rows) {
                T dq_io = dq, ddq_io = ddq;
                const bool dk = c.body && ((ENV ? env_damping : c.tab[LT_DAMPING]) != T(0) || c.tab[LT_STIFFNESS] != T(0));
                if (!lanes_constraints_fast<T, G>(c.sm + L::oP1 + L::oLT, inv_d, c.slot, c.l, nq, c.body, cfg.dt, f0, f1, f2, servo, vel_t,
                                                  servo ? c.tab[LT_EFFORT] : (ENV ? env_friction : c.tab[LT_FRICTION]), dk, &dq_io,
                                                  &ddq_io)) {
                    const unsigned env_bits = (1u << G) - 1u;
                    const unsigned servos = __ballot_sync(0xffffffffu, servo);
                    // ENV: lane 0 solves its env with the env's own inertias and friction (the pack holds its EnvParams)
                    const auto dense = [&](auto... prm) {
                        lanes_joint_constraints<T, G>(c.sm + L::oV, c.l, nq, c.body, c.l == 0 && ((rows >> (c.slot * G)) & env_bits) != 0u,
                                                      tables, cfg.dt, q, &dq_io, &ddq_io, (servos >> (c.slot * G)) & env_bits, vel_t,
                                                      prm...);
                    };
                    if constexpr (ENV) dense(env_rows.env(e, nq));
                    else dense();
                }
                dq = dq_io;
                ddq = ddq_io;
            }
            q += dq * cfg.dt;
            acc = ddq;
            stepped = true;
        }
    }
    if (c.body) {
        b.state[e * 2 * nq + c.l] = q;
        b.state[e * 2 * nq + nq + c.l] = dq;
        if (stepped) b.accel[e * nq + c.l] = acc;
        b.force_read[e * nq + c.l] = tau_read;
        b.force_cmd[e * nq + c.l] = T(0);
        if (control) {
#pragma unroll
            for (int k = 0; k < 3; ++k) b.pid_state[e * 3 * nq + 3 * c.l + k] = st[k];
        }
        if (CT && ct) b.pid_state[e * 3 * nq + 3 * c.l + 2] = ct_tau;
        if (COUPLED && stepped) v0[e * nvp + c.l] = dq;  // joint part of the solver's initial velocity
    }
}

}  // namespace b2
