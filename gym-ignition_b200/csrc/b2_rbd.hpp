// Rigid-body dynamics for fixed-base trees of 1-DoF joints, templated on the scalar type and
// callable from host and device. Body coordinates, spatial vectors ordered [angular; linear].
//
// What it replaces: the arithmetic the reference reaches through
//   cpp/scenario/plugins/Physics/Physics.cpp:1824-1835  (dartsim World::step -> ABA),
//   python/gym_ignition/rbd/idyntree/kindyncomputations.py:169-196,270-303,367-377 (FK, M, h, J).
// The articulated-body pass uses DART's implicit joint damping/spring:
//   psi = (S'AS + dt D + dt^2 K)^-1,   u = tau - D dq - K (q - q0 + dt dq) - S'(A eta + B).
#pragma once

#include <math.h>

#if defined(__CUDACC__)
#define B2_HD __host__ __device__ __forceinline__
#else
#define B2_HD inline
#endif

namespace b2 {

constexpr int kMaxDofs = 16;
constexpr int kMaxLinks = 32;
constexpr int kRevolute = 2;   // B2_JOINT_REVOLUTE
constexpr int kPrismatic = 3;  // B2_JOINT_PRISMATIC

template <typename T>
struct V3 {
    T x, y, z;
};
template <typename T> B2_HD V3<T> v3(T x, T y, T z) { return V3<T>{x, y, z}; }
template <typename T> B2_HD V3<T> operator+(V3<T> a, V3<T> b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
template <typename T> B2_HD V3<T> operator-(V3<T> a, V3<T> b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
template <typename T> B2_HD V3<T> operator*(T s, V3<T> a) { return {s * a.x, s * a.y, s * a.z}; }
template <typename T> B2_HD T dot(V3<T> a, V3<T> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <typename T> B2_HD V3<T> cross(V3<T> a, V3<T> b)
{
    return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}

// Row-major 3x3.
template <typename T>
struct M3 {
    T m[9];
};
template <typename T> B2_HD V3<T> mul(const M3<T>& A, V3<T> v)
{
    return {A.m[0] * v.x + A.m[1] * v.y + A.m[2] * v.z, A.m[3] * v.x + A.m[4] * v.y + A.m[5] * v.z,
            A.m[6] * v.x + A.m[7] * v.y + A.m[8] * v.z};
}
template <typename T> B2_HD V3<T> mulT(const M3<T>& A, V3<T> v)
{
    return {A.m[0] * v.x + A.m[3] * v.y + A.m[6] * v.z, A.m[1] * v.x + A.m[4] * v.y + A.m[7] * v.z,
            A.m[2] * v.x + A.m[5] * v.y + A.m[8] * v.z};
}
template <typename T> B2_HD M3<T> mul(const M3<T>& A, const M3<T>& B)
{
    M3<T> C;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            C.m[3 * i + j] = A.m[3 * i] * B.m[j] + A.m[3 * i + 1] * B.m[3 + j] + A.m[3 * i + 2] * B.m[6 + j];
    return C;
}
// A * B^T
template <typename T> B2_HD M3<T> mulBt(const M3<T>& A, const M3<T>& B)
{
    M3<T> C;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            C.m[3 * i + j] =
                A.m[3 * i] * B.m[3 * j] + A.m[3 * i + 1] * B.m[3 * j + 1] + A.m[3 * i + 2] * B.m[3 * j + 2];
    return C;
}
template <typename T> B2_HD M3<T> transpose(const M3<T>& A)
{
    return M3<T>{{A.m[0], A.m[3], A.m[6], A.m[1], A.m[4], A.m[7], A.m[2], A.m[5], A.m[8]}};
}
template <typename T> B2_HD M3<T> skew(V3<T> p)
{
    return M3<T>{{T(0), -p.z, p.y, p.z, T(0), -p.x, -p.y, p.x, T(0)}};
}
template <typename T> B2_HD M3<T> operator+(const M3<T>& A, const M3<T>& B)
{
    M3<T> C;
    for (int i = 0; i < 9; ++i) C.m[i] = A.m[i] + B.m[i];
    return C;
}
template <typename T> B2_HD M3<T> operator-(const M3<T>& A, const M3<T>& B)
{
    M3<T> C;
    for (int i = 0; i < 9; ++i) C.m[i] = A.m[i] - B.m[i];
    return C;
}
template <typename T> B2_HD M3<T> outer(V3<T> a, V3<T> b)
{
    return M3<T>{{a.x * b.x, a.x * b.y, a.x * b.z, a.y * b.x, a.y * b.y, a.y * b.z, a.z * b.x, a.z * b.y,
                  a.z * b.z}};
}

#if defined(__CUDA_ARCH__)
// sin / cos on the device: two-constant Cody-Waite reduction by pi/2 with FMAs (x - n HI is formed exactly inside the
// FMA, HI + LO carries pi/2 to 1e-33), then the fdlibm kernels on [-pi/4, pi/4]; about 1 ulp, a third of the library
// routine's instructions. Beyond 1e4 rad the library routine (Payne-Hanek reduction) takes over.
__device__ __forceinline__ void sincos_reduced(double x, double* s, double* c)
{
    if (!(fabs(x) < 1.0e4)) { sincos(x, s, c); return; }
    // round-to-nearest of x 2/pi by adding 1.5 * 2^52: the integer lands in the low mantissa bits (no conversion instructions)
    const double big = fma(x, 0.63661977236758134308, 6755399441055744.0);
    const int quad = __double2loint(big);
    const double n = big - 6755399441055744.0;
    double r = fma(-n, 1.57079632679489655800e+00, x);
    r = fma(-n, 6.12323399573676603587e-17, r);
    const double z = r * r;
    double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
    ps = fma(z, ps, 2.75573137070700676789e-06);
    ps = fma(z, ps, -1.98412698298579493134e-04);
    ps = fma(z, ps, 8.33333333332248946124e-03);
    ps = fma(z, ps, -1.66666666666666324348e-01);
    const double sn = fma(r * z, ps, r);
    double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
    pc = fma(z, pc, -2.75573143513906633035e-07);
    pc = fma(z, pc, 2.48015872894767294178e-05);
    pc = fma(z, pc, -1.38888888888741095749e-03);
    pc = fma(z, pc, 4.16666666666666019037e-02);
    const double cs = fma(z * z, pc, fma(z, -0.5, 1.0));
    const double a = (quad & 1) ? cs : sn, b = (quad & 1) ? sn : cs;
    *s = (quad & 2) ? -a : a;
    *c = ((quad + 1) & 2) ? -b : b;
}
#endif

B2_HD void sincos_t(double x, double* s, double* c)
{
#if defined(__CUDA_ARCH__)
    sincos(x, s, c);
#else
    *s = sin(x);
    *c = cos(x);
#endif
}
// Throughput variant for the HBM-bound cart-pole step kernel (k_task_chain): sincos_reduced has fewer instructions than
// the library routine (77 us against 78.4 us per launch at 4,194,304 envs) but a longer dependent chain, which costs the
// latency-bound kernels (pendulum trajectory 1.30 us against 1.09 us per step at 65,536 envs; the tree kernels do not
// move), so only that kernel uses it.
B2_HD void sincos_tp(double x, double* s, double* c)
{
#if defined(__CUDA_ARCH__)
    sincos_reduced(x, s, c);
#else
    sincos_t(x, s, c);
#endif
}
B2_HD void sincos_t(float x, float* s, float* c)
{
#if defined(__CUDA_ARCH__)
    sincosf(x, s, c);
#else
    *s = sinf(x);
    *c = cosf(x);
#endif
}

B2_HD double cos_t(double x)
{
#if defined(__CUDA_ARCH__)
    double s, c;
    sincos_reduced(x, &s, &c);  // the sine polynomial is dead code here
    return c;
#else
    return cos(x);
#endif
}
B2_HD float cos_t(float x) { return cosf(x); }
B2_HD void sincos_tp(float x, float* s, float* c) { sincos_t(x, s, c); }

// Rotation about the unit axis a by angle q (Rodrigues).
template <typename T> B2_HD M3<T> axis_angle(V3<T> a, T q)
{
    T s, c;
    sincos_t(q, &s, &c);
    const T t = T(1) - c;
    return M3<T>{{c + t * a.x * a.x, t * a.x * a.y - s * a.z, t * a.x * a.z + s * a.y,
                  t * a.x * a.y + s * a.z, c + t * a.y * a.y, t * a.y * a.z - s * a.x,
                  t * a.x * a.z - s * a.y, t * a.y * a.z + s * a.x, c + t * a.z * a.z}};
}

// Spatial motion / force vectors.
template <typename T>
struct Sv {
    V3<T> a;  // angular (motion) or moment (force)
    V3<T> l;  // linear (motion) or force (force)
};
template <typename T> B2_HD Sv<T> operator+(Sv<T> x, Sv<T> y) { return {x.a + y.a, x.l + y.l}; }
template <typename T> B2_HD Sv<T> operator-(Sv<T> x, Sv<T> y) { return {x.a - y.a, x.l - y.l}; }
template <typename T> B2_HD Sv<T> sv_zero() { return {{T(0), T(0), T(0)}, {T(0), T(0), T(0)}}; }

// Articulated inertia  [[A, B], [B^T, C]]  (A, C symmetric; stored full for simplicity).
template <typename T>
struct Ai {
    M3<T> A, B, C;
};
template <typename T> B2_HD Sv<T> mul(const Ai<T>& I, Sv<T> v)
{
    return {mul(I.A, v.a) + mul(I.B, v.l), mulT(I.B, v.a) + mul(I.C, v.l)};
}

// Flattened model tables in the scalar type of the kernels.
template <typename T>
struct alignas(16) ModelDev {
    int nq;
    int nlinks;
    int parent[kMaxDofs];
    int jtype[kMaxDofs];
    T axis[kMaxDofs][3];
    T R[kMaxDofs][9];
    T p[kMaxDofs][3];
    T mass[kMaxDofs];
    T mc[kMaxDofs][3];  // mass * com
    T Io[kMaxDofs][9];  // rotational inertia about the body origin
    T damping[kMaxDofs], friction[kMaxDofs], stiffness[kMaxDofs], rest[kMaxDofs];
    T lower[kMaxDofs], upper[kMaxDofs], effort[kMaxDofs];
    T g[3];             // gravity, world frame
    T baseR[9];         // world_H_base
    T basep[3];
    int link_body[kMaxLinks];
    T link_R[kMaxLinks][9];
    T link_p[kMaxLinks][3];
    T base_mass;        // links welded to the base: mass and first moment in the base frame
    T base_mc[3];
    T Icom[kMaxDofs][6]; // rotational inertia about the centre of mass, body frame (xx, xy, xz, yy, yz, zz)
    T com[kMaxDofs][3];  // centre of mass, body frame (b2_lanes.cuh builds world-frame inertias from these)
    T base_Io[6];        // links welded to the base: rotational inertia about the base origin, base frame (xx, xy, xz, yy, yz, zz)
};

// Per-body constants of a model packed for the lane-parallel kernels (b2_lanes.cuh): one 32-scalar, 16-byte aligned
// record per body that the lane owning the body reads with vector loads.
enum {
    LT_R = 0, LT_P = 9, LT_AXIS = 12, LT_MASS = 15, LT_ICOM = 16, LT_COM = 22, LT_DAMPING = 25, LT_STIFFNESS = 26,
    LT_REST = 27, LT_LOWER = 28, LT_UPPER = 29, LT_FRICTION = 30, LT_EFFORT = 31, LT_SIZE = 32
};
template <typename T>
struct alignas(16) LaneTable {
    T body[kMaxDofs][LT_SIZE];
};
template <typename T> inline void fill_lane_table(const ModelDev<T>& m, LaneTable<T>& o)
{
    for (int b = 0; b < kMaxDofs; ++b) {
        T* r = o.body[b];
        for (int k = 0; k < 9; ++k) r[LT_R + k] = m.R[b][k];
        for (int k = 0; k < 3; ++k) { r[LT_P + k] = m.p[b][k]; r[LT_AXIS + k] = m.axis[b][k]; r[LT_COM + k] = m.com[b][k]; }
        for (int k = 0; k < 6; ++k) r[LT_ICOM + k] = m.Icom[b][k];
        r[LT_MASS] = m.mass[b]; r[LT_DAMPING] = m.damping[b]; r[LT_STIFFNESS] = m.stiffness[b]; r[LT_REST] = m.rest[b];
        r[LT_LOWER] = m.lower[b]; r[LT_UPPER] = m.upper[b]; r[LT_FRICTION] = m.friction[b]; r[LT_EFFORT] = m.effort[b];
    }
}

template <typename T> B2_HD V3<T> ld3(const T* p) { return {p[0], p[1], p[2]}; }
template <typename T> B2_HD M3<T> ld9(const T* p)
{
    M3<T> A;
    for (int i = 0; i < 9; ++i) A.m[i] = p[i];
    return A;
}

// Where the run path reads a body's inertia, a joint's viscous damping and Coulomb friction, and the gravity.
// NominalParams: the model's shared tables. EnvParams: one env's rows of B2_BUF_BODY_INERTIA / B2_BUF_JOINT_DYNAMICS /
// B2_BUF_GRAVITY (b2sim_enable_env_params); the first moment and the inertia about the body origin are derived from the
// row where they are used, so no per-env copy of the model exists.
template <typename T>
struct NominalParams {
    static constexpr bool nominal = true;
    B2_HD T mass(const ModelDev<T>& m, int i) const { return m.mass[i]; }
    B2_HD V3<T> mc(const ModelDev<T>& m, int i) const { return ld3(m.mc[i]); }
    B2_HD M3<T> Io(const ModelDev<T>& m, int i) const { return ld9(m.Io[i]); }
    B2_HD T damping(const ModelDev<T>& m, int i) const { return m.damping[i]; }
    B2_HD T friction(const ModelDev<T>& m, int i) const { return m.friction[i]; }
    B2_HD V3<T> g(const ModelDev<T>& m) const { return ld3(m.g); }
    B2_HD bool undamped(const ModelDev<T>&) const { return true; }  // the host folded the tables' damping into the topology
};

// Row layouts: inertia [nq][10] = mass, centre of mass (x, y, z), rotational inertia about it (xx, xy, xz, yy, yz, zz),
// body frame; dynamics [nq][2] = viscous damping, Coulomb friction; gravity [3], world frame.
constexpr int kEnvInertiaCols = 10;
constexpr int kEnvJointCols = 2;

template <typename T>
struct EnvParams {
    static constexpr bool nominal = false;
    const T* inertia;
    const T* dyn;
    const T* grav;
    B2_HD T mass(const ModelDev<T>&, int i) const { return inertia[kEnvInertiaCols * i]; }
    B2_HD V3<T> com(int i) const { return ld3(inertia + kEnvInertiaCols * i + 1); }
    B2_HD V3<T> mc(const ModelDev<T>& m, int i) const { return mass(m, i) * com(i); }
    // Ic + m (c.c 1 - c c^T), as the loader forms the shared tables (b2_model.cpp to_device_tables)
    B2_HD M3<T> Io(const ModelDev<T>& m, int i) const
    {
        const T* r = inertia + kEnvInertiaCols * i;
        const T mi = r[0], cx = r[1], cy = r[2], cz = r[3];
        const T cc = cx * cx + cy * cy + cz * cz;
        const T xy = r[5] - mi * (cx * cy), xz = r[6] - mi * (cx * cz), yz = r[8] - mi * (cy * cz);
        return M3<T>{{r[4] + mi * (cc - cx * cx), xy, xz, xy, r[7] + mi * (cc - cy * cy), yz, xz, yz,
                      r[9] + mi * (cc - cz * cz)}};
    }
    B2_HD T damping(const ModelDev<T>&, int i) const { return dyn[kEnvJointCols * i]; }
    B2_HD T friction(const ModelDev<T>&, int i) const { return dyn[kEnvJointCols * i + 1]; }
    B2_HD V3<T> g(const ModelDev<T>&) const { return ld3(grav); }
    B2_HD bool undamped(const ModelDev<T>& m) const
    {
        bool z = true;
        for (int i = 0; i < m.nq; ++i) z = z && dyn[kEnvJointCols * i] == T(0);
        return z;
    }
};

// Pose of the child frame of joint i in its parent body frame at position q.
template <typename T> B2_HD void joint_pose(const ModelDev<T>& m, int i, T q, M3<T>& R, V3<T>& p)
{
    const V3<T> a = ld3(m.axis[i]);
    const M3<T> R0 = ld9(m.R[i]);
    const V3<T> p0 = ld3(m.p[i]);
    if (m.jtype[i] == kRevolute) {
        if (a.z == T(1)) {
            // rotation about the joint z axis (URDF convention of most arms, every Panda joint): the first two columns
            // of R0 mix, no Rodrigues matrix and no 3x3 product
            T s, c;
            sincos_t(q, &s, &c);
            R = M3<T>{{c * R0.m[0] + s * R0.m[1], c * R0.m[1] - s * R0.m[0], R0.m[2],
                       c * R0.m[3] + s * R0.m[4], c * R0.m[4] - s * R0.m[3], R0.m[5],
                       c * R0.m[6] + s * R0.m[7], c * R0.m[7] - s * R0.m[6], R0.m[8]}};
        } else {
            R = mul(R0, axis_angle(a, q));
        }
        p = p0;
    } else {
        R = R0;
        p = p0 + mul(R0, q * a);
    }
}

// Per-body scratch of the articulated-body algorithm.
template <typename T>
struct AbaBody {
    M3<T> R;      // child frame orientation in the parent frame
    V3<T> p;      // child origin in the parent frame
    Sv<T> V;      // spatial velocity
    Sv<T> eta;    // velocity-product acceleration
    Sv<T> B;      // bias force
    Ai<T> IA;     // articulated inertia (implicit)
    Sv<T> U;      // IA * S
    T psi, u;
    Sv<T> acc;
};

// Forward dynamics with implicit damping/spring. ddq = FD(q, dq, tau).
template <typename T, int NB>
B2_HD void forward_dynamics(const ModelDev<T>& m, T dt, const T* q, const T* dq, const T* tau, T* ddq)
{
    AbaBody<T> b[NB];
    V3<T> gb[NB];  // gravity expressed in each body frame
    const int nq = m.nq;
    const V3<T> g_base = mulT(ld9(m.baseR), ld3(m.g));

    for (int i = 0; i < nq; ++i) {
        const int par = m.parent[i];
        const V3<T> a = ld3(m.axis[i]);
        const bool rev = m.jtype[i] == kRevolute;
        joint_pose(m, i, q[i], b[i].R, b[i].p);
        Sv<T> Vp = par >= 0 ? b[par].V : sv_zero<T>();
        const V3<T> sd = dq[i] * a;
        Sv<T> V;
        V.a = mulT(b[i].R, Vp.a);
        V.l = mulT(b[i].R, Vp.l + cross(Vp.a, b[i].p));
        if (rev) {
            b[i].eta = {cross(V.a, sd), cross(V.l, sd)};  // uses the parent part only: sd x sd = 0
            V.a = V.a + sd;
        } else {
            b[i].eta = {v3(T(0), T(0), T(0)), cross(V.a, sd)};
            V.l = V.l + sd;
        }
        b[i].V = V;
        gb[i] = mulT(b[i].R, par >= 0 ? gb[par] : g_base);
        // rigid-body inertia and bias force
        const T mass = m.mass[i];
        const V3<T> mc = ld3(m.mc[i]);
        const M3<T> Io = ld9(m.Io[i]);
        const V3<T> n = mul(Io, V.a) + cross(mc, V.l);
        const V3<T> f = mass * V.l - cross(mc, V.a);
        b[i].B.a = cross(V.a, n) + cross(V.l, f) - cross(mc, gb[i]);
        b[i].B.l = cross(V.a, f) - mass * gb[i];
        b[i].IA.A = Io;
        b[i].IA.B = skew(mc);
        b[i].IA.C = M3<T>{{mass, T(0), T(0), T(0), mass, T(0), T(0), T(0), mass}};
    }
    for (int i = nq - 1; i >= 0; --i) {
        const int par = m.parent[i];
        const V3<T> a = ld3(m.axis[i]);
        const bool rev = m.jtype[i] == kRevolute;
        AbaBody<T>& bi = b[i];
        T d;
        if (rev) {
            bi.U = {mul(bi.IA.A, a), mulT(bi.IA.B, a)};
            d = dot(a, bi.U.a);
        } else {
            bi.U = {mul(bi.IA.B, a), mul(bi.IA.C, a)};
            d = dot(a, bi.U.l);
        }
        d += dt * m.damping[i] + dt * dt * m.stiffness[i];
        bi.psi = T(1) / d;
        const Sv<T> pa = mul(bi.IA, bi.eta) + bi.B;
        bi.u = tau[i] - m.damping[i] * dq[i] - m.stiffness[i] * (q[i] - m.rest[i] + dt * dq[i]) -
               (rev ? dot(a, pa.a) : dot(a, pa.l));
        if (par >= 0) {
            // Pi = IA - U psi U^T ; beta = B + IA eta + U psi u
            Ai<T> Pi;
            const V3<T> Ua = bi.psi * bi.U.a, Ul = bi.psi * bi.U.l;
            Pi.A = bi.IA.A - outer(Ua, bi.U.a);
            Pi.B = bi.IA.B - outer(Ua, bi.U.l);
            Pi.C = bi.IA.C - outer(Ul, bi.U.l);
            const T s = bi.psi * bi.u;
            Sv<T> beta = {pa.a + s * bi.U.a, pa.l + s * bi.U.l};
            // rotate into the parent orientation, then shift the reference point by p
            const M3<T>& R = bi.R;
            const M3<T> A1 = mulBt(mul(R, Pi.A), R), B1 = mulBt(mul(R, Pi.B), R), C1 = mulBt(mul(R, Pi.C), R);
            const M3<T> P = skew(bi.p);
            const M3<T> PC = mul(P, C1);
            const M3<T> TR = B1 + PC;                      // B' + P C'
            const M3<T> PBt = mulBt(P, B1);                // P B'^T
            const M3<T> TL = A1 + PBt - mul(TR, P);        // A' + P B'^T - (B' + P C') P
            AbaBody<T>& bp = b[par];
            bp.IA.A = bp.IA.A + TL;
            bp.IA.B = bp.IA.B + TR;
            bp.IA.C = bp.IA.C + C1;
            const V3<T> fl = mul(R, beta.l);
            bp.B.a = bp.B.a + mul(R, beta.a) + cross(bi.p, fl);
            bp.B.l = bp.B.l + fl;
        }
    }
    for (int i = 0; i < nq; ++i) {
        const int par = m.parent[i];
        const V3<T> a = ld3(m.axis[i]);
        const bool rev = m.jtype[i] == kRevolute;
        AbaBody<T>& bi = b[i];
        Sv<T> ap = sv_zero<T>();
        if (par >= 0) {
            const Sv<T>& A = b[par].acc;
            ap.a = mulT(bi.R, A.a);
            ap.l = mulT(bi.R, A.l + cross(A.a, bi.p));
        }
        const T acc = bi.psi * (bi.u - dot(bi.U.a, ap.a) - dot(bi.U.l, ap.l));
        ddq[i] = acc;
        bi.acc = ap + bi.eta;
        if (rev) bi.acc.a = bi.acc.a + acc * a;
        else bi.acc.l = bi.acc.l + acc * a;
    }
}

// Recursive Newton-Euler: tau = M ddq + C dq + g (gravity optional). No damping / spring terms.
template <typename T, int NB>
B2_HD void inverse_dynamics(const ModelDev<T>& m, const T* q, const T* dq, const T* ddq, bool gravity, T* tau,
                            const T* gravity_override = nullptr)
{
    M3<T> R[NB];
    V3<T> p[NB];
    Sv<T> V[NB], A[NB], F[NB];
    const int nq = m.nq;
    const V3<T> g_base = mulT(ld9(m.baseR), gravity_override ? ld3(gravity_override) : ld3(m.g));
    for (int i = 0; i < nq; ++i) {
        const int par = m.parent[i];
        const V3<T> a = ld3(m.axis[i]);
        const bool rev = m.jtype[i] == kRevolute;
        joint_pose(m, i, q[i], R[i], p[i]);
        Sv<T> Vp = sv_zero<T>(), Ap = sv_zero<T>();
        if (par >= 0) {
            Vp = V[par];
            Ap = A[par];
        } else if (gravity) {
            Ap.l = T(-1) * g_base;  // fictitious base acceleration
        }
        Sv<T> Vi, Ai_;
        Vi.a = mulT(R[i], Vp.a);
        Vi.l = mulT(R[i], Vp.l + cross(Vp.a, p[i]));
        Ai_.a = mulT(R[i], Ap.a);
        Ai_.l = mulT(R[i], Ap.l + cross(Ap.a, p[i]));
        const V3<T> sd = dq[i] * a, sdd = ddq[i] * a;
        if (rev) {
            Ai_.a = Ai_.a + cross(Vi.a, sd) + sdd;
            Ai_.l = Ai_.l + cross(Vi.l, sd);
            Vi.a = Vi.a + sd;
        } else {
            Ai_.l = Ai_.l + cross(Vi.a, sd) + sdd;
            Vi.l = Vi.l + sd;
        }
        V[i] = Vi;
        A[i] = Ai_;
        const T mass = m.mass[i];
        const V3<T> mc = ld3(m.mc[i]);
        const M3<T> Io = ld9(m.Io[i]);
        const V3<T> n = mul(Io, Vi.a) + cross(mc, Vi.l);
        const V3<T> f = mass * Vi.l - cross(mc, Vi.a);
        F[i].a = mul(Io, Ai_.a) + cross(mc, Ai_.l) + cross(Vi.a, n) + cross(Vi.l, f);
        F[i].l = mass * Ai_.l - cross(mc, Ai_.a) + cross(Vi.a, f);
    }
    for (int i = nq - 1; i >= 0; --i) {
        const V3<T> a = ld3(m.axis[i]);
        tau[i] = m.jtype[i] == kRevolute ? dot(a, F[i].a) : dot(a, F[i].l);
        const int par = m.parent[i];
        if (par >= 0) {
            const V3<T> fl = mul(R[i], F[i].l);
            F[par].a = F[par].a + mul(R[i], F[i].a) + cross(p[i], fl);
            F[par].l = F[par].l + fl;
        }
    }
}

// Composite-rigid-body algorithm: joint-space mass matrix, row-major nq x nq (full, symmetric).
// P: where the inertias come from (NominalParams / EnvParams); the controllers and KinDyn queries use the nominal model.
template <typename T, int NB, typename Prm = NominalParams<T>>
B2_HD void mass_matrix(const ModelDev<T>& m, const T* q, T* M, const Prm& prm = Prm())
{
    M3<T> R[NB];
    V3<T> p[NB];
    Ai<T> IC[NB];
    const int nq = m.nq;
    for (int k = 0; k < nq * nq; ++k) M[k] = T(0);  // entries between different branches stay zero
    for (int i = 0; i < nq; ++i) {
        joint_pose(m, i, q[i], R[i], p[i]);
        const T mass = prm.mass(m, i);
        IC[i].A = prm.Io(m, i);
        IC[i].B = skew(prm.mc(m, i));
        IC[i].C = M3<T>{{mass, T(0), T(0), T(0), mass, T(0), T(0), T(0), mass}};
    }
    for (int i = nq - 1; i >= 0; --i) {
        const int par = m.parent[i];
        if (par >= 0) {
            const M3<T> A1 = mulBt(mul(R[i], IC[i].A), R[i]), B1 = mulBt(mul(R[i], IC[i].B), R[i]),
                        C1 = mulBt(mul(R[i], IC[i].C), R[i]);
            const M3<T> P = skew(p[i]);
            const M3<T> TR = B1 + mul(P, C1);
            const M3<T> TL = A1 + mulBt(P, B1) - mul(TR, P);
            IC[par].A = IC[par].A + TL;
            IC[par].B = IC[par].B + TR;
            IC[par].C = IC[par].C + C1;
        }
        const V3<T> a = ld3(m.axis[i]);
        Sv<T> F;
        if (m.jtype[i] == kRevolute) F = {mul(IC[i].A, a), mulT(IC[i].B, a)};
        else F = {mul(IC[i].B, a), mul(IC[i].C, a)};
        M[i * nq + i] = m.jtype[i] == kRevolute ? dot(a, F.a) : dot(a, F.l);
        int j = i;
        while (m.parent[j] >= 0) {
            const V3<T> fl = mul(R[j], F.l);
            F.a = mul(R[j], F.a) + cross(p[j], fl);
            F.l = fl;
            j = m.parent[j];
            const V3<T> aj = ld3(m.axis[j]);
            const T v = m.jtype[j] == kRevolute ? dot(aj, F.a) : dot(aj, F.l);
            M[i * nq + j] = v;
            M[j * nq + i] = v;
        }
    }
}

// World pose of every body frame.
template <typename T, int NB>
B2_HD void forward_kinematics(const ModelDev<T>& m, const T* q, M3<T>* Rw, V3<T>* pw)
{
    const M3<T> Rb = ld9(m.baseR);
    const V3<T> pb = ld3(m.basep);
    for (int i = 0; i < m.nq; ++i) {
        M3<T> R;
        V3<T> p;
        joint_pose(m, i, q[i], R, p);
        const int par = m.parent[i];
        const M3<T>& Rp = par >= 0 ? Rw[par] : Rb;
        const V3<T>& pp = par >= 0 ? pw[par] : pb;
        Rw[i] = mul(Rp, R);
        pw[i] = pp + mul(Rp, p);
    }
}

// KinDynComputations centre of mass / momentum (python/gym_ignition/rbd/idyntree/kindyncomputations.py:305-342):
// total centre of mass com[3], its velocity vel[3], mom[12] = linear / angular momentum about the world origin then
// about the centre of mass (world orientation), and the joint columns jac[3][nq] of the centre-of-mass Jacobian.
// Links welded to the base count with their (constant) mass. Any output may be null.
template <typename T, int NB>
B2_HD void centroidal(const ModelDev<T>& m, const T* q, const T* dq, T* com_out, T* vel_out, T* mom_out, T* jac_out)
{
    const int nq = m.nq;
    M3<T> Rw[NB];
    V3<T> pw[NB], sub_s[NB];
    Sv<T> V[NB];
    T sub_m[NB];
    const M3<T> Rb = ld9(m.baseR);
    const V3<T> pb = ld3(m.basep);
    T mass = m.base_mass;
    V3<T> first = mass * pb + mul(Rb, ld3(m.base_mc));
    V3<T> L = v3(T(0), T(0), T(0)), H = L;
    for (int i = 0; i < nq; ++i) {
        const int par = m.parent[i];
        M3<T> R;
        V3<T> p;
        joint_pose(m, i, q[i], R, p);
        const M3<T>& Rp = par >= 0 ? Rw[par] : Rb;
        Rw[i] = mul(Rp, R);
        pw[i] = (par >= 0 ? pw[par] : pb) + mul(Rp, p);
        const Sv<T> Vp = par >= 0 ? V[par] : sv_zero<T>();
        Sv<T> Vi = {mulT(R, Vp.a), mulT(R, Vp.l + cross(Vp.a, p))};
        const V3<T> sd = dq[i] * ld3(m.axis[i]);
        if (m.jtype[i] == kRevolute) Vi.a = Vi.a + sd;
        else Vi.l = Vi.l + sd;
        V[i] = Vi;
        const T mi = m.mass[i];
        const V3<T> mc = ld3(m.mc[i]);
        const V3<T> cb = mi > T(0) ? (T(1) / mi) * mc : v3(T(0), T(0), T(0));
        const V3<T> cw = pw[i] + mul(Rw[i], cb);
        sub_m[i] = mi;
        sub_s[i] = mi * cw;
        mass += mi;
        first = first + mi * cw;
        // momentum of the body: m v_c, and I_c w + c x m v_c about the world origin (I_c w = I_o w - m c x (w x c))
        const V3<T> vc = mul(Rw[i], Vi.l + cross(Vi.a, cb));
        const V3<T> Icw = mul(ld9(m.Io[i]), Vi.a) - mi * cross(cb, cross(Vi.a, cb));
        L = L + mi * vc;
        H = H + mul(Rw[i], Icw) + cross(cw, mi * vc);
    }
    const V3<T> com = (T(1) / mass) * first;
    if (com_out) { com_out[0] = com.x; com_out[1] = com.y; com_out[2] = com.z; }
    if (vel_out) {
        const V3<T> v = (T(1) / mass) * L;
        vel_out[0] = v.x; vel_out[1] = v.y; vel_out[2] = v.z;
    }
    if (mom_out) {
        const V3<T> Hg = H - cross(com, L);
        mom_out[0] = L.x; mom_out[1] = L.y; mom_out[2] = L.z; mom_out[3] = H.x; mom_out[4] = H.y; mom_out[5] = H.z;
        mom_out[6] = L.x; mom_out[7] = L.y; mom_out[8] = L.z; mom_out[9] = Hg.x; mom_out[10] = Hg.y; mom_out[11] = Hg.z;
    }
    if (jac_out) {
        for (int i = nq - 1; i >= 0; --i) {
            const int par = m.parent[i];
            if (par >= 0) { sub_m[par] += sub_m[i]; sub_s[par] = sub_s[par] + sub_s[i]; }
        }
        for (int i = 0; i < nq; ++i) {
            const V3<T> aw = mul(Rw[i], ld3(m.axis[i]));
            const V3<T> col = m.jtype[i] == kRevolute ? (T(1) / mass) * cross(aw, sub_s[i] - sub_m[i] * pw[i])
                                                      : (sub_m[i] / mass) * aw;
            jac_out[0 * nq + i] = col.x; jac_out[1 * nq + i] = col.y; jac_out[2 * nq + i] = col.z;
        }
    }
}

// Momentum matrices of KinDynComputations (python/gym_ignition/rbd/idyntree/kindyncomputations.py:379-427:
// getLinearAngularMomentumJacobian, getCentroidalTotalMomentumJacobian, get*AverageVelocityJacobian). Everything is
// expressed in the frame iDynTree's MIXED representation uses for the momentum, B[A]: world orientation, origin at the
// model's base. A rigid sub-tree's spatial inertia about that origin is additive (rotational inertia 6, first moment 3,
// mass 1), so the momentum a unit velocity of joint j produces is Ic_j S_j with Ic_j the composite inertia of the
// sub-tree j carries.
//   jmom_out[6][nq]  joint columns of the momentum Jacobian: rows 0-2 linear, rows 3-5 angular about the base origin
//   locked_out[10]   locked inertia of the whole model about the base origin (xx, xy, xz, yy, yz, zz, m c (3), m), links
//                    welded to the base included; the base block of the Jacobian and the average-velocity Jacobians
//                    follow from it on the host side (gym_ignition/rbd/kindyn.py)
template <typename T, int NB>
B2_HD void momentum_matrices(const ModelDev<T>& m, const T* q, T* jmom_out, T* locked_out)
{
    const int nq = m.nq;
    M3<T> Rw[NB];
    V3<T> pr[NB];  // body origins relative to the base origin, world orientation
    T Ic[NB][10];
    const M3<T> Rb = ld9(m.baseR);
    for (int i = 0; i < nq; ++i) {
        const int par = m.parent[i];
        M3<T> R;
        V3<T> p;
        joint_pose(m, i, q[i], R, p);
        const M3<T>& Rp = par >= 0 ? Rw[par] : Rb;
        Rw[i] = mul(Rp, R);
        pr[i] = mul(Rp, p);
        if (par >= 0) pr[i] = pr[i] + pr[par];
        const T mi = m.mass[i];
        const V3<T> cw = pr[i] + mul(Rw[i], ld3(m.com[i]));
        const T* ic = m.Icom[i];
        const M3<T> Ib = {{ic[0], ic[1], ic[2], ic[1], ic[3], ic[4], ic[2], ic[4], ic[5]}};
        const M3<T> Iw = mulBt(mul(Rw[i], Ib), Rw[i]);
        const T cc = dot(cw, cw);
        Ic[i][0] = Iw.m[0] + mi * (cc - cw.x * cw.x);
        Ic[i][1] = Iw.m[1] - mi * cw.x * cw.y;
        Ic[i][2] = Iw.m[2] - mi * cw.x * cw.z;
        Ic[i][3] = Iw.m[4] + mi * (cc - cw.y * cw.y);
        Ic[i][4] = Iw.m[5] - mi * cw.y * cw.z;
        Ic[i][5] = Iw.m[8] + mi * (cc - cw.z * cw.z);
        Ic[i][6] = mi * cw.x; Ic[i][7] = mi * cw.y; Ic[i][8] = mi * cw.z;
        Ic[i][9] = mi;
    }
    T tot[10];
    {   // links welded to the base
        const T* b = m.base_Io;
        const M3<T> Ib = {{b[0], b[1], b[2], b[1], b[3], b[4], b[2], b[4], b[5]}};
        const M3<T> Iw = mulBt(mul(Rb, Ib), Rb);
        const V3<T> mc = mul(Rb, ld3(m.base_mc));
        tot[0] = Iw.m[0]; tot[1] = Iw.m[1]; tot[2] = Iw.m[2]; tot[3] = Iw.m[4]; tot[4] = Iw.m[5]; tot[5] = Iw.m[8];
        tot[6] = mc.x; tot[7] = mc.y; tot[8] = mc.z; tot[9] = m.base_mass;
    }
    for (int i = nq - 1; i >= 0; --i) {
        const int par = m.parent[i];
        T* up = par >= 0 ? Ic[par] : tot;
        for (int k = 0; k < 10; ++k) up[k] += Ic[i][k];
    }
    if (locked_out)
        for (int k = 0; k < 10; ++k) locked_out[k] = tot[k];
    if (!jmom_out) return;
    for (int i = 0; i < nq; ++i) {
        const V3<T> aw = mul(Rw[i], ld3(m.axis[i]));
        V3<T> w = v3(T(0), T(0), T(0)), v = aw;
        if (m.jtype[i] == kRevolute) { w = aw; v = cross(pr[i], aw); }
        const T* I = Ic[i];
        const V3<T> mc = v3(I[6], I[7], I[8]);
        const V3<T> n = v3(I[0] * w.x + I[1] * w.y + I[2] * w.z, I[1] * w.x + I[3] * w.y + I[4] * w.z,
                           I[2] * w.x + I[4] * w.y + I[5] * w.z) + cross(mc, v);
        const V3<T> f = I[9] * v - cross(mc, w);
        jmom_out[0 * nq + i] = f.x; jmom_out[1 * nq + i] = f.y; jmom_out[2 * nq + i] = f.z;
        jmom_out[3 * nq + i] = n.x; jmom_out[4 * nq + i] = n.y; jmom_out[5 * nq + i] = n.z;
    }
}

// Rotation matrix -> unit quaternion (w, x, y, z), w >= 0 branch selection as in Eigen.
template <typename T> B2_HD void rot_to_quat(const M3<T>& R, T* qw)
{
    const T tr = R.m[0] + R.m[4] + R.m[8];
    T w, x, y, z;
    if (tr > T(0)) {
        T s = sqrt(tr + T(1)) * T(2);
        w = T(0.25) * s;
        x = (R.m[7] - R.m[5]) / s;
        y = (R.m[2] - R.m[6]) / s;
        z = (R.m[3] - R.m[1]) / s;
    } else if (R.m[0] > R.m[4] && R.m[0] > R.m[8]) {
        T s = sqrt(T(1) + R.m[0] - R.m[4] - R.m[8]) * T(2);
        w = (R.m[7] - R.m[5]) / s;
        x = T(0.25) * s;
        y = (R.m[1] + R.m[3]) / s;
        z = (R.m[2] + R.m[6]) / s;
    } else if (R.m[4] > R.m[8]) {
        T s = sqrt(T(1) + R.m[4] - R.m[0] - R.m[8]) * T(2);
        w = (R.m[2] - R.m[6]) / s;
        x = (R.m[1] + R.m[3]) / s;
        y = T(0.25) * s;
        z = (R.m[5] + R.m[7]) / s;
    } else {
        T s = sqrt(T(1) + R.m[8] - R.m[0] - R.m[4]) * T(2);
        w = (R.m[3] - R.m[1]) / s;
        x = (R.m[2] + R.m[6]) / s;
        y = (R.m[5] + R.m[7]) / s;
        z = T(0.25) * s;
    }
    if (w < T(0)) { w = -w; x = -x; y = -y; z = -z; }
    qw[0] = w; qw[1] = x; qw[2] = y; qw[3] = z;
}

// Closed-form coefficients of the two specialised chain kinds (fitted by the loader from the general
// algorithms above, see b2_model.cpp):
//   CHAIN1   : (I + dt d) q'' = tau - d dq - (E cos q + F sin q)            (revolute)
//              (I + dt d) q'' = tau - d dq - E                               (prismatic, F = 0)
//   CHAIN_PR : M(q) = [[m11, A c + B s], [A c + B s, m22]],  c = cos q2, s = sin q2
//              h = [(-A s + B c) dq2^2 + G1,  E c + F s]
template <typename T>
struct ChainCoef {
    T m11, m22, A, B, G1, E, F;
    T d1, d2;      // viscous damping
    T dt;
    int revolute;  // CHAIN1: joint type
};

// Per-env domain randomisation of the chain kinds (reference: randomizers/cartpole.py:51-56,100-135: every link
// mass + U(-d, d), gravity_z ~ N(-9.8, sigma)). The closed-form coefficients are affine in the body masses and
// the gravity terms scale with g_z, so the loader also fits d(coef)/d(mass_k) and the kernel rebuilds the
// coefficients of an env from its (mass offsets, gravity scale):
//   m11, m22, A, B = base + sum_k dm_k * dmass[k] ;  G1, E, F = gscale * (base + sum_k dm_k * dmass[k]).
template <typename T>
struct ChainBasis {
    T dmass[2][7];  // d(m11, m22, A, B, G1, E, F) / d(mass of body k)
    T mass[2];      // nominal body masses (offsets are clamped so that masses stay positive)
};

template <typename T>
B2_HD ChainCoef<T> randomized_coef(const ChainCoef<T>& base, const ChainBasis<T>& bs, int nq, const T* dm, T gscale)
{
    ChainCoef<T> c = base;
    T v[7] = {base.m11, base.m22, base.A, base.B, base.G1, base.E, base.F};
    for (int k = 0; k < nq; ++k)
        for (int i = 0; i < 7; ++i) v[i] += dm[k] * bs.dmass[k][i];
    c.m11 = v[0]; c.m22 = v[1]; c.A = v[2]; c.B = v[3];
    c.G1 = gscale * v[4]; c.E = gscale * v[5]; c.F = gscale * v[6];
    return c;
}

// The closed-form steps are written with plain operators on purpose: which product of `a b + c d` joins the FMA is left
// to the compiler, which picks the one that shortens the dependent chain in each kernel. Pinning the rounding of every
// operation (so that k_task_chain and k_task_trajectory agree bit for bit) was measured: same instruction count, same
// registers and occupancy, but 11 % more time per launch of the HBM-bound k_task_chain (86 us against 77 us at 4.2 M
// envs), because a thread's lifetime is its fp64 chain. The two kernels therefore agree to rounding, not to the bit.
// `s`, `co`: sin q / cos q of the revolute joint on entry (callers that already hold them, e.g. from the previous
// step's observation, skip the sincos).
template <typename T>
B2_HD void chain1_step_sc(const ChainCoef<T>& c, T& q, T& dq, T tau, T& ddq, T s, T co)
{
    const T g = c.revolute ? c.E * co + c.F * s : c.E;
    ddq = (tau - c.d1 * dq - g) / (c.m11 + c.dt * c.d1);
    dq += ddq * c.dt;
    q += dq * c.dt;
}
template <typename T>
B2_HD void chain1_step(const ChainCoef<T>& c, T& q, T& dq, T tau, T& ddq)
{
    T s = T(0), co = T(1);
    if (c.revolute) sincos_t(q, &s, &co);
    chain1_step_sc(c, q, dq, tau, ddq, s, co);
}

template <typename T>
B2_HD void chain_pr_step_sc(const ChainCoef<T>& c, T& x, T& q, T& dx, T& dq, T fx, T fq, T& ddx, T& ddq, T s, T co)
{
    const T m12 = c.A * co + c.B * s;
    const T r1 = fx - c.d1 * dx - ((c.B * co - c.A * s) * dq * dq + c.G1);
    const T r2 = fq - c.d2 * dq - (c.E * co + c.F * s);
    const T a11 = c.m11 + c.dt * c.d1, a22 = c.m22 + c.dt * c.d2;
    const T inv = T(1) / (a11 * a22 - m12 * m12);
    ddx = (a22 * r1 - m12 * r2) * inv;
    ddq = (a11 * r2 - m12 * r1) * inv;
    dx += ddx * c.dt;
    dq += ddq * c.dt;
    x += dx * c.dt;
    q += dq * c.dt;
}
template <typename T>
B2_HD void chain_pr_step(const ChainCoef<T>& c, T& x, T& q, T& dx, T& dq, T fx, T fq, T& ddx, T& ddq)
{
    T s, co;
    sincos_tp(q, &s, &co);
    chain_pr_step_sc(c, x, q, dx, dq, fx, fq, ddx, ddq, s, co);
}

}  // namespace b2
