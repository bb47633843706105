// CUDA kernels of the b2sim engine (sm_100a). One thread per env for the chain kinds and the generic
// tree kernel; per-env state is env-major so that a thread's loads/stores are 16-byte vectors and a
// warp touches one contiguous span.
//
// Kernels:
//   k_task_chain<TASK, T>  fused env.step for pendulum / cartpole tasks: set_action -> DART-equivalent
//                          step (closed-form chain dynamics, semi-implicit Euler) -> observation,
//                          reward, done -> Philox-keyed masked auto-reset. HBM-bound.
//   k_run_tree<T, NB>      GazeboSimulator::run for any fixed-base tree: pending resets, PID
//                          (JointController::PreUpdate), command application, ABA step, joint
//                          constraints, one-shot command clearing (Physics::Update).
//   k_kinematics / k_kindyn   link poses, mass matrix, bias forces, Jacobians.
//   small column utilities used by the per-object ScenarI/O view.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/b2sim.h"
#include "b2_rbd.hpp"
#include "b2_tree_fast.hpp"
#include "b2_contact.hpp"

namespace b2 {

// ---------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC 2011), counter = (step, env, block), key = seed.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4])
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Four 53-bit uniforms in [0, 1) for (seed, global env, step).
__device__ __forceinline__ void reset_uniforms4(uint64_t seed, uint64_t env, uint64_t step, double u[4])
{
#pragma unroll
    for (int blk = 0; blk < 2; ++blk) {
        uint32_t r[4];
        philox4x32_10((uint32_t)step, (uint32_t)(step >> 32), (uint32_t)env,
                      ((uint32_t)(env >> 32) << 8) | (uint32_t)blk, (uint32_t)seed, (uint32_t)(seed >> 32), r);
        u[2 * blk] = ((double)(r[0] >> 5) * 67108864.0 + (double)(r[1] >> 6)) / 9007199254740992.0;
        u[2 * blk + 1] = ((double)(r[2] >> 5) * 67108864.0 + (double)(r[3] >> 6)) / 9007199254740992.0;
    }
}

// Four more uniforms from Philox blocks 2 and 3 of the same (seed, env, step): domain-randomisation draws.
__device__ __forceinline__ void rand_uniforms4(uint64_t seed, uint64_t env, uint64_t step, double u[4])
{
#pragma unroll
    for (int blk = 0; blk < 2; ++blk) {
        uint32_t r[4];
        philox4x32_10((uint32_t)step, (uint32_t)(step >> 32), (uint32_t)env,
                      ((uint32_t)(env >> 32) << 8) | (uint32_t)(blk + 2), (uint32_t)seed, (uint32_t)(seed >> 32), r);
        u[2 * blk] = ((double)(r[0] >> 5) * 67108864.0 + (double)(r[1] >> 6)) / 9007199254740992.0;
        u[2 * blk + 1] = ((double)(r[2] >> 5) * 67108864.0 + (double)(r[3] >> 6)) / 9007199254740992.0;
    }
}

// Per-env physical parameters of a new episode (randomizers/cartpole.py:51-56,100-135): mass offsets
// U(-delta, delta) per body (kept above -0.9 m so that masses stay positive) and the gravity scale g_z / g_z0 with
// g_z ~ N(g_z0, sigma) by Box-Muller. out = [dm_0 .. dm_{nq-1}, gscale].
__device__ __forceinline__ void sample_rand_params(uint64_t seed, uint64_t env, uint64_t step, int nq, double delta,
                                                   double sigma, double g0, const double* mass, double* out)
{
    double u[4];
    rand_uniforms4(seed, env, step, u);
    for (int k = 0; k < nq; ++k) {
        double dm = -delta + 2.0 * delta * u[k];
        const double lo = -0.9 * mass[k];
        out[k] = dm < lo ? lo : dm;
    }
    const double z = sqrt(-2.0 * log(1.0 - u[2])) * cos(6.283185307179586 * u[3]);
    out[nq] = (g0 + sigma * z) / g0;
}

// low + (high - low) * u with each operation individually rounded (numpy's uniform()).
__device__ __forceinline__ double affine_rn(double low, double range, double u)
{
    return __dadd_rn(low, __dmul_rn(range, u));
}

#define B2_PI 3.141592653589793

// ---------------------------------------------------------------------------------------------------
// Task definitions (python/gym_ignition_environments/tasks/*.py). State layouts:
//   pendulum  [q, dq]            obs [cos q, sin q, dq]
//   cartpole  [x, q, dx, dq]     obs [x, dx, q, dq]      (joint order of the URDF: linear, pivot)
// ---------------------------------------------------------------------------------------------------
template <int TASK> struct TaskTraits;
template <> struct TaskTraits<B2_TASK_PENDULUM_SWINGUP> { static constexpr int nq = 1, nobs = 3; };
template <> struct TaskTraits<B2_TASK_CARTPOLE_DISCRETE_BALANCING> { static constexpr int nq = 2, nobs = 4; };
template <> struct TaskTraits<B2_TASK_CARTPOLE_CONTINUOUS_BALANCING> { static constexpr int nq = 2, nobs = 4; };
template <> struct TaskTraits<B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP> { static constexpr int nq = 2, nobs = 4; };

// Fresh episode state; st = [q.., dq..] in double.
template <int TASK>
__device__ __forceinline__ void sample_reset(uint64_t seed, uint64_t env, uint64_t step, double* st)
{
    double u[4];
    reset_uniforms4(seed, env, step, u);
    if (TASK == B2_TASK_PENDULUM_SWINGUP) {
        // pendulum_swingup.py:118-127: float32 Box sample, q = arctan2(sin, cos) in float32
        const float c = (float)affine_rn(-1.0, 2.0, u[0]);
        const float s = (float)affine_rn(-1.0, 2.0, u[1]);
        const float w = (float)affine_rn(-10.0, 20.0, u[2]);
        st[0] = (double)(float)atan2((double)s, (double)c);
        st[1] = (double)w;
    } else if (TASK == B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP) {
        // cartpole_continuous_swingup.py:145-146
        const double deg = affine_rn(-60.0, 120.0, u[0]);
        st[1] = __dsub_rn(B2_PI, __dmul_rn(deg, B2_PI / 180.0));
        st[0] = affine_rn(-0.05, 0.05 - (-0.05), u[1]);
        st[2] = affine_rn(-0.05, 0.05 - (-0.05), u[2]);
        st[3] = affine_rn(-0.05, 0.05 - (-0.05), u[3]);
    } else {
        // cartpole_discrete_balancing.py:137: x, dx, q, dq
        st[0] = affine_rn(-0.05, 0.05 - (-0.05), u[0]);
        st[2] = affine_rn(-0.05, 0.05 - (-0.05), u[1]);
        st[1] = affine_rn(-0.05, 0.05 - (-0.05), u[2]);
        st[3] = affine_rn(-0.05, 0.05 - (-0.05), u[3]);
    }
}

// gym.spaces.Box(dtype=float32).contains: float32-rounded bounds, inclusive, NaN -> outside.
template <typename T> __device__ __forceinline__ bool inside(T v, double high)
{
    const T h = (T)(float)high;
    return (v >= -h) && (v <= h);
}

__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }

// Observation / reward / done on a post-step state. `tau_after` is the force target the task would
// read back, which Physics has already zeroed (Physics.cpp:2250-2254).
// KEEP_SC: the caller wants sin / cos of the revolute joint angle for the next step (k_task_trajectory); the tasks
// that evaluate a cosine anyway then take it from one sincos. Returns them in sc[0], sc[1] when it computed them.
template <int TASK, typename T, bool KEEP_SC = false>
__device__ __forceinline__ bool evaluate_task(const T* st, T* obs, T& reward, T* sc = nullptr)
{
    if (TASK == B2_TASK_PENDULUM_SWINGUP) {
        const T q = st[0], dq = st[1];
        T s, c;
        sincos_t(q, &s, &c);
        if (KEEP_SC) { sc[0] = s; sc[1] = c; }
        obs[0] = c; obs[1] = s; obs[2] = dq;
        const bool done = !(inside(c, 1.0) && inside(s, 1.0) && inside(dq, 10.0));
        // cost = (100 if done) + (q^2 + 0.1 dq^2 + 0.001 tau^2), tau = 0 after the step
        const T cost = add_rn(done ? T(100) : T(0), add_rn(mul_rn(q, q), mul_rn(T(0.1), mul_rn(dq, dq))));
        reward = -cost;
        return done;
    }
    const T x = st[0], q = st[1], dx = st[2], dq = st[3];
    obs[0] = x; obs[1] = dx; obs[2] = q; obs[3] = dq;
    const double dq_thr = (3 * 360) * (B2_PI / 180.0);
    if (TASK == B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP) {
        const double q_thr = (5 * 360) * (B2_PI / 180.0);
        const bool done = !(inside(x, 2.4) && inside(dx, 20.0) && inside(q, q_thr) && inside(dq, dq_thr));
        T cq;
        if (KEEP_SC) { sincos_t(q, &sc[0], &sc[1]); cq = sc[1]; }
        else cq = cos_t(q);
        T r = mul_rn(add_rn(cq, T(1)), T(0.5));
        r = add_rn(r, -mul_rn(T(0.1), mul_rn(dx, dx)));
        r = add_rn(r, x >= T(0.8 * 2.4) ? T(-10) : T(-0.0));
        reward = r;
        return done;
    }
    const double q_thr = 12 * (B2_PI / 180.0);
    const bool done = !(inside(x, 2.4) && inside(dx, 20.0) && inside(q, q_thr) && inside(dq, dq_thr));
    const T edge = TASK == B2_TASK_CARTPOLE_DISCRETE_BALANCING ? T(0.9 * 2.4) : T(2.4);
    T r = done ? T(0) : T(1);
    r = add_rn(r, -mul_rn(T(0.1), fabs(x)));
    r = add_rn(r, -mul_rn(T(0.1), fabs(dx)));
    r = add_rn(r, x >= edge ? T(-10) : T(-0.0));
    reward = r;
    return done;
}

template <int TASK, typename T> __device__ __forceinline__ T action_force(T a)
{
    if (TASK == B2_TASK_CARTPOLE_DISCRETE_BALANCING) return a == T(1) ? T(20) : T(-20);
    return a;
}

// 16-byte vector types per scalar.
template <typename T> struct Vec16;
template <> struct Vec16<double> { using type = double2; static constexpr int n = 2; };
template <> struct Vec16<float> { using type = float4; static constexpr int n = 4; };

template <typename T, int N> __device__ __forceinline__ void load_row(const T* __restrict__ base, size_t row, T* out)
{
    using V = typename Vec16<T>::type;
    constexpr int per = Vec16<T>::n;
    if constexpr (N % per == 0) {
        const V* p = reinterpret_cast<const V*>(base + row * N);
#pragma unroll
        for (int k = 0; k < N / per; ++k) {
            V v = __ldcs(p + k);
            const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
            for (int j = 0; j < per; ++j) out[k * per + j] = e[j];
        }
    } else {
#pragma unroll
        for (int k = 0; k < N; ++k) out[k] = __ldcs(base + row * N + k);
    }
}
template <typename T, int N> __device__ __forceinline__ void store_row(T* __restrict__ base, size_t row, const T* in)
{
    using V = typename Vec16<T>::type;
    constexpr int per = Vec16<T>::n;
    if constexpr (N % per == 0) {
        V* p = reinterpret_cast<V*>(base + row * N);
#pragma unroll
        for (int k = 0; k < N / per; ++k) {
            V v;
            T* e = reinterpret_cast<T*>(&v);
#pragma unroll
            for (int j = 0; j < per; ++j) e[j] = in[k * per + j];
            __stcs(p + k, v);
        }
    } else {
#pragma unroll
        for (int k = 0; k < N; ++k) __stcs(base + row * N + k, in[k]);
    }
}

// Episode statistics accumulated by the step kernels themselves (what an RL loop logs at the end of a rollout):
// totals = [sum of returns, sum of lengths, finished episodes, non-finite rewards], kept in kStatStripes copies that a
// block picks by its index so that a step on which every env finishes (a shared TimeLimit) does not serialise a
// million atomics on four addresses; readers add the stripes up.
constexpr int kStatStripes = 32;

// Called by every thread that owns an env, after the step's reward / done are known. `length` = steps of the episode
// that just finished (TimeLimit counter before it is cleared). Full warps reduce with shuffles and issue one set of
// atomics per warp; a partial warp (the tail of the grid) falls back to per-thread atomics.
template <typename T>
__device__ __forceinline__ void episode_stats_accumulate(T* __restrict__ ep_return, double* __restrict__ ep_totals, int64_t e,
                                                         T reward, bool done, unsigned length)
{
    const bool finite = isfinite(reward);
    const T ret = ep_return[e] + (finite ? reward : T(0));
    ep_return[e] = done ? T(0) : ret;
    double v0 = done ? (double)ret : 0.0, v1 = done ? (double)length : 0.0, v2 = done ? 1.0 : 0.0, v3 = finite ? 0.0 : 1.0;
    const unsigned mask = __activemask();
    if (__ballot_sync(mask, done || !finite) == 0u) return;
    double* tot = ep_totals + 4 * (blockIdx.x % kStatStripes);
    if (mask == 0xffffffffu) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            v0 += __shfl_xor_sync(mask, v0, o);
            v1 += __shfl_xor_sync(mask, v1, o);
            v2 += __shfl_xor_sync(mask, v2, o);
            v3 += __shfl_xor_sync(mask, v3, o);
        }
        if ((threadIdx.x & 31) != 0) return;
    }
    if (v2 != 0.0) { atomicAdd(tot + 0, v0); atomicAdd(tot + 1, v1); atomicAdd(tot + 2, v2); }
    if (v3 != 0.0) atomicAdd(tot + 3, v3);
}

// Block tickets of the graph-replayed step kernels: word 0 = top level, words 1.. = one per group of kTicketGroup blocks.
// Grids of up to (kTicketWords - 1) * kTicketGroup blocks (2^26 envs at 128 threads per block) never share a group word.
constexpr int kTicketGroup = 64;
constexpr int kTicketWords = 8193;

template <typename T>
struct TaskArgs {
    T* state;                  // [N, 2 nq]
    const T* actions;          // [N, 1]
    T* obs;                    // [N, nobs]
    T* reward;                 // [N]
    uint8_t* done;             // [N]
    uint16_t* elapsed;         // [N]
    ChainCoef<T> coef;
    int64_t n;
    uint64_t seed, env_offset, step;
    int max_episode_steps;
    int iterations;            // physics iterations per env step (steps_per_run = physics_rate / agent_rate)
    // Device-side step counter (optional): when set, the Philox step index is read from it instead of `step`, and
    // the last block to finish advances it. Launches captured in a CUDA graph then stay correct across replays.
    unsigned long long* step_counter;
    unsigned int* block_ticket;
    int advance_counter;
    // per-env domain randomisation (optional): rand = [N, nq + 1] mass offsets and gravity scale
    T* rand;
    ChainBasis<T> basis;
    double mass_delta, gravity_sigma, gravity_z0, body_mass[2];
    // episode statistics (optional): per-env running return and the striped totals they are folded into on `done`
    T* ep_return;          // [N]
    double* ep_totals;     // [kStatStripes][4]
};

// One GazeboRuntime.step of one env on register-resident state, in two halves so that the callers can send the step's
// outputs on their way before the (rare) reset path runs:
//   task_env_advance  Task.set_action -> gazebo.run() -> observation, reward, done -> TimeLimit
//   task_env_reset    Task.reset_task (if done). `dm` = the env's randomised parameters, redrawn on reset when domain
//                     randomisation is on (returns true: the caller stores them and rebuilds its coefficients).
// CARRY (k_task_trajectory): sc[0..1] = sin / cos of the revolute joint angle of the state on entry when `have_sc`, and
// of the state on return for the tasks whose evaluation computes them (pendulum, swing-up); the first physics iteration
// of the next step then skips its sincos, a quarter of the instructions of a step.
template <int TASK, typename T, bool CARRY = false>
__device__ __forceinline__ bool task_env_advance(const TaskArgs<T>& a, const ChainCoef<T>& coef, T* st, unsigned& el, T action,
                                                 T* obs, T& reward, T* sc = nullptr, bool* have_sc = nullptr)
{
    constexpr int nq = TaskTraits<TASK>::nq;
    constexpr bool kEvalTrig = TASK == B2_TASK_PENDULUM_SWINGUP || TASK == B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP;
    T acc0, acc1;
    // Task.set_action: one-shot force on the actuated joint ("pivot" / "linear" = dof 0)
    const T f = action_force<TASK, T>(action);
    // gazebo.run(): Physics applies the command and advances steps_per_run iterations; the force command is
    // one-shot, so it acts on the first iteration only (Physics.cpp:2250-2254)
    for (int it = 0; it < a.iterations; ++it) {
        const T fi = it == 0 ? f : T(0);
        if (CARRY && kEvalTrig && it == 0 && *have_sc) {
            if (nq == 1) chain1_step_sc(coef, st[0], st[1], fi, acc0, sc[0], sc[1]);
            else chain_pr_step_sc(coef, st[0], st[1], st[2], st[3], fi, T(0), acc0, acc1, sc[0], sc[1]);
        } else if (nq == 1) {
            chain1_step(coef, st[0], st[1], fi, acc0);
        } else {
            chain_pr_step(coef, st[0], st[1], st[2], st[3], fi, T(0), acc0, acc1);
        }
    }
    bool done;
    if (CARRY && kEvalTrig) {
        done = evaluate_task<TASK, T, true>(st, obs, reward, sc);
        *have_sc = true;
    } else {
        done = evaluate_task<TASK, T>(st, obs, reward);
    }
    el += 1;
    done = done || (int)el >= a.max_episode_steps;  // gym.wrappers.TimeLimit
    return done;
}

template <int TASK, typename T>
__device__ __forceinline__ bool task_env_reset(const TaskArgs<T>& a, T* st, unsigned& el, int64_t e, uint64_t step, T* dm)
{
    constexpr int nq = TaskTraits<TASK>::nq;
    // Task.reset_task + paused run, fused: the next step starts from a fresh episode
    double fresh[2 * nq];
    sample_reset<TASK>(a.seed, a.env_offset + (uint64_t)e, step, fresh);
#pragma unroll
    for (int k = 0; k < 2 * nq; ++k) st[k] = (T)fresh[k];
    el = 0;
    if (a.rand) {  // the randomizer re-inserts a freshly randomised model on every reset
        double rp[nq + 1];
        sample_rand_params(a.seed, a.env_offset + (uint64_t)e, step, nq, a.mass_delta, a.gravity_sigma, a.gravity_z0,
                           a.body_mass, rp);
#pragma unroll
        for (int k = 0; k <= nq; ++k) dm[k] = (T)rp[k];
        return true;
    }
    return false;
}

// One GazeboRuntime.step for every env (python/gym_ignition/runtimes/gazebo_runtime.py:91-120).
// COUNTER = false (eager launches): the Philox step index comes from the host (`a.step`); one thread also mirrors
// the next index into the device counter. COUNTER = true (launches captured in a CUDA graph): the index is read
// from the device counter and the block that takes the last ticket advances it, so replays stay exact.
template <int TASK, typename T, bool COUNTER>
__global__ void __launch_bounds__(256) k_task_chain(const TaskArgs<T> a)
{
    constexpr int nq = TaskTraits<TASK>::nq, nobs = TaskTraits<TASK>::nobs;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // Programmatic dependent launch (eager launches carry the stream-serialization attribute): the next launch on the
    // stream may be scheduled while this grid drains, and every grid waits here until the grids before it have completed
    // and flushed their memory. Without the attribute both instructions are no-ops. One step of a small batch is one
    // wave of blocks, so the launch-to-launch gap is a large share of it (131,072 envs: 2.3 us of HBM time in ~6 us).
    asm volatile("griddepcontrol.launch_dependents;");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    uint64_t step = a.step;
    __shared__ unsigned long long s_step;
    if (COUNTER) {
        if (threadIdx.x == 0) {
            s_step = *reinterpret_cast<volatile unsigned long long*>(a.step_counter);
            // thread 0 of every block reads the counter before it takes a ticket, so the block that takes the last
            // ticket can advance the counter without racing any reader
            if (a.advance_counter) {
                // two-level tickets: groups of kTicketGroup blocks share a word and the last block of each group takes
                // the top-level ticket, so no address sees more than a few hundred atomics per launch
                __threadfence();
                const unsigned g = blockIdx.x / kTicketGroup, ng = (gridDim.x + kTicketGroup - 1) / kTicketGroup;
                const unsigned gsize = min((unsigned)kTicketGroup, gridDim.x - g * kTicketGroup);
                unsigned int* gt = a.block_ticket + 1 + g;
                if (atomicAdd(gt, 1u) == gsize - 1) {
                    *gt = 0u;
                    __threadfence();
                    if (atomicAdd(a.block_ticket, 1u) == ng - 1) {
                        *a.block_ticket = 0u;
                        *reinterpret_cast<volatile unsigned long long*>(a.step_counter) = s_step + 1ull;
                    }
                }
            }
        }
    } else if (e == 0 && a.step_counter && a.advance_counter) {
        *a.step_counter = a.step + 1ull;
    }
    const bool live = e < a.n;
    if (!COUNTER && !live) return;
    T st[2 * nq], obs[nobs], reward, dm[nq + 1];
    unsigned el = 0;
    bool done = false;
    if (live) {
        load_row<T, 2 * nq>(a.state, e, st);
        ChainCoef<T> coef = a.coef;
        if (a.rand) {  // this env's own masses and gravity
#pragma unroll
            for (int k = 0; k <= nq; ++k) dm[k] = __ldcs(a.rand + e * (nq + 1) + k);
            coef = randomized_coef(a.coef, a.basis, nq, dm, dm[nq]);
        }
        el = a.elapsed[e];
        done = task_env_advance<TASK, T>(a, coef, st, el, __ldcs(a.actions + e), obs, reward);
        store_row<T, nobs>(a.obs, e, obs);
        __stcs(a.reward + e, reward);
        a.done[e] = done ? 1 : 0;
        if (a.ep_return) episode_stats_accumulate(a.ep_return, a.ep_totals, e, reward, done, el);
    }
    if (COUNTER) {
        // the step index is only needed by the reset path: the block's barrier sits behind the step's loads, arithmetic
        // and output stores instead of in front of them (a dependent global read + barrier at the top of every block
        // cost 14 us per replayed step at 4,194,304 envs)
        __syncthreads();
        step = s_step;
        if (!live) return;
    }
    if (done && task_env_reset<TASK, T>(a, st, el, e, step, dm)) {
#pragma unroll
        for (int k = 0; k <= nq; ++k) a.rand[e * (nq + 1) + k] = dm[k];
    }
    a.elapsed[e] = (uint16_t)el;
    store_row<T, 2 * nq>(a.state, e, st);
}

// `steps` consecutive env.steps of every env in ONE launch (open-loop action sequences: synthetic rollouts, replayed
// trajectories). The env's state, episode counter and model parameters stay in registers between steps, so per step
// only the action is read and the observation / reward / done are written: small batches (BASELINE config 2,
// 65,536 envs), which are launch-bound at one launch per step, become bound by HBM instead. Results are those of
// `steps` launches of k_task_chain (same Philox step indices, same resets; states agree to rounding). Actions are [steps, n]; the trajectory
// outputs [steps, n, nobs], [steps, n], [steps, n] are optional, the per-env buffers always receive the last step.
template <int TASK, typename T>
__global__ void __launch_bounds__(64) k_task_trajectory(const TaskArgs<T> a, int steps, T* __restrict__ traj_obs,
                                                        T* __restrict__ traj_reward, uint8_t* __restrict__ traj_done)
{
    constexpr int nq = TaskTraits<TASK>::nq, nobs = TaskTraits<TASK>::nobs;
    constexpr int PF = 8;  // actions are fetched PF steps ahead of their use
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e == 0 && a.step_counter && a.advance_counter) *a.step_counter = a.step + (unsigned long long)steps;
    if (e >= a.n) return;
    T st[2 * nq], obs[nobs], reward = T(0), dm[nq + 1];
    load_row<T, 2 * nq>(a.state, e, st);
    ChainCoef<T> coef = a.coef;
    if (a.rand) {
#pragma unroll
        for (int k = 0; k <= nq; ++k) dm[k] = __ldcs(a.rand + e * (nq + 1) + k);
        coef = randomized_coef(a.coef, a.basis, nq, dm, dm[nq]);
    }
    unsigned el = a.elapsed[e];
    bool any_fresh = false, done = false, have_sc = false;
    T sc[2] = {T(0), T(1)};
    const T* __restrict__ ap = a.actions + e;
    T act[PF];
#pragma unroll
    for (int k = 0; k < PF; ++k) act[k] = k < steps ? __ldcs(ap + (int64_t)k * a.n) : T(0);
    for (int t0 = 0; t0 < steps; t0 += PF) {
#pragma unroll
        for (int k = 0; k < PF; ++k) {
            const int t = t0 + k;
            if (t < steps) {
                const T action = act[k];
                act[k] = t + PF < steps ? __ldcs(ap + (int64_t)(t + PF) * a.n) : T(0);
                done = task_env_advance<TASK, T, true>(a, coef, st, el, action, obs, reward, sc, &have_sc);
                if (traj_obs) {
                    const int64_t row = (int64_t)t * a.n + e;
                    store_row<T, nobs>(traj_obs, row, obs);
                    __stcs(traj_reward + row, reward);
                    traj_done[row] = done ? 1 : 0;
                }
                if (a.ep_return) episode_stats_accumulate(a.ep_return, a.ep_totals, e, reward, done, el);
                if (done) {
                    have_sc = false;  // the fresh episode starts from another angle
                    if (task_env_reset<TASK, T>(a, st, el, e, a.step + (uint64_t)t, dm)) {
                        any_fresh = true;
                        coef = randomized_coef(a.coef, a.basis, nq, dm, dm[nq]);
                    }
                }
            }
        }
    }
    store_row<T, nobs>(a.obs, e, obs);
    __stcs(a.reward + e, reward);
    a.done[e] = done ? 1 : 0;
    if (any_fresh) {
#pragma unroll
        for (int k = 0; k <= nq; ++k) a.rand[e * (nq + 1) + k] = dm[k];
    }
    a.elapsed[e] = (uint16_t)el;
    store_row<T, 2 * nq>(a.state, e, st);
}

// Task.get_observation / get_reward / is_done on the current state, without stepping (what
// GazeboRuntime.reset returns after its paused run, gazebo_runtime.py:122-140).
template <int TASK, typename T>
__global__ void k_task_observe(const T* __restrict__ state, T* __restrict__ obs, T* __restrict__ reward,
                               uint8_t* __restrict__ done, int64_t n)
{
    constexpr int nq = TaskTraits<TASK>::nq, nobs = TaskTraits<TASK>::nobs;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    T st[2 * nq], o[nobs], r;
    load_row<T, 2 * nq>(state, e, st);
    const bool d = evaluate_task<TASK, T>(st, o, r);
    store_row<T, nobs>(obs, e, o);
    reward[e] = r;
    done[e] = d ? 1 : 0;
}

// Initial reset of every env (step index 0 of the Philox stream).
template <int TASK, typename T>
__global__ void k_task_reset_all(T* state, uint16_t* elapsed, int64_t n, uint64_t seed, uint64_t env_offset,
                                 uint64_t step, T* rand, double mass_delta, double gravity_sigma, double gravity_z0,
                                 double mass0, double mass1)
{
    constexpr int nq = TaskTraits<TASK>::nq;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    double fresh[2 * nq];
    sample_reset<TASK>(seed, env_offset + (uint64_t)e, step, fresh);
    T st[2 * nq];
#pragma unroll
    for (int k = 0; k < 2 * nq; ++k) st[k] = (T)fresh[k];
    store_row<T, 2 * nq>(state, e, st);
    elapsed[e] = 0;
    if (rand) {
        const double mass[2] = {mass0, mass1};
        double rp[nq + 1];
        sample_rand_params(seed, env_offset + (uint64_t)e, step, nq, mass_delta, gravity_sigma, gravity_z0, mass, rp);
#pragma unroll
        for (int k = 0; k <= nq; ++k) rand[e * (nq + 1) + k] = (T)rp[k];
    }
}

// ---------------------------------------------------------------------------------------------------
// Generic path: GazeboSimulator::run for a fixed-base tree.
// ---------------------------------------------------------------------------------------------------
template <typename T>
struct RunCfg {
    int nq;
    int iterations;           // steps_per_run, or 1 when paused
    int paused;
    int controller_loaded;
    uint32_t compute_new_bits; // bit it: JointController recomputes the PID on iteration `it`
    T dt;
    uint8_t mode[kMaxDofs];
    uint8_t has_force_cmd[kMaxDofs];
    uint8_t has_vel_cmd[kMaxDofs];
    T pid[kMaxDofs][8];       // p, i, d, i_max, i_min, cmd_max, cmd_min, cmd_offset
    // ComputedTorqueFixedBase run by ControllerRunner (controllers/src/ComputedTorqueFixedBase.cpp:205-271)
    int ct_active;            // controller loaded and every reference (position, velocity, acceleration) is set
    uint32_t ct_compute_bits; // bit it: the controller recomputes the torque on iteration `it`
    T ct_kp[kMaxDofs], ct_kd[kMaxDofs];
    T ct_gravity[3];          // the controller's own gravity (context/gazebo/controllers.py:9)
    // external link wrenches with duration (Link::applyWorldWrench, Physics.cpp:1483-1532), as J^T F joint torques
    int nwrench;
    int wrench_link[4];
    int wrench_iters[4];      // applied on iterations [0, wrench_iters)
    int64_t wrench_env[4];    // -1: every env
    T wrench[4][6];           // force, torque in the world frame, applied at the link origin
};

template <typename T>
struct RunBuffers {
    T* state;        // [N, 2 nq]
    T* accel;        // [N, nq]
    T* force_cmd;    // [N, nq]
    T* force_read;   // [N, nq] JointForce readback
    T* pos_target;   // [N, nq]
    T* vel_target;   // [N, nq]
    T* pid_state;    // [N, 3 nq]
    T* reset_state;  // [N, 2 nq]
    T* acc_target;   // [N, nq]
    uint32_t* reset_mask;
    int64_t n;
};

template <typename T> __device__ __forceinline__ T clampt(T v, T lo, T hi) { return v < lo ? lo : (v > hi ? hi : v); }

// ignition::math::PID::Update (ign-math6; call site JointController.cpp:309).
template <typename T>
__device__ __forceinline__ T pid_update(const T* g, T* st /* iErr, pErrLast, cmd */, T error, T dt)
{
    if (dt == T(0) || isnan(error) || isinf(error)) return T(0);
    const T p_term = g[0] * error;
    T i_err = st[0] + g[1] * dt * error;
    if (g[3] >= g[4]) i_err = clampt(i_err, g[4], g[3]);
    const T d_err = (error - st[1]) / dt;
    T cmd = g[7] - p_term - i_err - g[2] * d_err;
    if (g[5] >= g[6]) cmd = clampt(cmd, g[6], g[5]);
    st[0] = i_err; st[1] = error; st[2] = cmd;
    return cmd;
}

// Joint-space constraint stage (joint limits, Coulomb friction, velocity servo): boxed LCP on
// w = Minv lambda + b solved by projected Gauss-Seidel, Minv from CRBA + Cholesky.
template <typename T, int NB, typename P = NominalParams<T>>
__device__ void joint_constraints(const ModelDev<T>& m, T dt, const T* q, T* dq, const uint8_t* servo,
                                  const T* servo_target, T* ddq, const P& prm = P())
{
    int rj[3 * NB];
    T rb[3 * NB], rlo[3 * NB], rhi[3 * NB], lam[3 * NB];
    int nr = 0;
    const int nq = m.nq;
    const T inf = T(INFINITY);
    for (int j = 0; j < nq; ++j) {
        if (servo[j]) {
            rj[nr] = j; rb[nr] = dq[j] - servo_target[j]; rlo[nr] = -m.effort[j] * dt; rhi[nr] = m.effort[j] * dt; ++nr;
            continue;
        }
        const T friction = prm.friction(m, j);
        if (friction != T(0)) { rj[nr] = j; rb[nr] = dq[j]; rlo[nr] = -friction * dt; rhi[nr] = friction * dt; ++nr; }
        if (q[j] <= m.lower[j]) { rj[nr] = j; rb[nr] = dq[j]; rlo[nr] = T(0); rhi[nr] = inf; ++nr; }
        if (q[j] >= m.upper[j]) { rj[nr] = j; rb[nr] = dq[j]; rlo[nr] = -inf; rhi[nr] = T(0); ++nr; }
    }
    if (nr == 0) return;
    T M[NB * NB], Minv[NB * NB];
    mass_matrix<T, NB>(m, q, M, prm);
    spd_inverse(nq, M, Minv);
    for (int a = 0; a < nr; ++a) lam[a] = T(0);
    for (int it = 0; it < 200; ++it) {
        T change = T(0);
        for (int a = 0; a < nr; ++a) {
            T w = rb[a];
            for (int c = 0; c < nr; ++c) w += Minv[rj[a] * nq + rj[c]] * lam[c];
            const T nl = clampt(lam[a] - w / Minv[rj[a] * nq + rj[a]], rlo[a], rhi[a]);
            change += fabs(nl - lam[a]);
            lam[a] = nl;
        }
        if (change < T(1e-18)) break;
    }
    for (int i = 0; i < nq; ++i) {
        T dv = T(0);
        for (int a = 0; a < nr; ++a) dv += Minv[i * nq + rj[a]] * lam[a];
        dq[i] += dv;
        ddq[i] += dv / dt;
    }
}

// Branching information of the tree (which bodies park their children's articulated inertia in scratch).
struct TreeTopo {
    int nbranch;
    int slot[kMaxDofs];
    int has_friction;  // any joint with Coulomb friction: the constraint stage always runs
    int impulse_ok;    // no joint damping / stiffness: constraint rows can use the articulated-body impulse path
};

template <typename T>
__device__ __forceinline__ void stage_model(const ModelDev<T>* __restrict__ tables, ModelDev<T>& m)
{
    static_assert(sizeof(ModelDev<T>) % 16 == 0, "ModelDev is copied in 16-byte pieces");
    const uint4* src = reinterpret_cast<const uint4*>(tables);
    uint4* dst = reinterpret_cast<uint4*>(&m);
    for (int k = threadIdx.x; k < (int)(sizeof(ModelDev<T>) / 16); k += blockDim.x) dst[k] = __ldg(src + k);
    __syncthreads();
}

// The world description (free bodies, static shapes, robot shapes) into shared memory, 16 bytes per thread and step.
// The caller's barrier (stage_model's, or its own __syncthreads) publishes it.
template <typename T>
__device__ __forceinline__ void stage_world(const WorldDev<T>* __restrict__ world, WorldDev<T>& W)
{
    static_assert(sizeof(WorldDev<T>) % 16 == 0, "WorldDev is copied in 16-byte pieces");
    const uint4* src = reinterpret_cast<const uint4*>(world);
    uint4* dst = reinterpret_cast<uint4*>(&W);
    for (int k = threadIdx.x; k < (int)(sizeof(WorldDev<T>) / 16); k += blockDim.x) dst[k] = __ldg(src + k);
}

// Rare path: some joint sits on a limit, has Coulomb friction or is velocity-servoed. Kept out of line so the
// common path stays lean; works on local copies of q / dq. `prm`: an env's EnvParams, or nothing for the model's tables.
template <typename T, typename W, typename... P>
__device__ __noinline__ void constraints_from_scratch(const ModelDev<T>& m, T dt, const W& w, uint32_t servo_bits,
                                                      const T* __restrict__ vel_target_row, P... prm)
{
    T q[kMaxDofs], dq[kMaxDofs], ddq[kMaxDofs], target[kMaxDofs];
    uint8_t servo[kMaxDofs];
    const int nq = m.nq;
    for (int j = 0; j < nq; ++j) {
        q[j] = w[kSlotsPerBody * j + SL_Q];
        dq[j] = w[kSlotsPerBody * j + SL_DQ];
        ddq[j] = w[kSlotsPerBody * j + SL_TAU];
        servo[j] = (servo_bits >> j) & 1u;
        target[j] = servo[j] ? vel_target_row[j] : T(0);
    }
    joint_constraints<T, kMaxDofs>(m, dt, q, dq, servo, target, ddq, prm...);
    for (int j = 0; j < nq; ++j) {
        w[kSlotsPerBody * j + SL_DQ] = dq[j];
        w[kSlotsPerBody * j + SL_TAU] = ddq[j];
    }
}

// Hook of the constraint stage. NoCoupling: the joint rows of the tree are solved on their own. A coupled world
// (CoupledWorld, further down) solves them together with the contacts between the tree's link shapes, free bodies
// and static shapes.
struct NoCoupling {
    static constexpr bool active = false;
    static constexpr bool deferred = false;
    static constexpr bool keeps_M = false;          // wants the controller's M(q) for its constraint rows
    static constexpr bool keeps_reset_mask = false; // leaves the pending-reset mask for the kernels that run next to it
};
template <typename T, typename C> __device__ __forceinline__ T* mass_matrix_slot(C& c, bool valid)
{
    if constexpr (C::keeps_M) { c.have_M = valid; return valid ? c.Mq : nullptr; }
    else return nullptr;
}

// One physics iteration on the scratch state: ABA -> dq += ddq dt -> joint constraints -> q += dq dt.
// SL_TAU holds the applied force on entry and the joint acceleration on return.
// P: NominalParams, or the env's EnvParams (then topo.impulse_ok only covers the stiffness; the env's damping decides too).
template <typename T, typename W, typename C, typename P = NominalParams<T>>
__device__ __forceinline__ void tree_physics_iteration(const ModelDev<T>& m, const TreeTopo& topo, T dt, const W& w,
                                                       uint32_t servo_bits, const T* __restrict__ vel_target_row, C& coupling,
                                                       const P& prm = P())
{
    const int nq = m.nq;
    clear_parking_t<T>(nq, topo.nbranch, w);
    forward_dynamics_fast(m, topo.slot, dt, w, prm);
    for (int j = 0; j < nq; ++j) {
        const int o = kSlotsPerBody * j;
        w[o + SL_DQ] += w[o + SL_TAU] * dt;
    }
    if constexpr (C::active) {
        coupling.solve(m, dt, w, servo_bits, vel_target_row);
    } else {
        int rj[kMaxRows];
        T rb[kMaxRows], rlo[kMaxRows], rhi[kMaxRows];
        const int nr = collect_rows(m, dt, w, servo_bits, vel_target_row, rj, rb, rlo, rhi, prm);
        if constexpr (P::nominal) {
            if (nr > 0 && topo.impulse_ok) constraints_fast(m, dt, w, nr, rj, rb, rlo, rhi);
            else if (nr != 0) constraints_from_scratch(m, dt, w, servo_bits, vel_target_row);
        } else {
            if (nr > 0 && topo.impulse_ok && prm.undamped(m)) constraints_fast(m, dt, w, nr, rj, rb, rlo, rhi);
            else if (nr != 0) constraints_from_scratch(m, dt, w, servo_bits, vel_target_row, prm);
        }
    }
    if constexpr (!C::deferred) {  // deferred: the finishing kernel integrates after the warp-cooperative solve
        for (int j = 0; j < nq; ++j) {
            const int o = kSlotsPerBody * j;
            w[o + SL_Q] += w[o + SL_DQ] * dt;
        }
    }
}

// JointController::PreUpdate for one env (JointController.cpp:114-287): PID joints write JointForceCmd.
template <typename T, typename W>
__device__ __forceinline__ void tree_pid(const RunCfg<T>& cfg, const RunBuffers<T>& b, int64_t e, const W& w,
                                         bool compute_new)
{
    const int nq = cfg.nq;
    for (int j = 0; j < nq; ++j) {
        const int md = cfg.mode[j];
        if (md == B2_MODE_POSITION || md == B2_MODE_VELOCITY) {
            T* ps = b.pid_state + e * 3 * nq + 3 * j;
            const T cur = md == B2_MODE_POSITION ? w[kSlotsPerBody * j + SL_Q] : w[kSlotsPerBody * j + SL_DQ];
            const T ref = md == B2_MODE_POSITION ? b.pos_target[e * nq + j] : b.vel_target[e * nq + j];
            T st[3] = {ps[0], ps[1], ps[2]};
            T f = st[2];
            if (compute_new) {
                f = pid_update(cfg.pid[j], st, cur - ref, cfg.dt);
                ps[0] = st[0]; ps[1] = st[1]; ps[2] = st[2];
            }
            b.force_cmd[e * nq + j] = f;
        }
    }
}

// ComputedTorqueFixedBase::step: tau = M(q) (ddq_ref - kp (q - q_ref) - kd (dq - dq_ref)) + h(q, dq), with the
// mass matrix and bias forces of the controller's own model / gravity. The torque is kept in the PID `cmd` slot
// so that it can be re-applied between controller updates.
template <typename T, typename W>
__device__ __noinline__ void computed_torque(const ModelDev<T>& m, const RunCfg<T>& cfg, const RunBuffers<T>& b, int64_t e,
                                             const W& w, T* M_keep = nullptr)
{
    const int nq = m.nq;
    T q[kMaxDofs], dq[kMaxDofs], zero[kMaxDofs], h[kMaxDofs], acc[kMaxDofs], M_own[kMaxDofs * kMaxDofs];
    T* const M = M_keep ? M_keep : M_own;  // a coupled world reuses M(q) for its constraint rows
    for (int j = 0; j < nq; ++j) {
        q[j] = w[kSlotsPerBody * j + SL_Q];
        dq[j] = w[kSlotsPerBody * j + SL_DQ];
        zero[j] = T(0);
        acc[j] = b.acc_target[e * nq + j] - cfg.ct_kp[j] * (q[j] - b.pos_target[e * nq + j]) -
                 cfg.ct_kd[j] * (dq[j] - b.vel_target[e * nq + j]);
    }
    mass_matrix<T, kMaxDofs>(m, q, M);
    inverse_dynamics<T, kMaxDofs>(m, q, dq, zero, true, h, cfg.ct_gravity);
    for (int i = 0; i < nq; ++i) {
        T tau = h[i];
        for (int j = 0; j < nq; ++j) tau += M[i * nq + j] * acc[j];
        b.pid_state[e * 3 * nq + 3 * i + 2] = tau;
    }
}

// Adds J^T F of the active external link wrenches to the joint forces in the SL_TAU slots.
template <typename T, typename W>
__device__ __noinline__ void add_wrench_torques(const ModelDev<T>& m, const RunCfg<T>& cfg, int64_t e, int it, const W& w)
{
    for (int k = 0; k < cfg.nwrench; ++k) {
        if ((cfg.wrench_env[k] >= 0 && cfg.wrench_env[k] != e) || it >= cfg.wrench_iters[k]) continue;
        const int link = cfg.wrench_link[k], body = m.link_body[link];
        if (body < 0) continue;
        int chain[kMaxDofs], depth = 0;
        for (int i = body; i >= 0; i = m.parent[i]) chain[depth++] = i;
        M3<T> Rw = ld9(m.baseR);
        V3<T> pw = ld3(m.basep);
        V3<T> aw[kMaxDofs], po[kMaxDofs];
        for (int d = depth - 1; d >= 0; --d) {
            const int i = chain[d];
            const T q = w[kSlotsPerBody * i + SL_Q];
            T s = T(0), c = T(1);
            if (m.jtype[i] == kRevolute) sincos_t(q, &s, &c);
            M3<T> R;
            V3<T> p;
            joint_pose_sc(m, i, s, c, q, R, p);
            pw = pw + mul(Rw, p);
            Rw = mul(Rw, R);
            aw[d] = mul(Rw, ld3(m.axis[i]));
            po[d] = pw;
        }
        const V3<T> pl = pw + mul(Rw, ld3(m.link_p[link]));
        const V3<T> f = v3(cfg.wrench[k][0], cfg.wrench[k][1], cfg.wrench[k][2]);
        const V3<T> t = v3(cfg.wrench[k][3], cfg.wrench[k][4], cfg.wrench[k][5]);
        for (int d = 0; d < depth; ++d) {
            const int i = chain[d];
            const T gen = m.jtype[i] == kRevolute ? dot(cross(aw[d], pl - po[d]), f) + dot(aw[d], t) : dot(aw[d], f);
            w[kSlotsPerBody * i + SL_TAU] += gen;
        }
    }
}

// GazeboSimulator::run for every env of a fixed-base tree. One thread per env; per-thread scratch columns in
// dynamic shared memory (scratch_slots(nq, nbranch) * blockDim.x scalars). `prm` feeds the physics only: the
// computed-torque controller keeps the nominal model (it loads its own copy of the model file in the reference).
template <typename T, typename W, typename C, typename P = NominalParams<T>>
__device__ __forceinline__ void run_tree_env(const ModelDev<T>& m, const RunCfg<T>& cfg, const RunBuffers<T>& b,
                                             const TreeTopo& topo, int64_t e, const W& w, C& coupling, const P& prm = P())
{
    const int nq = cfg.nq;
    for (int j = 0; j < nq; ++j) {
        w[kSlotsPerBody * j + SL_Q] = b.state[e * 2 * nq + j];
        w[kSlotsPerBody * j + SL_DQ] = b.state[e * 2 * nq + nq + j];
    }
    const bool control = !cfg.paused && cfg.controller_loaded;
    // PreUpdate of the first iteration sees the last readback, i.e. the state before pending resets are
    // consumed by Physics::Update
    if (control) tree_pid(cfg, b, e, w, cfg.compute_new_bits & 1u);
    const bool ct = !cfg.paused && cfg.ct_active;
    // Physics::UpdatePhysics: velocity reset, then position reset (Physics.cpp:1330-1375)
    const uint32_t mask = b.reset_mask[e];
    // the controller's M(q) stays valid for the constraint stage of this iteration unless a position reset moves q
    if (ct && (cfg.ct_compute_bits & 1u)) computed_torque(m, cfg, b, e, w, mass_matrix_slot<T>(coupling, (mask & 0xffffu) == 0));
    if (mask) {
        for (int j = 0; j < nq; ++j) {
            if (mask & (1u << (16 + j))) w[kSlotsPerBody * j + SL_DQ] = b.reset_state[e * 2 * nq + nq + j];
            if (mask & (1u << j)) w[kSlotsPerBody * j + SL_Q] = b.reset_state[e * 2 * nq + j];
        }
        if constexpr (!C::keeps_reset_mask) b.reset_mask[e] = 0;
    }
    bool stepped = false;
    for (int it = 0; it < cfg.iterations; ++it) {
        if (control && it > 0) tree_pid(cfg, b, e, w, (cfg.compute_new_bits >> it) & 1u);
        if (ct && it > 0 && ((cfg.ct_compute_bits >> it) & 1u)) computed_torque(m, cfg, b, e, w, mass_matrix_slot<T>(coupling, true));
        if (ct)  // ControllerRunner re-applies the last torque every iteration (ControllerRunner.cpp:276-281)
            for (int j = 0; j < nq; ++j) b.force_cmd[e * nq + j] = b.pid_state[e * 3 * nq + 3 * j + 2];
        uint32_t servo_bits = 0;
        for (int j = 0; j < nq; ++j) {
            const int md = cfg.mode[j];
            const bool pid_joint = cfg.controller_loaded && (md == B2_MODE_POSITION || md == B2_MODE_VELOCITY);
            T tau = T(0);
            if (cfg.has_force_cmd[j] || (pid_joint && !cfg.paused)) {
                tau = b.force_cmd[e * nq + j];
            } else if (md == B2_MODE_VELOCITY_FOLLOWER_DART && !cfg.paused && !(mask & (1u << (16 + j)))) {
                servo_bits |= 1u << j;  // JointVelocityCmd = target (JointController.cpp:263-286)
            }
            w[kSlotsPerBody * j + SL_TAU] = tau;
            // UpdateSim: one-shot commands are zeroed after every iteration (Physics.cpp:2250-2267)
            b.force_read[e * nq + j] = cfg.paused ? tau : T(0);
            b.force_cmd[e * nq + j] = T(0);
        }
        if (!cfg.paused) {
            if (cfg.nwrench) add_wrench_torques(m, cfg, e, it, w);
            tree_physics_iteration(m, topo, cfg.dt, w, servo_bits, b.vel_target + e * nq, coupling, prm);
            stepped = true;
        }
    }
    for (int j = 0; j < nq; ++j) {
        b.state[e * 2 * nq + j] = w[kSlotsPerBody * j + SL_Q];
        b.state[e * 2 * nq + nq + j] = w[kSlotsPerBody * j + SL_DQ];
        if (stepped) b.accel[e * nq + j] = w[kSlotsPerBody * j + SL_TAU];
    }
}

// Per-env physical parameters of a model (b2sim_enable_env_params): B2_BUF_BODY_INERTIA [N][nq][10],
// B2_BUF_JOINT_DYNAMICS [N][nq][2], B2_BUF_GRAVITY [N][3] (layouts: EnvParams, b2_rbd.hpp).
template <typename T>
struct EnvRows {
    const T* inertia = nullptr;
    const T* dyn = nullptr;
    const T* grav = nullptr;
    __host__ __device__ EnvParams<T> env(int64_t e, int nq) const
    {
        return EnvParams<T>{inertia + e * kEnvInertiaCols * nq, dyn + e * kEnvJointCols * nq, grav + 3 * e};
    }
};
template <typename T, bool ENV> struct ParamsOf { using type = NominalParams<T>; };
template <typename T> struct ParamsOf<T, true> { using type = EnvParams<T>; };
template <bool ENV, typename T> __device__ __forceinline__ typename ParamsOf<T, ENV>::type params_of(const EnvRows<T>& rows, int64_t e, int nq)
{
    if constexpr (ENV) return rows.env(e, nq);
    else return NominalParams<T>{};
}

// Shared-memory scratch: 64 threads per block, scratch_slots * 64 scalars of dynamic shared memory.
// ENV: the physics reads every env's own inertias, damping, friction and gravity from `rows`.
template <typename T, bool ENV = false>
__global__ void __launch_bounds__(64) k_run_tree(const ModelDev<T>* __restrict__ tables, const RunCfg<T> cfg,
                                                 const RunBuffers<T> b, const TreeTopo topo, const EnvRows<T> rows)
{
    __shared__ ModelDev<T> m;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= b.n) return;
    NoCoupling none;
    run_tree_env(m, cfg, b, topo, e, Scratch<T>{reinterpret_cast<T*>(smem_raw) + threadIdx.x, (int)blockDim.x}, none,
                 params_of<ENV>(rows, e, cfg.nq));
}

// Local-memory scratch (L1 / L2 backed): more resident threads per SM, for large env counts.
template <typename T, bool ENV = false>
__global__ void __launch_bounds__(128) k_run_tree_local(const ModelDev<T>* __restrict__ tables, const RunCfg<T> cfg,
                                                        const RunBuffers<T> b, const TreeTopo topo, const EnvRows<T> rows)
{
    __shared__ ModelDev<T> m;
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= b.n) return;
    T buf[kSlotsPerBody * kMaxDofs + kSlotsPerBranch * kMaxBranch];
    NoCoupling none;
    run_tree_env(m, cfg, b, topo, e, Scratch<T, 1>{buf, 1}, none, params_of<ENV>(rows, e, cfg.nq));
}

// ---------------------------------------------------------------------------------------------------------
// Fused Panda task (BASELINE config C4): position PID at the physics rate (models/panda.py gains,
// tests/test_scenario/test_pid_controllers.py) -> articulated-body step -> KinDyn-style observation
//   obs[115] = q(9), dq(9), end-effector position(3) + quaternion wxyz(4), MIXED frame Jacobian 6 x (6+9)
// (rbd/idyntree/kindyncomputations.py:169-176,367-377), reward = -|p_ee - goal|, done on the TimeLimit only,
// reset = models/panda.py initial configuration. One thread per env, scratch columns in shared memory,
// global I/O staged through the scratch so that every global access of a block is contiguous.
// ---------------------------------------------------------------------------------------------------------
constexpr int kPandaObs = 115;  // 2*9 + 7 + 6*(6+9) for the 9-DoF Panda; panda_obs_size(nq) in general
__host__ __device__ inline int panda_obs_size(int nq) { return 2 * nq + 7 + 6 * (6 + nq); }

template <typename T>
struct PandaArgs {
    T* state;          // [N, 2 nq]
    const T* targets;  // [N, nq] joint position targets (the action)
    T* pid_state;      // [N, 3 nq]
    T* obs;            // [N, 115]
    T* reward;
    uint8_t* done;
    uint16_t* elapsed;
    int64_t n;
    int nq, iterations, max_episode_steps, ee_link;
    int ee_body;       // body the end-effector link is attached to (ModelDev::link_body[ee_link])
    int observe_only;  // compute obs / reward / done of the current state: no step, no TimeLimit tick, no reset
    T dt;
    T goal[3];
    T q0[kMaxDofs];
    T pid[kMaxDofs][8];
    T* ep_return;          // episode statistics (optional), see episode_stats_accumulate
    double* ep_totals;
};

// Copies rows [row0, row0 + rows) of a [N, cols] global array into scratch slots (coalesced global reads).
template <typename T, typename SlotOf>
__device__ __forceinline__ void block_load(const T* __restrict__ g, int64_t row0, int rows, int cols, T* scratch, int stride,
                                           SlotOf slot_of)
{
    const int total = rows * cols;
    const T* src = g + row0 * cols;
    for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
        const int r = idx / cols, k = idx - r * cols;
        scratch[slot_of(k) * stride + r] = __ldcs(src + idx);
    }
}
template <typename T, typename SlotOf>
__device__ __forceinline__ void block_store(T* __restrict__ g, int64_t row0, int rows, int cols, const T* scratch, int stride,
                                            SlotOf slot_of)
{
    const int total = rows * cols;
    T* dst = g + row0 * cols;
    for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
        const int r = idx / cols, k = idx - r * cols;
        __stcs(dst + idx, scratch[slot_of(k) * stride + r]);
    }
}

// Writes `cols` values per lane (vals[0..cols) of each lane = one row of a [N, cols] array, lane l owning row
// row0 + l) through a per-warp shared-memory tile, so that global stores go out as contiguous 128-byte pieces of
// each row instead of 32 scattered 8-byte stores per instruction.
constexpr int kTileCols = 16;
template <typename T>
__device__ __forceinline__ void warp_store_rows(T* __restrict__ g, int64_t row0, int rows, int cols, const T* vals, T* tile)
{
    const int lane = threadIdx.x & 31;
    for (int c0 = 0; c0 < cols; c0 += kTileCols) {
        const int nc = min(kTileCols, cols - c0);
        for (int k = 0; k < nc; ++k) tile[lane * (kTileCols + 1) + k] = vals[c0 + k];
        __syncwarp();
        if (nc == kTileCols) {
            // full tile: two rows per store instruction, 128 contiguous bytes each
#pragma unroll
            for (int it = 0; it < kTileCols; ++it) {
                const int r = 2 * it + (lane >> 4), k = lane & (kTileCols - 1);
                if (r < rows) __stcs(g + (row0 + r) * cols + c0 + k, tile[r * (kTileCols + 1) + k]);
            }
        } else {
            for (int idx = lane; idx < 32 * nc; idx += 32) {
                const int r = idx / nc, k = idx - r * nc;
                if (r < rows) __stcs(g + (row0 + r) * cols + c0 + k, tile[r * (kTileCols + 1) + k]);
            }
        }
        __syncwarp();
    }
}

// ENV: the physics reads every env's own inertias, damping, Coulomb friction and gravity from `rows`
// (b2sim_enable_env_params); the observation is kinematic and reads none of them.
template <typename T, bool ENV = false>
__global__ void __launch_bounds__(128) k_task_panda(const ModelDev<T>* __restrict__ tables, const PandaArgs<T> a, const TreeTopo topo,
                                                    const EnvRows<T> rows)
{
    __shared__ ModelDev<T> m;
    __shared__ T tiles[4][32 * (kTileCols + 1)];
    stage_model(tables, m);
    const int nq = a.nq;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int warp = threadIdx.x >> 5;
    const int64_t warp_row0 = e - (threadIdx.x & 31);
    const int warp_rows = (int)max((int64_t)0, min((int64_t)32, a.n - warp_row0));
    const bool active = e < a.n;
    // per-thread scratch in local memory (L1 / L2 backed): physics slots, then the observation vector
    T buf[kSlotsPerBody * kMaxDofs + kSlotsPerBranch * kMaxBranch];
    T out[kPandaObs + 1];
    T pst[3 * kMaxDofs];
    const Scratch<T, 1> w{buf, 1};
    const int nobs = panda_obs_size(nq);
    if (active) {
        unsigned el = a.elapsed[e];
        for (int j = 0; j < nq; ++j) {
            w[kSlotsPerBody * j + SL_Q] = __ldcs(a.state + e * 2 * nq + j);
            w[kSlotsPerBody * j + SL_DQ] = __ldcs(a.state + e * 2 * nq + nq + j);
        }
        for (int k = 0; k < 3 * nq; ++k) pst[k] = __ldcs(a.pid_state + e * 3 * nq + k);
        for (int it = 0; it < a.iterations; ++it) {
            // JointController::PreUpdate: error = current - reference, force = pid.Update(error, dt)
            for (int j = 0; j < nq; ++j) {
                const T target = __ldg(a.targets + e * nq + j);
                w[kSlotsPerBody * j + SL_TAU] = pid_update(a.pid[j], pst + 3 * j, w[kSlotsPerBody * j + SL_Q] - target, a.dt);
            }
            NoCoupling none;
            tree_physics_iteration(m, topo, a.dt, w, 0u, (const T*)nullptr, none, params_of<ENV>(rows, e, nq));
        }
        // ---- forward kinematics along the chain to the end effector (world axis / origin go to the V slots) ----
        const int body = m.link_body[a.ee_link];
        int chain[kMaxDofs], depth = 0;
        unsigned on_chain = 0;
        for (int i = body; i >= 0; i = m.parent[i]) { chain[depth++] = i; on_chain |= 1u << i; }
        M3<T> Rw = ld9(m.baseR);
        V3<T> pw = ld3(m.basep);
        for (int d = depth - 1; d >= 0; --d) {
            const int i = chain[d], o = kSlotsPerBody * i;
            const T q = w[o + SL_Q];
            T s = T(0), c = T(1);
            if (m.jtype[i] == kRevolute) sincos_t(q, &s, &c);
            M3<T> R;
            V3<T> p;
            joint_pose_sc(m, i, s, c, q, R, p);
            pw = pw + mul(Rw, p);
            Rw = mul(Rw, R);
            const V3<T> aw = mul(Rw, ld3(m.axis[i]));
            w[o + SL_V + 0] = aw.x; w[o + SL_V + 1] = aw.y; w[o + SL_V + 2] = aw.z;
            w[o + SL_V + 3] = pw.x; w[o + SL_V + 4] = pw.y; w[o + SL_V + 5] = pw.z;
        }
        const V3<T> pe = pw + mul(Rw, ld3(m.link_p[a.ee_link]));
        const M3<T> Re = mul(Rw, ld9(m.link_R[a.ee_link]));
        // ---- observation vector ----
        for (int j = 0; j < nq; ++j) {
            out[j] = w[kSlotsPerBody * j + SL_Q];
            out[nq + j] = w[kSlotsPerBody * j + SL_DQ];
        }
        int k = 2 * nq;
        out[k + 0] = pe.x; out[k + 1] = pe.y; out[k + 2] = pe.z;
        rot_to_quat(Re, out + k + 3);
        k += 7;
        const int ncol = 6 + nq;
        const V3<T> r = pe - ld3(m.basep);
        for (int rr = 0; rr < 6; ++rr)
            for (int c = 0; c < 6; ++c) out[k + rr * ncol + c] = rr == c ? T(1) : T(0);
        out[k + 0 * ncol + 4] = r.z;  out[k + 0 * ncol + 5] = -r.y;   // -S(p_ee - p_base)
        out[k + 1 * ncol + 3] = -r.z; out[k + 1 * ncol + 5] = r.x;
        out[k + 2 * ncol + 3] = r.y;  out[k + 2 * ncol + 4] = -r.x;
        for (int j = 0; j < nq; ++j) {
            V3<T> lin = v3(T(0), T(0), T(0)), ang = lin;
            if ((on_chain >> j) & 1u) {
                const int o = kSlotsPerBody * j;
                const V3<T> aw = v3(w[o + SL_V + 0], w[o + SL_V + 1], w[o + SL_V + 2]);
                const V3<T> po = v3(w[o + SL_V + 3], w[o + SL_V + 4], w[o + SL_V + 5]);
                if (m.jtype[j] == kRevolute) { lin = cross(aw, pe - po); ang = aw; }
                else lin = aw;
            }
            out[k + 0 * ncol + 6 + j] = lin.x; out[k + 1 * ncol + 6 + j] = lin.y; out[k + 2 * ncol + 6 + j] = lin.z;
            out[k + 3 * ncol + 6 + j] = ang.x; out[k + 4 * ncol + 6 + j] = ang.y; out[k + 5 * ncol + 6 + j] = ang.z;
        }
        const V3<T> gd = pe - v3(a.goal[0], a.goal[1], a.goal[2]);
        a.reward[e] = -sqrt(dot(gd, gd));
        if (!a.observe_only) el += 1;
        const bool done = !a.observe_only && (int)el >= a.max_episode_steps;  // gym TimeLimit; the task itself never terminates
        a.done[e] = done ? 1 : 0;
        if (a.ep_return && !a.observe_only) episode_stats_accumulate(a.ep_return, a.ep_totals, e, a.reward[e], done, el);
        if (done) {  // Task.reset_task + paused run: models/panda.py initial configuration, PID reset
            for (int j = 0; j < nq; ++j) {
                w[kSlotsPerBody * j + SL_Q] = a.q0[j];
                w[kSlotsPerBody * j + SL_DQ] = T(0);
            }
            for (int c = 0; c < 3 * nq; ++c) pst[c] = T(0);
            el = 0;
        }
        a.elapsed[e] = (uint16_t)el;
    }
    // every lane of a warp takes part in the tiled stores (inactive lanes own no row)
    warp_store_rows(a.obs, warp_row0, warp_rows, nobs, out, tiles[warp]);
    if (!a.observe_only) {
        T st[2 * kMaxDofs];
        if (active)
            for (int j = 0; j < nq; ++j) {
                st[j] = w[kSlotsPerBody * j + SL_Q];
                st[nq + j] = w[kSlotsPerBody * j + SL_DQ];
            }
        warp_store_rows(a.state, warp_row0, warp_rows, 2 * nq, st, tiles[warp]);
        warp_store_rows(a.pid_state, warp_row0, warp_rows, 3 * nq, pst, tiles[warp]);
    }
}

// Link world poses [N, 7 nlinks] (xyz + quaternion wxyz), Link.cpp:71-103.
template <typename T, int NB>
__global__ void __launch_bounds__(128) k_kinematics(const ModelDev<T>* __restrict__ tables, const T* __restrict__ state,
                                                    T* __restrict__ link_pose, int64_t n)
{
    __shared__ ModelDev<T> m;
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int nq = m.nq;
    T q[NB];
    M3<T> Rw[NB];
    V3<T> pw[NB];
    for (int j = 0; j < nq; ++j) q[j] = state[e * 2 * nq + j];
    forward_kinematics<T, NB>(m, q, Rw, pw);
    const M3<T> Rb = ld9(m.baseR);
    const V3<T> pb = ld3(m.basep);
    for (int l = 0; l < m.nlinks; ++l) {
        const int body = m.link_body[l];
        const M3<T> R = mul(body >= 0 ? Rw[body] : Rb, ld9(m.link_R[l]));
        const V3<T> p = (body >= 0 ? pw[body] : pb) + mul(body >= 0 ? Rw[body] : Rb, ld3(m.link_p[l]));
        T* out = link_pose + (e * m.nlinks + l) * 7;
        out[0] = p.x; out[1] = p.y; out[2] = p.z;
        rot_to_quat(R, out + 3);
    }
}

// KinDyn: mass matrix, bias forces, frame Jacobian (MIXED: world orientation, linear rows first).
template <typename T, int NB>
__global__ void __launch_bounds__(128) k_kindyn(const ModelDev<T>* __restrict__ tables, const T* __restrict__ state,
                                                int link, T* __restrict__ M_out, T* __restrict__ h_out,
                                                T* __restrict__ J_out, int64_t n)
{
    __shared__ ModelDev<T> m;
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int nq = m.nq;
    T q[NB], dq[NB];
    for (int j = 0; j < nq; ++j) {
        q[j] = state[e * 2 * nq + j];
        dq[j] = state[e * 2 * nq + nq + j];
    }
    if (M_out) {
        T M[NB * NB];
        mass_matrix<T, NB>(m, q, M);
        for (int k = 0; k < nq * nq; ++k) M_out[e * nq * nq + k] = M[k];
    }
    if (h_out) {
        T zero[NB], h[NB];
        for (int j = 0; j < nq; ++j) zero[j] = T(0);
        inverse_dynamics<T, NB>(m, q, dq, zero, true, h);
        for (int j = 0; j < nq; ++j) h_out[e * nq + j] = h[j];
    }
    if (J_out) {
        M3<T> Rw[NB];
        V3<T> pw[NB];
        forward_kinematics<T, NB>(m, q, Rw, pw);
        T* J = J_out + e * 6 * nq;
        for (int k = 0; k < 6 * nq; ++k) J[k] = T(0);
        const int body = m.link_body[link];
        if (body >= 0) {
            const V3<T> pt = pw[body] + mul(Rw[body], ld3(m.link_p[link]));
            for (int i = body; i >= 0; i = m.parent[i]) {
                const V3<T> aw = mul(Rw[i], ld3(m.axis[i]));
                if (m.jtype[i] == kRevolute) {
                    const V3<T> lin = cross(aw, pt - pw[i]);
                    J[0 * nq + i] = lin.x; J[1 * nq + i] = lin.y; J[2 * nq + i] = lin.z;
                    J[3 * nq + i] = aw.x; J[4 * nq + i] = aw.y; J[5 * nq + i] = aw.z;
                } else {
                    J[0 * nq + i] = aw.x; J[1 * nq + i] = aw.y; J[2 * nq + i] = aw.z;
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Free bodies + contacts: one thread per env steps every free body of its world (b2_contact.hpp).
// ---------------------------------------------------------------------------------------------------------
template <typename T>
struct WorldBuffers {
    T* base_state[kMaxFree];       // [N, 13] per free body
    T* base_reset[kMaxFree];       // [N, 13] pending Model::resetBase* values
    uint32_t* reset_mask[kMaxFree];// bit 0: pose pending, bit 1: velocity pending
    T* base_accel[kMaxFree];       // [N, 6] per free body: (velocity after - velocity before the step) / dt, linear then angular
    int32_t* contact_count;        // [N]
    int32_t* contact_ids;          // [N, kMaxContacts, 4]: free body a, shape of a, b (free body or -1 - static shape), 0
    T* contact_data;               // [N, kMaxContacts, 10]: position, normal (b -> a), depth, force on a
    int64_t n;
    int paused;
};

template <typename T>
__device__ __forceinline__ void write_contact_records(const WorldBuffers<T>& b, int64_t e, const Contact<T>* cs, int nc, T dt)
{
    b.contact_count[e] = nc;
    for (int k = 0; k < nc; ++k) {
        int32_t* id = b.contact_ids + (e * kMaxContacts + k) * 4;
        id[0] = cs[k].a; id[1] = cs[k].shape_a; id[2] = cs[k].b; id[3] = 0;
        T* o = b.contact_data + (e * kMaxContacts + k) * kContactRec;
        const V3<T> f = contact_force(cs[k], dt);
        o[0] = cs[k].pos.x; o[1] = cs[k].pos.y; o[2] = cs[k].pos.z;
        o[3] = cs[k].n.x; o[4] = cs[k].n.y; o[5] = cs[k].n.z;
        o[6] = cs[k].depth;
        o[7] = f.x; o[8] = f.y; o[9] = f.z;
    }
}

// Loads the free bodies of env e and consumes pending Model::resetBasePose / resetBaseWorldVelocity values
// (WorldPoseCmd / WorldVelocityCmd, Physics.cpp:1535-1590,1716-1753), paused or not.
template <typename T>
__device__ __forceinline__ void load_free_bodies(const WorldDev<T>& W, const WorldBuffers<T>& b, int64_t e, T* X)
{
    for (int i = 0; i < W.nfree; ++i) {
        for (int k = 0; k < 13; ++k) X[13 * i + k] = b.base_state[i][e * 13 + k];
        const uint32_t mask = b.reset_mask[i][e];
        if (mask) {
            if (mask & 1u)
                for (int k = 0; k < 7; ++k) X[13 * i + k] = b.base_reset[i][e * 13 + k];
            if (mask & 2u)
                for (int k = 7; k < 13; ++k) X[13 * i + k] = b.base_reset[i][e * 13 + k];
            b.reset_mask[i][e] = 0;
        }
    }
}

// Acceleration of free body i over the step that took its 13 state values from `before` to `after`: the change of the
// world velocity of the base origin and of the angular velocity divided by dt. DART folds the velocity change of the
// constraint stage into the accelerations the same way (GenericJoint::updateConstrainedTerms), which is what
// Link::world{Linear,Angular}Acceleration read back (Physics.cpp:2040-2079).
template <typename T>
__device__ __forceinline__ void write_base_accel(const WorldBuffers<T>& b, int i, int64_t e, const T* vel_before /* 6 */,
                                                 const T* after /* 13 */, T dt)
{
    T* o = b.base_accel[i] + e * 6;
    const T idt = T(1) / dt;
    for (int k = 0; k < 6; ++k) o[k] = (after[7 + k] - vel_before[k]) * idt;
}

// ENV: the world kernels read the per-env rows of `rows` (WorldEnv) wherever a slot has them; otherwise the shared world
// description (WorldNominal), and `rows` is not read. The rows come last, so the ENV = false kernels keep their parameter
// layout; __grid_constant__: the coupled stages reach them through a pointer without a local copy.
template <bool ENV, typename T>
__device__ __forceinline__ auto world_params(const WorldRows<T>& rows, int64_t e)
{
    if constexpr (ENV) return WorldEnv<T>{rows, (long long)e};
    else return WorldNominal<T>{};
}
template <typename T, bool ENV> struct WorldRowsRef {
    __device__ __forceinline__ WorldNominal<T> params(int64_t) const { return {}; }
};
template <typename T> struct WorldRowsRef<T, true> {
    const WorldRows<T>* rows;
    __device__ __forceinline__ WorldEnv<T> params(int64_t e) const { return WorldEnv<T>{*rows, (long long)e}; }
};
template <bool ENV, typename T> __device__ __forceinline__ WorldRowsRef<T, ENV> rows_ref(const WorldRows<T>& rows)
{
    if constexpr (ENV) return WorldRowsRef<T, true>{&rows};
    else return WorldRowsRef<T, false>{};
}

template <typename T, bool ENV = false>
__global__ void __launch_bounds__(64) k_world_free(const WorldDev<T>* __restrict__ world, const WorldBuffers<T> b,
                                                   const __grid_constant__ WorldRows<T> rows)
{
    __shared__ WorldDev<T> W;
    stage_world(world, W);
    __syncthreads();
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= b.n) return;
    T X[kMaxFree * 13];
    load_free_bodies(W, b, e, X);
    if (!b.paused) {
        T before[kMaxFree * 6];
        for (int i = 0; i < W.nfree; ++i)
            for (int k = 0; k < 6; ++k) before[6 * i + k] = X[13 * i + 7 + k];
        Contact<T> cs[kMaxContacts];
        const int nc = world_step(W, X, cs, (long long)e, world_params<ENV>(rows, e));
        write_contact_records(b, e, cs, nc, W.dt);
        for (int i = 0; i < W.nfree; ++i) write_base_accel(b, i, e, before + 6 * i, X + 13 * i, W.dt);
    }
    for (int i = 0; i < W.nfree; ++i)
        for (int k = 0; k < 13; ++k) b.base_state[i][e * 13 + k] = X[13 * i + k];
}

// ---------------------------------------------------------------------------------------------------------
// Coupled world (BASELINE config C5, examples/panda_pick_and_place.py): a fixed-base tree whose moving links carry
// collision shapes (the Panda's fingers), free bodies (the cube) and static shapes (table, ground). One thread per
// env runs the whole GazeboSimulator::run iteration: controllers -> ABA -> unconstrained velocities of the tree and
// of the free bodies -> contact points -> ONE projected Gauss-Seidel solve over the tree's joint rows and every
// contact (b2_contact.hpp coupled_step) -> position integration -> contact records.
// ---------------------------------------------------------------------------------------------------------
template <typename T, bool ENV = false>
struct CoupledWorld : WorldRowsRef<T, ENV> {
    static constexpr bool active = true;
    static constexpr bool deferred = false;
    static constexpr bool keeps_M = false;
    static constexpr bool keeps_reset_mask = false;
    const WorldDev<T>& W;
    const WorldBuffers<T>& wb;
    int64_t e;
    T* X;

    template <typename Wk>
    __device__ __noinline__ void solve(const ModelDev<T>& m, T dt, const Wk& w, uint32_t servo_bits,
                                       const T* __restrict__ vel_target_row)
    {
        const int nq = m.nq;
        T q[kMaxDofs], dq[kMaxDofs], before[kMaxDofs];
        for (int j = 0; j < nq; ++j) {
            q[j] = w[kSlotsPerBody * j + SL_Q];
            dq[j] = before[j] = w[kSlotsPerBody * j + SL_DQ];
        }
        Contact<T> cs[kMaxContacts];
        RobotWork<T> rw;
        T vel_before[kMaxFree * 6];
        for (int i = 0; i < W.nfree; ++i)
            for (int k = 0; k < 6; ++k) vel_before[6 * i + k] = X[13 * i + 7 + k];
        const int nc = coupled_step(W, m, q, dq, servo_bits, vel_target_row, X, cs, rw, (long long)e, this->params(e));
        for (int i = 0; i < W.nfree; ++i) write_base_accel(wb, i, e, vel_before + 6 * i, X + 13 * i, dt);
        for (int j = 0; j < nq; ++j) {
            w[kSlotsPerBody * j + SL_DQ] = dq[j];
            w[kSlotsPerBody * j + SL_TAU] += (dq[j] - before[j]) / dt;
        }
        write_contact_records(wb, e, cs, nc, dt);
    }
};

// Single-thread variant: the whole coupled step, solve included, in one launch (worlds whose generalized velocity
// does not fit the warp-cooperative solver).
template <typename T, bool ENV = false>
__global__ void __launch_bounds__(64) k_world_coupled(const ModelDev<T>* __restrict__ tables, const RunCfg<T> cfg,
                                                      const RunBuffers<T> b, const TreeTopo topo,
                                                      const WorldDev<T>* __restrict__ world, const WorldBuffers<T> wb,
                                                      const __grid_constant__ WorldRows<T> rows)
{
    __shared__ ModelDev<T> m;
    __shared__ WorldDev<T> W;
    stage_world(world, W);
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= b.n) return;
    T X[kMaxFree * 13];
    load_free_bodies(W, wb, e, X);
    T buf[kSlotsPerBody * kMaxDofs + kSlotsPerBranch * kMaxBranch];
    CoupledWorld<T, ENV> cw{rows_ref<ENV>(rows), W, wb, e, X};
    run_tree_env(m, cfg, b, topo, e, Scratch<T, 1>{buf, 1}, cw);
    for (int i = 0; i < W.nfree; ++i)
        for (int k = 0; k < 13; ++k) wb.base_state[i][e * 13 + k] = X[13 * i + k];
}

// ---------------------------------------------------------------------------------------------------------
// Three-launch pipeline of a world step with contacts (the default):
//   k_world_prepare / k_coupled_prepare  one thread per env: controllers + ABA of the articulated model,
//                                        unconstrained free-body velocities, contact points, dense rows -> HBM
//   k_pgs_solve                          one warp per env, lane = one constraint row: projected Gauss-Seidel in impulse
//                                        space (A = J M^-1 J^T in shared memory). At 4,096 envs this is what fills
//                                        the GPU: 4,096 threads would be 128 warps for 592 schedulers.
//   k_world_finish                       one thread per env: joint / free-body integration, contact forces
// ---------------------------------------------------------------------------------------------------------
template <typename T>
struct PgsBuffers {
    T* v;      // [N, nvp]
    T* J;      // [N, kMaxPgsRows, nvp]
    T* par;    // [N, kMaxPgsRows, 4]
    T* aux;    // [N, aux_stride] M^-1 of the articulated model, inverse mass / inertia of the free bodies
    T* Y;      // [N, kMaxPgsRows, nvp] rows of M^-1 J^T, written and read by the solver's generic path only
    T* lam;    // [N, kMaxPgsRows]
    int* cnt;  // [N, 2] rows, joint rows
    int nvp, nq, nfree, aux_stride;
    int64_t n;
};

template <typename T>
__device__ __forceinline__ PgsEnv<T> pgs_env(const PgsBuffers<T>& g, int64_t e)
{
    return PgsEnv<T>{g.v + e * g.nvp, g.J + e * kMaxPgsRows * g.nvp, g.par + e * kMaxPgsRows * 4, g.aux + e * g.aux_stride,
                     g.cnt + 2 * e, g.nvp};
}

// Contact records without the forces (filled by k_world_finish once the impulses are known).
template <typename T>
__device__ __forceinline__ void write_contact_geometry(const WorldBuffers<T>& b, int64_t e, const Contact<T>* cs, int nc)
{
    b.contact_count[e] = nc;
    for (int k = 0; k < nc; ++k) {
        int32_t* id = b.contact_ids + (e * kMaxContacts + k) * 4;
        id[0] = cs[k].a; id[1] = cs[k].shape_a; id[2] = cs[k].b; id[3] = 0;
        T* o = b.contact_data + (e * kMaxContacts + k) * kContactRec;
        o[0] = cs[k].pos.x; o[1] = cs[k].pos.y; o[2] = cs[k].pos.z;
        o[3] = cs[k].n.x; o[4] = cs[k].n.y; o[5] = cs[k].n.z;
        o[6] = cs[k].depth;
    }
}

template <typename T, bool ENV = false>
__global__ void __launch_bounds__(64) k_world_prepare(const WorldDev<T>* __restrict__ world, const WorldBuffers<T> b,
                                                      const PgsBuffers<T> g, const __grid_constant__ WorldRows<T> rows)
{
    __shared__ WorldDev<T> W;
    stage_world(world, W);
    __syncthreads();
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= b.n) return;
    T X[kMaxFree * 13];
    load_free_bodies(W, b, e, X);
    for (int i = 0; i < W.nfree; ++i)  // resets are consumed here: the finishing kernel starts from this state
        for (int k = 0; k < 13; ++k) b.base_state[i][e * 13 + k] = X[13 * i + k];
    if (b.paused) return;
    BodyWork<T> bw[kMaxFree];
    Contact<T> cs[kMaxContacts];
    const auto prm = world_params<ENV>(rows, e);
    bodies_begin(W, X, bw, (long long)e, prm);
    int nc = 0;
    free_contacts(W, bw, cs, nc, prm);
    contact_frames(cs, nc);
    write_dense_rows(W, (const ModelDev<T>*)nullptr, 0, (const RobotWork<T>*)nullptr, bw, cs, nc, pgs_env(g, e));
    write_contact_geometry(b, e, cs, nc);
}

template <typename T, bool ENV = false>
struct CoupledPrepare : WorldRowsRef<T, ENV> {
    static constexpr bool active = true;
    static constexpr bool deferred = true;
    static constexpr bool keeps_M = true;
    static constexpr bool keeps_reset_mask = false;
    const WorldDev<T>& W;
    const WorldBuffers<T>& wb;
    const PgsBuffers<T>& g;
    int64_t e;
    const T* X;
    bool have_M;                    // Mq holds M(q) of this iteration (left by the computed-torque controller)
    T Mq[kMaxDofs * kMaxDofs];

    template <typename Wk>
    __device__ __noinline__ void solve(const ModelDev<T>& m, T dt, const Wk& w, uint32_t servo_bits,
                                       const T* __restrict__ vel_target_row)
    {
        const int nq = m.nq;
        T q[kMaxDofs], dq[kMaxDofs];
        for (int j = 0; j < nq; ++j) {
            q[j] = w[kSlotsPerBody * j + SL_Q];
            dq[j] = w[kSlotsPerBody * j + SL_DQ];
        }
        BodyWork<T> bw[kMaxFree];
        Contact<T> cs[kMaxContacts];
        RobotWork<T> rw;
        int nc = coupled_prepare_rows(W, m, q, dq, servo_bits, vel_target_row, X, have_M ? Mq : (const T*)nullptr, bw, cs, rw, true, (long long)e,
                                      this->params(e));
        write_dense_rows(W, &m, nq, &rw, bw, cs, nc, pgs_env(g, e));
        write_contact_geometry(wb, e, cs, nc);
        have_M = false;
    }
};

template <typename T, bool ENV = false>
__global__ void __launch_bounds__(64) k_coupled_prepare(const ModelDev<T>* __restrict__ tables, const RunCfg<T> cfg,
                                                        const RunBuffers<T> b, const TreeTopo topo,
                                                        const WorldDev<T>* __restrict__ world, const WorldBuffers<T> wb,
                                                        const PgsBuffers<T> g, const __grid_constant__ WorldRows<T> rows)
{
    __shared__ ModelDev<T> m;
    __shared__ WorldDev<T> W;
    stage_world(world, W);
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= b.n) return;
    T X[kMaxFree * 13];
    load_free_bodies(W, wb, e, X);
    for (int i = 0; i < W.nfree; ++i)
        for (int k = 0; k < 13; ++k) wb.base_state[i][e * 13 + k] = X[13 * i + k];
    T buf[kSlotsPerBody * kMaxDofs + kSlotsPerBranch * kMaxBranch];
    CoupledPrepare<T, ENV> cp{rows_ref<ENV>(rows), W, wb, g, e, X, false};
    // leaves q (not yet integrated), the unconstrained dq and ddq in the state / acceleration buffers
    run_tree_env(m, cfg, b, topo, e, Scratch<T, 1>{buf, 1}, cp);
}

// ---------------------------------------------------------------------------------------------------------
// Split prepare (unpaused steps): k_coupled_prepare is one dependent chain per env, and at the 4,096 envs of BASELINE
// config 5 the step time IS that chain (one warp per SM, the machine idle). Its three parts only share the joint
// positions, so they run as three kernels on forked streams and the chain becomes the longest of them:
//   k_coupled_dynamics  controllers, articulated-body algorithm, dq += ddq dt   -> joint part of v0, state bookkeeping
//   k_coupled_rows      kinematics, free-body velocities, contact points, frames -> Jacobian rows, bounds, free part of v0
//   k_coupled_minv      M(q) and its inverse                                     -> aux
// All three read q as run_tree_env sees it (pending position resets applied); the pending-reset mask of the articulated
// model is left in place by k_coupled_dynamics and cleared by k_world_finish. k_coupled_dynamics rewrites q in the state
// buffer with the value the other two derive on their own, so their concurrent reads see the same number either way.
// ---------------------------------------------------------------------------------------------------------
// Shared-memory carve-out (percent) of the three forked kernels and of k_run_tree_lanes<COUPLED>, which replaces
// k_coupled_dynamics on small batches: they must share SMs, and an SM has one shared-memory / L1 split at a time
// (b2_sim.cu, launch_coupled).
constexpr int kCoupledCarveout = 25;

template <typename T>
struct CoupledDynamics {
    static constexpr bool active = true;
    static constexpr bool deferred = true;
    static constexpr bool keeps_M = false;
    static constexpr bool keeps_reset_mask = true;
    T* v;  // this env's row of PgsBuffers::v

    template <typename Wk>
    __device__ __forceinline__ void solve(const ModelDev<T>& m, T, const Wk& w, uint32_t, const T* __restrict__)
    {
        for (int j = 0; j < m.nq; ++j) v[j] = w[kSlotsPerBody * j + SL_DQ];
    }
};

template <typename T>
__global__ void __launch_bounds__(64) k_coupled_dynamics(const ModelDev<T>* __restrict__ tables, const RunCfg<T> cfg,
                                                         const RunBuffers<T> b, const TreeTopo topo, const PgsBuffers<T> g)
{
    __shared__ ModelDev<T> m;
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= b.n) return;
    T buf[kSlotsPerBody * kMaxDofs + kSlotsPerBranch * kMaxBranch];
    CoupledDynamics<T> cd{g.v + e * g.nvp};
    run_tree_env(m, cfg, b, topo, e, Scratch<T, 1>{buf, 1}, cd);
}

// Joint positions of env e as the physics iteration sees them: pending position resets applied (Physics.cpp:1352-1375).
template <typename T>
__device__ __forceinline__ uint32_t load_positions(const RunBuffers<T>& b, int nq, int64_t e, T* q)
{
    const uint32_t mask = b.reset_mask[e];
    for (int j = 0; j < nq; ++j) q[j] = (mask & (1u << j)) ? b.reset_state[e * 2 * nq + j] : b.state[e * 2 * nq + j];
    return mask;
}

template <typename T, bool ENV = false>
__global__ void __launch_bounds__(64) k_coupled_rows(const ModelDev<T>* __restrict__ tables, const RunCfg<T> cfg,
                                                     const RunBuffers<T> b, const WorldDev<T>* __restrict__ world,
                                                     const WorldBuffers<T> wb, const PgsBuffers<T> g,
                                                     const __grid_constant__ WorldRows<T> rows)
{
    __shared__ ModelDev<T> m;
    __shared__ WorldDev<T> W;
    stage_world(world, W);
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= b.n) return;
    const int nq = m.nq;
    T X[kMaxFree * 13];
    load_free_bodies(W, wb, e, X);
    for (int i = 0; i < W.nfree; ++i)  // resets are consumed here: the finishing kernel starts from this state
        for (int k = 0; k < 13; ++k) wb.base_state[i][e * 13 + k] = X[13 * i + k];
    T q[kMaxDofs], dq[kMaxDofs];
    const uint32_t mask = load_positions(b, nq, e, q);
    uint32_t servo_bits = 0;  // the joints run_tree_env puts under a velocity servo
    for (int j = 0; j < nq; ++j) {
        const int md = cfg.mode[j];
        const bool pid_joint = cfg.controller_loaded && (md == B2_MODE_POSITION || md == B2_MODE_VELOCITY);
        if (!(cfg.has_force_cmd[j] || pid_joint) && md == B2_MODE_VELOCITY_FOLLOWER_DART && !(mask & (1u << (16 + j))))
            servo_bits |= 1u << j;
        dq[j] = T(0);  // the rows do not depend on the joint velocities; v0 comes from k_coupled_dynamics
    }
    BodyWork<T> bw[kMaxFree];
    Contact<T> cs[kMaxContacts];
    RobotWork<T> rw;
    int nc = coupled_prepare_rows(W, m, q, dq, servo_bits, b.vel_target + e * nq, X, (const T*)nullptr, bw, cs, rw, false, (long long)e,
                                  world_params<ENV>(rows, e));
    write_dense_rows(W, &m, nq, &rw, bw, cs, nc, pgs_env(g, e), false);
    write_contact_geometry(wb, e, cs, nc);
}

template <typename T>
__global__ void __launch_bounds__(64) k_coupled_minv(const ModelDev<T>* __restrict__ tables, const RunBuffers<T> b,
                                                     const PgsBuffers<T> g)
{
    __shared__ ModelDev<T> m;
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= b.n) return;
    const int nq = m.nq;
    T q[kMaxDofs], M[kMaxDofs * kMaxDofs], Minv[kMaxDofs * kMaxDofs];
    load_positions(b, nq, e, q);
    mass_matrix<T, kMaxDofs>(m, q, M);
    spd_inverse(nq, M, Minv);
    T* aux = g.aux + e * g.aux_stride;
    for (int k = 0; k < nq * nq; ++k) aux[k] = Minv[k];
}

// ---------------------------------------------------------------------------------------------------------
// k_pgs_solve: projected Gauss-Seidel over the rows of every env; NVP (16 or 32) lanes per env, lane = one UNIT.
//
// Impulse-space form (what DART's constraint solver builds too): A = J M^-1 J^T, residual velocities w = J v - c and
//     lambda_r <- clamp(lambda_r - w_r / A_rr),   w += A[:, r] dlambda_r
// A unit is up to three consecutive rows solved by one lane: the normal / t1 / t2 rows of one contact, or three
// joint rows. Per round the owner lane of unit c solves its rows in sequence in registers (its own 3x3 diagonal block
// couples them), the three impulse changes are broadcast with shuffles, and every lane updates its three residuals
// with the 3x3 block A[own rows][rows of c] (9 FMAs). That is exactly the sequential sweep of b2_contact.hpp (joint
// rows, then the rows of every contact), so the results agree with it to rounding, at a third of the shuffle /
// clamp / loop instructions per row of a one-row-per-lane mapping, and two envs share a warp when NVP = 16.
// Shared memory holds only the lower block triangle of A (kFastUnits (kFastUnits + 1) / 2 blocks of 9 scalars,
// 7.6 KB per env in fp64): 28 envs are resident per SM, which puts the 4,096 envs of BASELINE config 5 in one wave.
// Lane i reads block (max(i, c), min(i, c)), transposed through its load offsets when c > i.
// At the end v = v0 + M^-1 J^T lambda. Envs with more than kFastUnits units (rare: > 13 simultaneous contact points)
// take the streaming velocity-space path (pgs_generic), which keeps the rows in L1 / L2.
// ---------------------------------------------------------------------------------------------------------
// N scalars (N a multiple of the 16-byte vector width) from a 16-byte aligned row, with 16-byte loads.
template <typename T, int N> __device__ __forceinline__ void load_row16(const T* __restrict__ row, T* out)
{
    using V = typename Vec16<T>::type;
    constexpr int per = Vec16<T>::n;
    static_assert(N % per == 0, "row length must be a multiple of the vector width");
    const V* p = reinterpret_cast<const V*>(row);
#pragma unroll
    for (int k = 0; k < N / per; ++k) {
        const V v = p[k];
        const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
        for (int j = 0; j < per; ++j) out[k * per + j] = e[j];
    }
}

template <typename T, int NVP>
__device__ __forceinline__ T group_sum(T x)
{
#pragma unroll
    for (int o = NVP / 2; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

// This lane's entry of Y = M^-1 J^T for one row: joints through the lane's row of the joint-space M^-1, free-body lanes
// through 1 / mass (linear part) or the lane's row of the world inverse inertia (angular part). `Jrow(k)`: entry k of the row.
template <typename T, typename F>
__device__ __forceinline__ T y_entry(int nq, int nfree, const T* __restrict__ aux, int i, F Jrow)
{
    if (i < nq) {
        T y = T(0);
        for (int j = 0; j < nq; ++j) y += aux[i * nq + j] * Jrow(j);
        return y;
    }
    const int f = i - nq;
    if (f >= 6 * nfree) return T(0);
    const int b = f / 6, c = f - 6 * b;
    const T* a = aux + nq * nq + 10 * b;
    if (c < 3) return a[0] * Jrow(i);
    const int o = nq + 6 * b + 3;
    return a[1 + (c - 3) * 3] * Jrow(o) + a[2 + (c - 3) * 3] * Jrow(o + 1) + a[3 + (c - 3) * 3] * Jrow(o + 2);
}

// Streaming velocity-space path, 32 lanes per env (lanes >= nvp idle): lane = generalized velocity, a row is a
// butterfly reduction of J v, a contact is a block of three rows solved with its own 3x3 coupling terms.
// Rows, Y = M^-1 J^T (written to g.Y first) and parameters come from L1 / L2; impulses live in `scratch`.
template <typename T>
__device__ __noinline__ void pgs_generic(const PgsBuffers<T>& g, int64_t e, int lane, int nr, int njr, int iterations,
                                         T* scratch /* >= 2 * kMaxPgsRows + 3 * kMaxContacts scalars */)
{
    const int nvp = g.nvp;
    const bool on_lane = lane < nvp;
    const int col = on_lane ? lane : 0;
    T* const sL = scratch;
    T* const sK = scratch + 2 * kMaxPgsRows;
    const int nc = (nr - njr) / 3;
    const T* __restrict__ gJ = g.J + e * kMaxPgsRows * nvp + col;
    T* __restrict__ gY = g.Y + e * kMaxPgsRows * nvp + col;
    T* __restrict__ gp = g.par + e * kMaxPgsRows * 4;
    const T* __restrict__ aux = g.aux + e * g.aux_stride;
    for (int r = lane; r < 2 * kMaxPgsRows; r += 32) sL[r] = T(0);
    for (int r = 0; r < nr; ++r) {  // Y rows and reciprocal effective masses
        const T* row = g.J + e * kMaxPgsRows * nvp + r * nvp;
        const T y = on_lane ? y_entry(g.nq, g.nfree, aux, lane, [&](int k) { return row[k]; }) : T(0);
        if (on_lane) gY[r * nvp] = y;
        const T jy = group_sum<T, 32>(on_lane ? gJ[r * nvp] * y : T(0));
        if (lane == 0) gp[4 * r + 1] = T(1) / jy;
    }
    __syncwarp();
    auto J = [&](int r) { return on_lane ? gJ[r * nvp] : T(0); };
    auto Y = [&](int r) { return on_lane ? gY[r * nvp] : T(0); };
    for (int k = 0; k < nc; ++k) {
        const int r = njr + 3 * k;
        const T jn = J(r), jt = J(r + 1);
        const T a = group_sum<T, 32>(jn * Y(r + 1)), b = group_sum<T, 32>(jn * Y(r + 2)), c = group_sum<T, 32>(jt * Y(r + 2));
        if (lane == 0) { sK[3 * k] = a; sK[3 * k + 1] = b; sK[3 * k + 2] = c; }
    }
    __syncwarp();
    T v = on_lane ? g.v[e * nvp + lane] : T(0);
    for (int it = 0; it < iterations; ++it) {
        const T* rd = sL + (it & 1) * kMaxPgsRows;
        T* wr = sL + ((it + 1) & 1) * kMaxPgsRows;
        for (int a = 0; a < njr; ++a) {
            const T c = gp[4 * a], ik = gp[4 * a + 1], lo = gp[4 * a + 2], hi = gp[4 * a + 3], old = rd[a];
            const T w = group_sum<T, 32>(J(a) * v);
            T nl = old + (c - w) * ik;
            nl = nl < lo ? lo : (nl > hi ? hi : nl);
            v += Y(a) * (nl - old);
            if (lane == 0) wr[a] = nl;
        }
        for (int k = 0; k < nc; ++k) {
            const int r = njr + 3 * k;
            const T c0 = gp[4 * r], i0 = gp[4 * r + 1], i1 = gp[4 * r + 5], i2 = gp[4 * r + 9], mu = gp[4 * r + 6];
            const T k01 = sK[3 * k], k02 = sK[3 * k + 1], k12 = sK[3 * k + 2];
            const T l0 = rd[r], l1 = rd[r + 1], l2 = rd[r + 2];
            const T Y0 = Y(r), Y1 = Y(r + 1), Y2 = Y(r + 2);
            const T w0 = group_sum<T, 32>(J(r) * v), w1 = group_sum<T, 32>(J(r + 1) * v), w2 = group_sum<T, 32>(J(r + 2) * v);
            T n0 = l0 + (c0 - w0) * i0;
            n0 = n0 > T(0) ? n0 : T(0);
            const T d0 = n0 - l0, lim = mu * n0;
            T n1 = l1 - (w1 + k01 * d0) * i1;
            n1 = n1 < -lim ? -lim : (n1 > lim ? lim : n1);
            const T d1 = n1 - l1;
            T n2 = l2 - (w2 + k02 * d0 + k12 * d1) * i2;
            n2 = n2 < -lim ? -lim : (n2 > lim ? lim : n2);
            const T d2 = n2 - l2;
            v += Y0 * d0 + Y1 * d1 + Y2 * d2;
            if (lane == 0) { wr[r] = n0; wr[r + 1] = n1; wr[r + 2] = n2; }
        }
        __syncwarp();
    }
    if (on_lane) g.v[e * nvp + lane] = v;
    const T* fin = sL + (iterations & 1) * kMaxPgsRows;
    for (int r = lane; r < nr; r += 32) g.lam[e * kMaxPgsRows + r] = fin[r];
}

constexpr int kFastUnits = 13;   // units (3 rows each) of an env whose A is kept in shared memory
constexpr int kFastBlocks = kFastUnits * (kFastUnits + 1) / 2;
// M^-1 and the inverse inertias of the free bodies are staged next to the blocks: nq <= NVP - 6 joints and
// (NVP - nq) / 6 free bodies fit NVP lanes
template <int NVP> constexpr int pgs_aux_cap() { return NVP == 16 ? 112 : 320; }
// shared memory of one env in scalars: lower block triangle of A, staged aux, v0 / J^T lambda
template <typename T, int NVP>
constexpr int pgs_smem_per_env() { return (kFastBlocks * 9 + pgs_aux_cap<NVP>() + NVP + 1) / 2 * 2; }
static_assert(kFastBlocks * 9 >= 2 * kMaxPgsRows + 3 * kMaxContacts, "the streaming path borrows the A area");
static_assert(kFastUnits <= 16, "one lane per unit, 16 lanes per env when NVP = 16");

template <typename T> __device__ __forceinline__ T clamp_sel(T x, T lo, T hi) { return x < lo ? lo : (x > hi ? hi : x); }

template <typename T, int NVP>
__global__ void __launch_bounds__(64, 7) k_pgs_solve(const PgsBuffers<T> g, int iterations)
{
    constexpr int EPW = 32 / NVP;  // envs per warp
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int half = lane / NVP, li = lane % NVP;  // env of the warp, lane of the env = unit index
    T* const sS = reinterpret_cast<T*>(smem_raw) + (warp * EPW + half) * pgs_smem_per_env<T, NVP>();  // blocks [p (p + 1) / 2 + q][9]
    T* const sAux = sS + kFastBlocks * 9;                                                           // [aux_stride]
    T* const sG = sAux + pgs_aux_cap<NVP>();                                                        // v0, then J^T lambda
    const int64_t e = ((int64_t)blockIdx.x * (blockDim.x >> 5) + warp) * EPW + half;
    const bool valid = e < g.n;
    const int64_t ee = valid ? e : 0;
    const int nr = valid ? g.cnt[2 * ee] : 0, njr = valid ? g.cnt[2 * ee + 1] : 0;
    const int nju = (njr + 2) / 3, nun = nju + (nr - njr) / 3;  // joint units, units
    const bool fast = nr > 0 && nun <= kFastUnits && g.aux_stride <= pgs_aux_cap<NVP>();
    const bool slow = nr > 0 && !fast;
    const int U = fast ? nun : 0;
    int Uw = U;  // rounds per sweep: the larger unit count of the envs that share the warp (extra rounds change nothing)
#pragma unroll
    for (int o = NVP; o < 32; o <<= 1) Uw = max(Uw, __shfl_xor_sync(0xffffffffu, Uw, o));
    const int nq = g.nq, nfree = g.nfree, nv = nq + 6 * nfree;
    const T* __restrict__ gJ = g.J + ee * kMaxPgsRows * NVP;
    const T* __restrict__ gp = g.par + ee * kMaxPgsRows * 4;
    // row of (unit u, slot a), -1 if the unit has no such row
    auto row_of = [&](int u, int a) {
        if (u >= U) return -1;
        if (u < nju) return 3 * u + a < njr ? 3 * u + a : -1;
        return njr + 3 * (u - nju) + a;
    };
    if (Uw > 0) {
        // ---- M^-1, the inverse inertias of the free bodies and v0 go through shared memory (every lane needs all) ----
        for (int k = li; k < g.aux_stride; k += NVP) sAux[k] = g.aux[ee * g.aux_stride + k];
        const T v0_own = g.v[ee * NVP + li];
        sG[li] = v0_own;
        __syncwarp();
        // ---- this lane's unit, one of its rows (slot b) at a time: Y row in registers, initial residual, bounds, and
        //      column b of every block A[rows of c][rows of i]; the lane keeps the blocks with c <= i ----
        // bounds of slot b as affine functions of the unit's slot-0 impulse n0: [loA + loB n0, hiA + hiB n0]
        // (joint and normal rows: constants; friction rows: -/+ mu n0), so the sweep needs no per-row branching
        T w[3], lam[3] = {T(0), T(0), T(0)}, pik[3], loA[3], loB[3], hiA[3], hiB[3];
        const int Ti = li * (li + 1) / 2;
        const bool keeper = li < kFastUnits;
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            const int r = row_of(li, b);
            const bool on = r >= 0;
            T Yb[NVP];
            {
                const T* row = gJ + (on ? r : 0) * NVP;
                T jr[NVP];
                load_row16<T, NVP>(row, jr);  // 16-byte loads: a row is NVP scalars, aligned to its own size
#pragma unroll
                for (int i = 0; i < NVP; ++i) jr[i] = on ? jr[i] : T(0);
                T jv = T(0);
#pragma unroll
                for (int i = 0; i < NVP; ++i) {
                    Yb[i] = i < nv ? y_entry(nq, nfree, sAux, i, [&](int k) { return jr[k]; }) : T(0);
                    jv += jr[i] * sG[i];
                }
                const bool friction = on && li >= nju && b > 0;
                const T c = on ? gp[4 * r] : T(0), p2 = on ? gp[4 * r + 2] : T(0), p3 = on ? gp[4 * r + 3] : T(0);
                loA[b] = friction ? T(0) : p2; loB[b] = friction ? -p2 : T(0);
                hiA[b] = friction ? T(0) : p3; hiB[b] = friction ? p2 : T(0);
                w[b] = jv - c;
            }
            for (int c = 0; c < Uw; ++c) {
                T sa[3];
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    const int rc = row_of(c, a);
                    const T* row = gJ + (rc >= 0 ? rc : 0) * NVP;
                    T jc[NVP];
                    load_row16<T, NVP>(row, jc);
                    T acc = T(0);
#pragma unroll
                    for (int i = 0; i < NVP; ++i) acc += jc[i] * Yb[i];
                    sa[a] = rc >= 0 ? acc : T(0);  // A[(c, a)][(i, b)] = A[(i, b)][(c, a)]
                }
                if (c <= li && keeper) {
                    T* d = sS + (Ti + c) * 9 + 3 * b;
                    d[0] = sa[0]; d[1] = sa[1]; d[2] = sa[2];
                }
            }
        }
        __syncwarp();
        // own diagonal block: reciprocal effective masses and the coupling inside the unit
        const int lic = li < kFastUnits ? li : 0;  // lanes beyond the unit range read valid memory and contribute nothing
        const int Tic = lic * (lic + 1) / 2;
        const T* dg = sS + (Tic + lic) * 9;
#pragma unroll
        for (int a = 0; a < 3; ++a) pik[a] = row_of(li, a) >= 0 ? T(1) / dg[4 * a] : T(0);
        // coupling inside the unit, premultiplied by the reciprocal effective mass of the row it feeds
        const T P10 = dg[3] * pik[1], P20 = dg[6] * pik[2], P21 = dg[7] * pik[2];
        // ---- sweeps ----
        // Block read by lane i in round c: (max, min) of the pair; when c > i the stored block is the transpose of the
        // one needed, which the load offsets of the six off-diagonal entries undo. The loads sit at the top of the
        // round and are only consumed after the shuffles, so the owner's clamp chain hides their latency.
        // fp64 operations have a long dependent latency on this part, and the round IS one dependent chain
        // (residuals -> three clamps in sequence -> broadcast -> residuals), so the sequential solve of the unit
        //     n0 = clamp(l0 - w0 k0), n1 = clamp(l1 - (w1 + D10 d0) k1), n2 = clamp(l2 - (w2 + D20 d0 + D21 d1) k2)
        // is regrouped as n1 = clamp((l1 + P10 l0 - w1 k1) - P10 n0) etc. (P = D k): one FMA and one compare per row on
        // the chain, everything else hangs off it.
        T c1 = T(0), c2 = T(0);  // l1 + P10 l0, l2 + P20 l0 + P21 l1 (change only when this lane's unit is solved)
        auto round = [&](int c, int Tc) {
            const bool tr = c > lic;
            const T* b = sS + (tr ? Tc + lic : Tic + c) * 9;
            const int t2 = tr ? 2 : 0, t4 = tr ? 4 : 0;
            const T m0 = b[0], m1 = b[1 + t2], m2 = b[2 + t4], m3 = b[3 - t2], m4 = b[4], m5 = b[5 + t2], m6 = b[6 - t4],
                    m7 = b[7 - t2], m8 = b[8];
            // every lane solves its own unit from its own residuals; only the owner's result is used
            const T q0 = lam[0] - w[0] * pik[0], q1 = c1 - w[1] * pik[1], q2 = c2 - w[2] * pik[2];
            const T n0 = clamp_sel(q0, loA[0], hiA[0]);
            const T n1 = clamp_sel(fma(-P10, n0, q1), fma(loB[1], n0, loA[1]), fma(hiB[1], n0, hiA[1]));
            const T n2 = clamp_sel(fma(-P21, n1, fma(-P20, n0, q2)), fma(loB[2], n0, loA[2]), fma(hiB[2], n0, hiA[2]));
            const T b0 = __shfl_sync(0xffffffffu, n0 - lam[0], c, NVP);
            const T b1 = __shfl_sync(0xffffffffu, n1 - lam[1], c, NVP);
            const T b2 = __shfl_sync(0xffffffffu, n2 - lam[2], c, NVP);
            if (li == c) {
                lam[0] = n0; lam[1] = n1; lam[2] = n2;
                c1 = fma(P10, n0, n1);
                c2 = fma(P21, n1, fma(P20, n0, n2));
            }
            w[0] = ((w[0] + m0 * b0) + m1 * b1) + m2 * b2;  // the last impulse change to arrive is applied last
            w[1] = ((w[1] + m3 * b0) + m4 * b1) + m5 * b2;
            w[2] = ((w[2] + m6 * b0) + m7 * b1) + m8 * b2;
        };
        // The unit counts of the pick scene's phases (joint unit + 4 / 8 / 12 contacts) and of resting cubes (4 / 8 contacts)
        // get a fully unrolled sweep: the
        // owner index, the triangular block offset and the loop itself become immediates (a tenth of a round's instructions).
        auto sweeps = [&](auto uwc) {
            constexpr int UW = decltype(uwc)::value;
            for (int it = 0; it < iterations; ++it) {
                if constexpr (UW > 0) {
#pragma unroll
                    for (int c = 0; c < UW; ++c) round(c, c * (c + 1) / 2);
                } else {
                    int Tc = 0;
                    for (int c = 0; c < Uw; ++c) {
                        round(c, Tc);
                        Tc += c + 1;
                    }
                }
            }
        };
        if (Uw == 13) sweeps(std::integral_constant<int, 13>{});
        else if (Uw == 9) sweeps(std::integral_constant<int, 9>{});
        else if (Uw == 8) sweeps(std::integral_constant<int, 8>{});  // two stacked cubes
        else if (Uw == 5) sweeps(std::integral_constant<int, 5>{});
        else if (Uw == 4) sweeps(std::integral_constant<int, 4>{});  // one cube on the ground
        else sweeps(std::integral_constant<int, 0>{});
        // ---- v = v0 + M^-1 J^T lambda (lane = generalized velocity), impulses -> HBM ----
        T gsum = T(0);
        for (int c = 0; c < Uw; ++c) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const T l = __shfl_sync(0xffffffffu, lam[a], c, NVP);
                const int r = row_of(c, a);
                if (r >= 0) gsum += gJ[r * NVP + li] * l;
            }
        }
        __syncwarp();
        sG[li] = gsum;
        __syncwarp();
        if (fast) {
            const T dv = li < nv ? y_entry(nq, nfree, sAux, li, [&](int k) { return sG[k]; }) : T(0);
            g.v[e * NVP + li] = v0_own + dv;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const int r = row_of(li, a);
                if (r >= 0) g.lam[e * kMaxPgsRows + r] = lam[a];
            }
        }
        __syncwarp();
    }
    // ---- envs with too many units for the shared-memory form: the whole warp streams them, one after the other ----
    const unsigned slow_lanes = __ballot_sync(0xffffffffu, slow);
    if (slow_lanes) {
#pragma unroll
        for (int h = 0; h < EPW; ++h) {
            if (!((slow_lanes >> (h * NVP)) & 1u)) continue;  // warp-uniform
            const int64_t eh = e - half + h;
            T* scratch = reinterpret_cast<T*>(smem_raw) + (warp * EPW + h) * pgs_smem_per_env<T, NVP>();
            pgs_generic<T>(g, eh, lane, g.cnt[2 * eh], g.cnt[2 * eh + 1], iterations, scratch);
            __syncwarp();
        }
    }
}

// kFinishLanes threads per env: the stage is a handful of dependent loads per joint / body / contact, so its duration is
// the longest of those chains; lanes take them side by side (lane = joint, lane = free body, lane = contact).
constexpr int kFinishLanes = 16;
template <typename T, bool ENV = false>
__global__ void __launch_bounds__(128) k_world_finish(const WorldDev<T>* __restrict__ world, const WorldBuffers<T> b,
                                                      const PgsBuffers<T> g, T* __restrict__ state, T* __restrict__ accel,
                                                      int nq, uint32_t* __restrict__ robot_reset_mask,
                                                      const __grid_constant__ WorldRows<T> rows)
{
    __shared__ WorldDev<T> W;
    stage_world(world, W);
    __syncthreads();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t e = t / kFinishLanes;
    const int l = (int)(t % kFinishLanes);
    if (e >= b.n) return;
    const T dt = W.dt;
    const T* v = g.v + e * g.nvp;
    if (l == 0 && robot_reset_mask) robot_reset_mask[e] = 0;  // split prepare: the pending resets were left for its kernels
    // articulated model: constrained velocities, the acceleration they imply, position integration
    for (int j = l; j < nq; j += kFinishLanes) {
        const T unc = state[e * 2 * nq + nq + j], dq = v[j];
        accel[e * nq + j] += (dq - unc) / dt;
        state[e * 2 * nq + nq + j] = dq;
        state[e * 2 * nq + j] += dq * dt;
    }
    // free bodies: pose integration from the constrained velocities (lanes from the top, away from the joint lanes)
    for (int i = kFinishLanes - 1 - l; i < W.nfree; i += kFinishLanes) {
        T X[13], before[6];
        BodyWork<T> bw;
        for (int k = 0; k < 13; ++k) X[k] = b.base_state[i][e * 13 + k];
        for (int k = 0; k < 6; ++k) before[k] = X[7 + k];
        const auto prm = world_params<ENV>(rows, e);
        body_pose(W, i, X, bw, prm);
        const T* vb = v + nq + 6 * i;
        bw.vc = v3(vb[0], vb[1], vb[2]);
        bw.w = v3(vb[3], vb[4], vb[5]);
        body_end(W, i, X, bw, prm);
        for (int k = 0; k < 13; ++k) b.base_state[i][e * 13 + k] = X[k];
        write_base_accel(b, i, e, before, X, dt);
    }
    // contact forces on side a: (ln n + lt1 t1 + lt2 t2) / dt, tangents as in contact_frames
    const int nr = g.cnt[2 * e], njr = g.cnt[2 * e + 1], nc = (nr - njr) / 3;
    const T* lam = g.lam + e * kMaxPgsRows + njr;
    for (int k = l; k < nc; k += kFinishLanes) {
        T* o = b.contact_data + (e * kMaxContacts + k) * kContactRec;
        Contact<T> c;
        c.n = v3(o[3], o[4], o[5]);
        contact_frames(&c, 1);
        c.ln = lam[3 * k]; c.lt1 = lam[3 * k + 1]; c.lt2 = lam[3 * k + 2];
        const V3<T> f = contact_force(c, dt);
        o[7] = f.x; o[8] = f.y; o[9] = f.z;
    }
}

// Link world velocity and acceleration (Link::world{Linear,Angular}{Velocity,Acceleration}, Link.cpp:206-294;
// filled by Physics.cpp:1989-2079 in the reference): velocity and classical acceleration of the link frame origin,
// world orientation, from q, dq and the joint accelerations of the last step. out rows: [linear(3), angular(3)].
template <typename T, int NB>
__global__ void __launch_bounds__(128) k_link_motion(const ModelDev<T>* __restrict__ tables, const T* __restrict__ state,
                                                     const T* __restrict__ accel, int link, T* __restrict__ twist_out,
                                                     T* __restrict__ accel_out, int64_t n)
{
    __shared__ ModelDev<T> m;
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int nq = m.nq, body = m.link_body[link];
    int chain[NB], depth = 0;
    for (int i = body; i >= 0; i = m.parent[i]) chain[depth++] = i;
    M3<T> Rw = ld9(m.baseR);
    Sv<T> V = sv_zero<T>(), A = sv_zero<T>();  // spatial velocity / acceleration, body coordinates
    for (int d = depth - 1; d >= 0; --d) {
        const int i = chain[d];
        const T q = state[e * 2 * nq + i], dq = state[e * 2 * nq + nq + i], ddq = accel[e * nq + i];
        M3<T> R;
        V3<T> p;
        joint_pose(m, i, q, R, p);
        const V3<T> a = ld3(m.axis[i]), sd = dq * a, sdd = ddq * a;
        Sv<T> Vi = {mulT(R, V.a), mulT(R, V.l + cross(V.a, p))};
        Sv<T> Ai = {mulT(R, A.a), mulT(R, A.l + cross(A.a, p))};
        if (m.jtype[i] == kRevolute) {
            Ai.a = Ai.a + cross(Vi.a, sd) + sdd;
            Ai.l = Ai.l + cross(Vi.l, sd);
            Vi.a = Vi.a + sd;
        } else {
            Ai.l = Ai.l + cross(Vi.a, sd) + sdd;
            Vi.l = Vi.l + sd;
        }
        V = Vi;
        A = Ai;
        Rw = mul(Rw, R);
    }
    const V3<T> r = ld3(m.link_p[link]);
    const V3<T> v_pt = V.l + cross(V.a, r);
    const V3<T> a_pt = A.l + cross(A.a, r) + cross(V.a, v_pt);  // classical acceleration of the link origin
    const V3<T> vw = mul(Rw, v_pt), ww = mul(Rw, V.a), aw = mul(Rw, a_pt), alw = mul(Rw, A.a);
    if (twist_out) {
        T* o = twist_out + e * 6;
        o[0] = vw.x; o[1] = vw.y; o[2] = vw.z; o[3] = ww.x; o[4] = ww.y; o[5] = ww.z;
    }
    if (accel_out) {
        T* o = accel_out + e * 6;
        o[0] = aw.x; o[1] = aw.y; o[2] = aw.z; o[3] = alw.x; o[4] = alw.y; o[5] = alw.z;
    }
}

// KinDynComputations centre of mass / momentum for every env (b2_rbd.hpp centroidal).
template <typename T, int NB>
__global__ void __launch_bounds__(128) k_centroidal(const ModelDev<T>* __restrict__ tables, const T* __restrict__ state,
                                                    T* __restrict__ com_out, T* __restrict__ vel_out,
                                                    T* __restrict__ mom_out, T* __restrict__ jac_out, int64_t n)
{
    __shared__ ModelDev<T> m;
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int nq = m.nq;
    T q[NB], dq[NB];
    for (int j = 0; j < nq; ++j) {
        q[j] = state[e * 2 * nq + j];
        dq[j] = state[e * 2 * nq + nq + j];
    }
    centroidal<T, NB>(m, q, dq, com_out ? com_out + e * 3 : nullptr, vel_out ? vel_out + e * 3 : nullptr,
                      mom_out ? mom_out + e * 12 : nullptr, jac_out ? jac_out + e * 3 * nq : nullptr);
}

// KinDynComputations momentum Jacobian / locked inertia for every env (b2_rbd.hpp momentum_matrices).
template <typename T, int NB>
__global__ void __launch_bounds__(128) k_momentum(const ModelDev<T>* __restrict__ tables, const T* __restrict__ state,
                                                  T* __restrict__ jmom_out, T* __restrict__ locked_out, int64_t n)
{
    __shared__ ModelDev<T> m;
    stage_model(tables, m);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int nq = m.nq;
    T q[NB];
    for (int j = 0; j < nq; ++j) q[j] = state[e * 2 * nq + j];
    momentum_matrices<T, NB>(m, q, jmom_out ? jmom_out + e * 6 * nq : nullptr, locked_out ? locked_out + e * 10 : nullptr);
}

// ---- column utilities for the per-object view ------------------------------------------------------
template <typename T>
__global__ void k_col_fill(T* dst, int64_t n, int stride, int col, T value)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n) dst[e * stride + col] = value;
}
template <typename T>
__global__ void k_col_copy(T* dst, int dstride, int dcol, const T* src, int sstride, int scol, int64_t n)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n) dst[e * dstride + dcol] = src[e * sstride + scol];
}
static __global__ void k_or_mask(uint32_t* mask, int64_t n, int64_t env, uint32_t bits)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t e = env >= 0 ? env : t;
    if (t < (env >= 0 ? 1 : n)) mask[e] |= bits;
}

// Joint::resetPosition / resetVelocity for one env (or all envs when env < 0): stores the value, raises
// the dirty bit and resets the PID state (Joint.cpp:132-180).
template <typename T>
__global__ void k_set_reset(T* reset_state, uint32_t* mask, T* pid_state, int64_t n, int nq, int64_t env, int joint,
                            int is_velocity, T value)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t e = env >= 0 ? env : t;
    if (t >= (env >= 0 ? 1 : n)) return;
    reset_state[e * 2 * nq + (is_velocity ? nq : 0) + joint] = value;
    mask[e] |= 1u << ((is_velocity ? 16 : 0) + joint);
    pid_state[e * 3 * nq + 3 * joint + 0] = T(0);
    pid_state[e * 3 * nq + 3 * joint + 1] = T(0);
    pid_state[e * 3 * nq + 3 * joint + 2] = T(0);
}

}  // namespace b2
