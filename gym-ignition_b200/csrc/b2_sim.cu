// b2sim: simulator object and C ABI (include/b2sim.h). Host side of the engine: owns the per-env
// device buffers, keeps the per-model ScenarI/O bookkeeping (control modes, PID gains, controller
// period, which one-shot components exist), and launches the kernels of b2_kernels.cuh.
//
// There is deliberately no CPU execution path in this file: every state-touching entry point needs a
// CUDA device and reports B2_ERR_CUDA otherwise.
#include <cuda_runtime.h>

#include <cfloat>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <array>
#include <fstream>
#include <memory>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/b2sim.h"
#include "b2_kernels.cuh"
#include "b2_lanes.hpp"
#include "b2_model.hpp"

namespace {

thread_local std::string g_error;

int fail(int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
    return code;
}

#define B2_CUDA(call)                                                                                   \
    do {                                                                                                \
        cudaError_t err__ = (call);                                                                     \
        if (err__ != cudaSuccess)                                                                       \
            return fail(B2_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(err__));               \
    } while (0)

// Every entry point that launches, copies or allocates runs on the simulator's device and leaves the caller's current
// device as it found it (a process may hold simulators on several GPUs, and torch has its own current device).
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int device)
    {
        if (cudaGetDevice(&prev) != cudaSuccess || prev == device) prev = -1;
        if (prev >= 0) cudaSetDevice(device);
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

int64_t to_ns(double seconds) { return (int64_t)llround(seconds * 1e9); }  // helpers.cpp:98-108

constexpr int64_t kWarpSolverMaxEnvs = 8192;  // free-body worlds up to this size use the warp-cooperative contact pipeline

struct ModelState {
    std::unique_ptr<b2model> model;
    std::string name;
    b2::Pose base;
    bool removed = false;
    int kind = B2_KIND_STATIC;
    void* d_tables = nullptr;
    void* d_lane_table = nullptr;  // inside the d_tables allocation
    double* d_ep_totals = nullptr; // [B2_STAT_STRIPES][4] episode statistics (b2sim_episode_stats_enable)
    void* buf[B2_BUF_COUNT] = {};
    void* force_read = nullptr;
    // shared joint configuration
    int mode[B2_MAX_DOFS];
    b2_pid pid[B2_MAX_DOFS];
    bool has_force_cmd[B2_MAX_DOFS], has_vel_cmd[B2_MAX_DOFS], has_pos_target[B2_MAX_DOFS],
        has_vel_target[B2_MAX_DOFS];
    double effort[B2_MAX_DOFS];
    int64_t period_ns = INT64_MAX, prev_update_ns = 0;
    bool controller_loaded = false;
    // ComputedTorqueFixedBase (ControllerRunner)
    bool ct_loaded = false;
    bool has_acc_target[B2_MAX_DOFS] = {};
    double ct_kp[B2_MAX_DOFS] = {}, ct_kd[B2_MAX_DOFS] = {}, ct_gravity[3] = {0, 0, -9.80665};
    int64_t ct_prev_update_ns = 0;
    // external link wrenches (Link::applyWorldWrench)
    struct LinkWrench { int link; int64_t env; double w[6]; int64_t expiry_ns; };
    std::vector<LinkWrench> wrenches;
    // task
    int task = B2_TASK_NONE;
    uint64_t seed = 0, env_offset = 0, task_steps = 0;
    int max_episode_steps = 5000;
    double rand_mass_delta = 0, rand_gravity_sigma = 0;
    bool env_params = false;  // B2_BUF_BODY_INERTIA / JOINT_DYNAMICS / GRAVITY allocated (b2sim_enable_env_params)
    void* body_rows = nullptr;  // [N, b2::kFreeBodyCols] per-env inertial data of a free body (b2sim_enable_free_body_params)
    void* mu_rows = nullptr;    // [N, nshapes] per-env friction coefficient of every collision shape (b2sim_enable_shape_friction)
    unsigned long long* d_step = nullptr;  // device-side step counter of the fused task (next Philox step index)
    unsigned int* d_ticket = nullptr;
    bool graph_recorded = false;
    double task_goal[3] = {0.5, 0.0, 0.5};
    double task_q0[B2_MAX_DOFS] = {};
    int task_ee_link = 0;
    void* pinned_actions = nullptr;
    void* pinned_obs = nullptr;
    void* pinned_reward = nullptr;
    void* pinned_done = nullptr;
};

}  // namespace

struct b2sim {
    int device = 0;
    int64_t n = 0;
    int64_t dt_ns = 0, time_ns = 0;
    double step_size = 0;
    int steps_per_run = 1;
    int dtype = B2_F64;
    double gravity[3] = {0, 0, -9.8};  // SDF default world gravity
    cudaStream_t stream = nullptr;
    cudaStream_t copy_in = nullptr, copy_out = nullptr;  // host-buffer path: H2D / D2H overlap with the kernels
    cudaStream_t fork[2] = {nullptr, nullptr};           // coupled worlds: the parts of the prepare stage run concurrently
    cudaEvent_t fork_ev[3] = {nullptr, nullptr, nullptr};
    std::vector<cudaEvent_t> events;
    int64_t win_begin = 0, win_count = -1;               // env window of the fused launches (-1 = all envs)
    // free bodies + contacts (world level)
    void* d_world = nullptr;
    bool world_dirty = true;
    std::vector<int> free_models;                        // model ids of the free bodies, in world order
    std::vector<int> static_shape_model, static_shape_link;
    int robot_model = -1;                                // articulated model whose link shapes take part in contacts
    std::vector<int> robot_shape_link;                   // link of each robot shape (reporting)
    // loader shape (column of the model's friction rows) of every shape slot of the world description
    std::vector<std::array<int, b2::kMaxBodyShapes>> free_shape_col;
    std::vector<int> static_shape_col, robot_shape_col;
    int32_t* contact_count = nullptr;
    int32_t* contact_ids = nullptr;
    void* contact_data = nullptr;
    // dense rows of the warp-cooperative contact solver (k_pgs_solve); nvp = 0: single-thread kernels are used
    void *pgs_v = nullptr, *pgs_J = nullptr, *pgs_Y = nullptr, *pgs_par = nullptr, *pgs_lam = nullptr, *pgs_aux = nullptr;
    int* pgs_cnt = nullptr;
    int pgs_nvp = 0, pgs_nq = 0, pgs_nfree = 0;
    double contact_erp = 0.01, contact_max_erv = 1e-3;
    int contact_iterations = 50;
    uint64_t launches = 0;
    bool free_wrench_dirty = false;  // the ext / ext_env block of the device world is stale
    std::vector<std::unique_ptr<ModelState>> models;

    size_t esize() const { return dtype == B2_F64 ? 8 : 4; }
};

namespace {

ModelState* get_model(const b2sim* s, int id)
{
    if (!s || id < 0 || id >= (int)s->models.size() || s->models[id]->removed) return nullptr;
    return s->models[id].get();
}

int grid_for(int64_t n, int block) { return (int)((n + block - 1) / block); }

template <typename T>
int upload_tables(b2sim* s, ModelState* ms)
{
    b2::ModelDev<T> md;
    ms->model->to_device_tables<T>(ms->base, s->gravity, md);
    for (int j = 0; j < md.nq; ++j) md.effort[j] = (T)ms->effort[j];
    // one allocation: the model tables, then the same constants packed per body for the lane-parallel kernels
    if (!ms->d_tables) B2_CUDA(cudaMalloc(&ms->d_tables, sizeof(b2::ModelDev<double>) + sizeof(b2::LaneTable<double>)));
    ms->d_lane_table = (char*)ms->d_tables + sizeof(b2::ModelDev<double>);
    b2::LaneTable<T> lt;
    b2::fill_lane_table(md, lt);
    B2_CUDA(cudaMemcpyAsync(ms->d_tables, &md, sizeof md, cudaMemcpyHostToDevice, s->stream));
    B2_CUDA(cudaMemcpyAsync(ms->d_lane_table, &lt, sizeof lt, cudaMemcpyHostToDevice, s->stream));
    B2_CUDA(cudaStreamSynchronize(s->stream));
    return B2_OK;
}

int refresh_tables(b2sim* s, ModelState* ms)
{
    ms->kind = ms->model->fit(ms->base, s->gravity, s->step_size);
    if (ms->kind == B2_KIND_STATIC) return B2_OK;
    return s->dtype == B2_F64 ? upload_tables<double>(s, ms) : upload_tables<float>(s, ms);
}

int alloc_buffer(b2sim* s, ModelState* ms, int which, size_t bytes)
{
    if (ms->buf[which]) return B2_OK;
    if (bytes == 0) return B2_OK;
    B2_CUDA(cudaMalloc(&ms->buf[which], bytes));
    B2_CUDA(cudaMemsetAsync(ms->buf[which], 0, bytes, s->stream));
    return B2_OK;
}

void buffer_shape(const b2sim* s, const ModelState* ms, int which, int64_t* cols, int* dtype, int* itemsize)
{
    const int nq = ms->model->t.nq;
    *dtype = s->dtype;
    *itemsize = (int)s->esize();
    switch (which) {
    case B2_BUF_STATE: *cols = 2 * nq; break;
    case B2_BUF_ACCELERATION: *cols = nq; break;
    case B2_BUF_FORCE_CMD: *cols = nq; break;
    case B2_BUF_POS_TARGET: *cols = nq; break;
    case B2_BUF_VEL_TARGET: *cols = nq; break;
    case B2_BUF_ACC_TARGET: *cols = nq; break;
    case B2_BUF_RAND_PARAMS: *cols = (ms->rand_mass_delta != 0 || ms->rand_gravity_sigma != 0) ? nq + 1 : 0; break;
    case B2_BUF_PID_STATE: *cols = 3 * nq; break;
    case B2_BUF_RESET_STATE: *cols = 2 * nq; break;
    case B2_BUF_RESET_MASK: *cols = (nq > 0 || ms->kind == B2_KIND_FREE) ? 1 : 0; *dtype = -32; *itemsize = 4; break;
    case B2_BUF_OBS: *cols = ms->task == B2_TASK_PANDA_REACH ? b2::panda_obs_size(nq) : b2sim_task_nobs(ms->task); break;
    case B2_BUF_REWARD: *cols = 1; break;
    case B2_BUF_DONE: *cols = 1; *dtype = -8; *itemsize = 1; break;
    case B2_BUF_ELAPSED: *cols = 1; *dtype = -16; *itemsize = 2; break;
    case B2_BUF_ACTION: *cols = ms->task == B2_TASK_PANDA_REACH ? nq : b2sim_task_nact(ms->task); break;
    case B2_BUF_LINK_POSE: *cols = 7 * ms->model->t.nlinks; break;
    case B2_BUF_BASE_STATE: *cols = ms->kind == B2_KIND_FREE ? 13 : 0; break;
    case B2_BUF_BASE_RESET: *cols = ms->kind == B2_KIND_FREE ? 13 : 0; break;
    case B2_BUF_EP_RETURN: *cols = ms->d_ep_totals ? 1 : 0; break;
    case B2_BUF_BASE_ACCEL: *cols = ms->kind == B2_KIND_FREE ? 6 : 0; break;
    case B2_BUF_BODY_INERTIA: *cols = ms->env_params ? b2::kEnvInertiaCols * nq : 0; break;
    case B2_BUF_JOINT_DYNAMICS: *cols = ms->env_params ? b2::kEnvJointCols * nq : 0; break;
    case B2_BUF_GRAVITY: *cols = ms->env_params ? 3 : 0; break;
    default: *cols = 0; break;
    }
}

int ensure_buffer(b2sim* s, ModelState* ms, int which)
{
    int64_t cols;
    int dtype, itemsize;
    buffer_shape(s, ms, which, &cols, &dtype, &itemsize);
    return alloc_buffer(s, ms, which, (size_t)s->n * cols * itemsize);
}

template <typename T>
b2::RunBuffers<T> run_buffers(b2sim* s, ModelState* ms)
{
    b2::RunBuffers<T> b;
    b.state = (T*)ms->buf[B2_BUF_STATE];
    b.accel = (T*)ms->buf[B2_BUF_ACCELERATION];
    b.force_cmd = (T*)ms->buf[B2_BUF_FORCE_CMD];
    b.force_read = (T*)ms->force_read;
    b.pos_target = (T*)ms->buf[B2_BUF_POS_TARGET];
    b.vel_target = (T*)ms->buf[B2_BUF_VEL_TARGET];
    b.pid_state = (T*)ms->buf[B2_BUF_PID_STATE];
    b.reset_state = (T*)ms->buf[B2_BUF_RESET_STATE];
    b.acc_target = (T*)ms->buf[B2_BUF_ACC_TARGET];
    b.reset_mask = (uint32_t*)ms->buf[B2_BUF_RESET_MASK];
    b.n = s->n;
    return b;
}

int tree_topology(const ModelState* ms, b2::TreeTopo* topo)
{
    const b2_model_tables& t = ms->model->t;
    topo->nbranch = b2::branch_slots(t.nq, t.parent, topo->slot);
    if (topo->nbranch < 0) return fail(B2_ERR_UNSUPPORTED, "the kinematic tree has more than %d branching bodies", b2::kMaxBranch);
    topo->has_friction = 0;
    topo->impulse_ok = 1;
    for (int j = 0; j < t.nq; ++j) {
        if (t.friction[j] != 0.0) topo->has_friction = 1;
        if (t.damping[j] != 0.0 || t.stiffness[j] != 0.0) topo->impulse_ok = 0;
    }
    return B2_OK;
}

// Whether a tree's dynamics run on lanes (k_run_tree_lanes, an env on G lanes of a warp) rather than one thread per env.
// Small batches of trees with several joints (BASELINE configs 4 / 5: 16,384 / 4,096 Pandas) leave one thread per env
// with less than a warp per scheduler and the run lasts as long as ONE env's dependent chain, so up to 16,384 envs the
// step is spread over lanes (Pandas under position PIDs, measured on the B200: 15 us against 38 us per run at 4,096 envs,
// 42 against 43 us at 16,384; 21 against 60 us at 4,096 envs with both fingers on their limits). By default lanes are
// used for trees of at least `min_nq` joints. B2_RUN_KERNEL=thread / lanes forces one side (tests run both).
bool run_on_lanes(const b2sim* s, const ModelState* ms, int min_nq)
{
    static const char* forced = getenv("B2_RUN_KERNEL");
    if (!ms->d_lane_table) return false;
    if (forced) return !strcmp(forced, "lanes");
    return s->n <= 16384 && ms->model->t.nq >= min_nq;
}

// A joint's PID gains in the kernels' order: p, i, d, i_max, i_min, cmd_max, cmd_min, cmd_offset.
template <typename T>
void pack_pid(const b2_pid& p, T* gains)
{
    const double g[8] = {p.p, p.i, p.d, p.i_max, p.i_min, p.cmd_max, p.cmd_min, p.cmd_offset};
    for (int k = 0; k < 8; ++k) gains[k] = (T)g[k];
}

template <typename T>
b2::RunCfg<T> build_run_cfg(b2sim* s, ModelState* ms, int paused, int iterations, uint32_t compute_bits, uint32_t ct_bits,
                            const int* wrench_iters)
{
    const int nq = ms->model->t.nq;
    b2::RunCfg<T> cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.nq = nq;
    cfg.iterations = iterations;
    cfg.paused = paused;
    cfg.controller_loaded = ms->controller_loaded;
    cfg.compute_new_bits = compute_bits;
    cfg.dt = (T)((double)s->dt_ns / 1e9);
    for (int j = 0; j < nq; ++j) {
        cfg.mode[j] = (uint8_t)ms->mode[j];
        cfg.has_force_cmd[j] = ms->has_force_cmd[j];
        cfg.has_vel_cmd[j] = ms->has_vel_cmd[j];
        pack_pid(ms->pid[j], cfg.pid[j]);
        cfg.ct_kp[j] = (T)ms->ct_kp[j];
        cfg.ct_kd[j] = (T)ms->ct_kd[j];
    }
    // the controller steps only once every reference exists (ControllerRunner.cpp:253-274)
    cfg.ct_active = ms->ct_loaded;
    for (int j = 0; j < nq; ++j)
        if (!(ms->has_pos_target[j] && ms->has_vel_target[j] && ms->has_acc_target[j])) cfg.ct_active = 0;
    cfg.ct_compute_bits = ct_bits;
    for (int k = 0; k < 3; ++k) cfg.ct_gravity[k] = (T)ms->ct_gravity[k];
    cfg.nwrench = 0;
    for (size_t k = 0; k < ms->wrenches.size() && cfg.nwrench < 4; ++k) {
        if (wrench_iters[k] <= 0) continue;
        const int o = cfg.nwrench++;
        cfg.wrench_link[o] = ms->wrenches[k].link;
        cfg.wrench_env[o] = ms->wrenches[k].env;
        cfg.wrench_iters[o] = wrench_iters[k];
        for (int a = 0; a < 6; ++a) cfg.wrench[o][a] = (T)ms->wrenches[k].w[a];
    }
    return cfg;
}

// The model's per-env parameter rows from env w0 on (all null while b2sim_enable_env_params is off). With rows, the impulse
// path of the constraint stage needs undamped joints: the tables' stiffness decides in `topo`, every env's damping row in
// the kernel.
template <typename T>
b2::EnvRows<T> env_rows(const ModelState* ms, int64_t w0, b2::TreeTopo* topo)
{
    b2::EnvRows<T> env;
    if (!ms->env_params) return env;
    const int nq = ms->model->t.nq;
    env.inertia = (const T*)ms->buf[B2_BUF_BODY_INERTIA] + w0 * b2::kEnvInertiaCols * nq;
    env.dyn = (const T*)ms->buf[B2_BUF_JOINT_DYNAMICS] + w0 * b2::kEnvJointCols * nq;
    env.grav = (const T*)ms->buf[B2_BUF_GRAVITY] + w0 * 3;
    topo->impulse_ok = 1;
    for (int j = 0; j < nq; ++j)
        if (ms->model->t.stiffness[j] != 0.0) topo->impulse_ok = 0;
    return env;
}

// One thread per env: k_run_tree (scratch in shared memory, 64-thread blocks) or k_run_tree_local; ENV = the model's
// per-env parameter rows are allocated.
template <typename T, bool ENV>
cudaError_t launch_run_thread(b2sim* s, const b2::ModelDev<T>* tb, const b2::RunCfg<T>& cfg, const b2::RunBuffers<T>& b,
                              const b2::TreeTopo& topo, const b2::EnvRows<T>& env, size_t smem, bool local)
{
    cudaError_t rc = cudaFuncSetAttribute(b2::k_run_tree<T, ENV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc != cudaSuccess) return rc;
    if (local) b2::k_run_tree_local<T, ENV><<<grid_for(s->n, 128), 128, 0, s->stream>>>(tb, cfg, b, topo, env);
    else b2::k_run_tree<T, ENV><<<grid_for(s->n, 64), 64, smem, s->stream>>>(tb, cfg, b, topo, env);
    return cudaGetLastError();
}

template <typename T>
int launch_run(b2sim* s, ModelState* ms, int paused, int iterations, uint32_t compute_bits, uint32_t ct_bits,
               const int* wrench_iters)
{
    const int nq = ms->model->t.nq;
    const b2::RunCfg<T> cfg = build_run_cfg<T>(s, ms, paused, iterations, compute_bits, ct_bits, wrench_iters);
    b2::RunBuffers<T> b = run_buffers<T>(s, ms);
    b2::TreeTopo topo;
    int rc = tree_topology(ms, &topo);
    if (rc != B2_OK) return rc;
    const b2::ModelDev<T>* tb = (const b2::ModelDev<T>*)ms->d_tables;
    const b2::EnvRows<T> env = env_rows<T>(ms, 0, &topo);
    if (nq >= 1 && nq <= b2::kMaxDofs && run_on_lanes(s, ms, 4)) {
        B2_CUDA(b2::launch_run_tree_lanes<T>(tb, (const b2::LaneTable<T>*)ms->d_lane_table, cfg, b, ms->model->t.parent,
                                             ms->model->t.jtype, s->stream, nullptr, 0, env));
        ++s->launches;
        return B2_OK;
    }
    const size_t smem = (size_t)b2::scratch_slots(nq, topo.nbranch) * 64 * sizeof(T);  // 64-thread blocks
    // Scratch placement: shared memory keeps small batches fastest (two 64-thread blocks per SM); from ~64 k envs on,
    // L1/L2-backed local memory wins because more threads stay resident (1.4x at 1 M envs). B2_TREE_SCRATCH overrides.
    static const char* variant = getenv("B2_TREE_SCRATCH");
    const bool local = variant ? !strcmp(variant, "local") : s->n >= 65536;
    B2_CUDA((ms->env_params ? launch_run_thread<T, true>(s, tb, cfg, b, topo, env, smem, local)
                            : launch_run_thread<T, false>(s, tb, cfg, b, topo, env, smem, local)));
    ++s->launches;
    return B2_OK;
}

template <int TASK, typename T>
int launch_task(b2sim* s, ModelState* ms, const void* actions, int traj_steps = 0, void* traj_obs = nullptr,
                void* traj_reward = nullptr, uint8_t* traj_done = nullptr)
{
    constexpr int nq2 = 2 * b2::TaskTraits<TASK>::nq, nobs = b2::TaskTraits<TASK>::nobs;
    const int64_t w0 = s->win_begin, wn = s->win_count < 0 ? s->n : s->win_count;
    b2::TaskArgs<T> a;
    a.state = (T*)ms->buf[B2_BUF_STATE] + w0 * nq2;
    a.actions = (const T*)actions + w0;
    a.obs = (T*)ms->buf[B2_BUF_OBS] + w0 * nobs;
    a.reward = (T*)ms->buf[B2_BUF_REWARD] + w0;
    a.done = (uint8_t*)ms->buf[B2_BUF_DONE] + w0;
    a.elapsed = (uint16_t*)ms->buf[B2_BUF_ELAPSED] + w0;
    const b2::ChainCoef<double>& c = ms->model->coef;
    a.coef.m11 = (T)c.m11; a.coef.m22 = (T)c.m22; a.coef.A = (T)c.A; a.coef.B = (T)c.B;
    a.coef.G1 = (T)c.G1; a.coef.E = (T)c.E; a.coef.F = (T)c.F;
    a.coef.d1 = (T)c.d1; a.coef.d2 = (T)c.d2; a.coef.dt = (T)c.dt; a.coef.revolute = c.revolute;
    a.n = wn;
    a.seed = ms->seed;
    a.env_offset = ms->env_offset + (uint64_t)w0;
    // Philox step index (0 is the initial reset). Eager launches take it from the host and mirror the next index into
    // a device counter; launches recorded into a CUDA graph read and advance that counter themselves. Once a graph
    // has been recorded the host copy may be stale (replays are invisible to the host), so it is refreshed first.
    cudaStreamCaptureStatus capture = cudaStreamCaptureStatusNone;
    if (s->stream) cudaStreamIsCapturing(s->stream, &capture);
    const bool capturing = capture == cudaStreamCaptureStatusActive;
    if (capturing) {
        ms->graph_recorded = true;
    } else if (ms->graph_recorded && w0 == 0) {
        unsigned long long next = 0;
        B2_CUDA(cudaMemcpyAsync(&next, ms->d_step, sizeof next, cudaMemcpyDeviceToHost, s->stream));
        B2_CUDA(cudaStreamSynchronize(s->stream));
        if (next > 0) ms->task_steps = next - 1;
    }
    a.step = ms->task_steps + 1;
    a.step_counter = ms->d_step;
    a.block_ticket = ms->d_ticket;
    a.advance_counter = (w0 + wn == s->n) ? 1 : 0;
    a.max_episode_steps = ms->max_episode_steps;
    a.iterations = s->steps_per_run;
    a.rand = ms->buf[B2_BUF_RAND_PARAMS] ? (T*)ms->buf[B2_BUF_RAND_PARAMS] + w0 * (nq2 / 2 + 1) : nullptr;
    for (int k = 0; k < 2; ++k) {
        for (int i = 0; i < 7; ++i) a.basis.dmass[k][i] = (T)ms->model->basis.dmass[k][i];
        a.basis.mass[k] = (T)ms->model->basis.mass[k];
        a.body_mass[k] = ms->model->basis.mass[k];
    }
    a.mass_delta = ms->rand_mass_delta;
    a.gravity_sigma = ms->rand_gravity_sigma;
    a.gravity_z0 = s->gravity[2];
    a.ep_return = ms->d_ep_totals ? (T*)ms->buf[B2_BUF_EP_RETURN] + w0 : nullptr;
    a.ep_totals = ms->d_ep_totals;
    if (traj_steps > 0) {
        // one launch for the whole action sequence; 64-thread blocks spread small batches over all SMs
        if (capturing) return fail(B2_ERR_UNSUPPORTED, "b2sim_task_trajectory cannot be captured into a CUDA graph");
        if (w0 != 0 || wn != s->n) return fail(B2_ERR_UNSUPPORTED, "b2sim_task_trajectory steps all envs");
        const int block = 64, grid = grid_for(wn, block);
        b2::k_task_trajectory<TASK, T><<<grid, block, 0, s->stream>>>(a, traj_steps, (T*)traj_obs, (T*)traj_reward, traj_done);
        ms->task_steps += (uint64_t)(traj_steps - 1);  // the caller adds the last one, as for a single step
        ++s->launches;
        B2_CUDA(cudaGetLastError());
        return B2_OK;
    }
    // 128-thread blocks (measured on the B200 with eager launches, 64 / 128 / 256 threads: 131,072 envs 4.9 / 4.9 / 5.1 us,
    // 1,048,576 envs 18.9 / 18.9 / 20.0 us, 4,194,304 envs - / 74.1 / 74.7 us per step).
    // One pass over all envs: a grid-stride variant that keeps the next env's loads in flight during the arithmetic was
    // measured on the B200 at 4,194,304 envs at 82 - 103 us for 2 - 8 blocks per SM against 78 us for this launch (131 k
    // warps queued keep HBM busier than 1,184 resident warps that prefetch).
    const int block = 128, grid = grid_for(wn, block);
    if (capturing) {
        if ((grid + b2::kTicketGroup - 1) / b2::kTicketGroup > b2::kTicketWords - 1)
            return fail(B2_ERR_UNSUPPORTED, "too many envs for a graph-captured step (%lld)", (long long)wn);
        b2::k_task_chain<TASK, T, true><<<grid, block, 0, s->stream>>>(a);
    } else {
        // eager steps follow each other on the stream: programmatic dependent launch hides the launch-to-launch gap
        // (k_task_chain waits with griddepcontrol.wait before it touches memory)
        B2_CUDA(b2::launch_pdl(b2::k_task_chain<TASK, T, false>, grid, block, 0, s->stream, true, a));
    }
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

template <typename T>
int launch_panda(b2sim* s, ModelState* ms, const void* actions, int observe_only)
{
    const int nq = ms->model->t.nq;
    b2::PandaArgs<T> a;
    memset(&a, 0, sizeof a);
    const int64_t w0 = s->win_begin, wn = s->win_count < 0 ? s->n : s->win_count;
    a.state = (T*)ms->buf[B2_BUF_STATE] + w0 * 2 * nq;
    a.targets = (const T*)(actions ? actions : ms->buf[B2_BUF_POS_TARGET]) + w0 * nq;
    a.pid_state = (T*)ms->buf[B2_BUF_PID_STATE] + w0 * 3 * nq;
    a.obs = (T*)ms->buf[B2_BUF_OBS] + w0 * b2::panda_obs_size(nq);
    a.reward = (T*)ms->buf[B2_BUF_REWARD] + w0;
    a.done = (uint8_t*)ms->buf[B2_BUF_DONE] + w0;
    a.elapsed = (uint16_t*)ms->buf[B2_BUF_ELAPSED] + w0;
    a.n = wn;
    a.nq = nq;
    a.iterations = observe_only ? 0 : s->steps_per_run;
    a.max_episode_steps = ms->max_episode_steps;
    a.ee_link = ms->task_ee_link;
    a.ee_body = ms->model->t.link_body[ms->task_ee_link];
    a.observe_only = observe_only;
    a.dt = (T)((double)s->dt_ns / 1e9);
    a.ep_return = ms->d_ep_totals ? (T*)ms->buf[B2_BUF_EP_RETURN] + w0 : nullptr;
    a.ep_totals = ms->d_ep_totals;
    for (int k = 0; k < 3; ++k) a.goal[k] = (T)ms->task_goal[k];
    for (int j = 0; j < nq; ++j) {
        a.q0[j] = (T)ms->task_q0[j];
        pack_pid(ms->pid[j], a.pid[j]);
    }
    b2::TreeTopo topo;
    int rc = tree_topology(ms, &topo);
    if (rc != B2_OK) return rc;
    if (b2::panda_obs_size(nq) > b2::kPandaObs) return fail(B2_ERR_UNSUPPORTED, "the reach task supports up to 9 joints");
    const b2::EnvRows<T> env = env_rows<T>(ms, w0, &topo);  // offset by the window like every per-env pointer above
    // Up to 32,768 envs an env's step is spread over G lanes of a warp (b2_lanes.cuh): measured on the B200 at 4,096 /
    // 16,384 / 65,536 / 262,144 envs, lanes 18 / 46 / 149 / 550 us against 46 / 51 / 137 / 480 us for one thread per env
    // (the lane kernel executes ~1.4x the thread-instruction slots per env, so it loses once the batch fills the
    // schedulers). B2_PANDA_KERNEL=thread / lanes forces one of them (tests run both).
    static const char* variant = getenv("B2_PANDA_KERNEL");
    const bool lanes = variant ? strcmp(variant, "thread") != 0 : wn <= 32768;
    if (lanes) {
        B2_CUDA(b2::launch_task_panda_lanes<T>((const b2::ModelDev<T>*)ms->d_tables, (const b2::LaneTable<T>*)ms->d_lane_table, a,
                                               ms->model->t.parent, ms->model->t.jtype, s->stream, env));
        ++s->launches;
        return B2_OK;
    }
    // small batches: 64-thread blocks spread the envs over more SMs; large batches: 128-thread blocks
    const int block = wn >= 148 * 256 ? 128 : 64, grid = grid_for(wn, block);
    // 246 registers, 2 blocks of 128 threads per SM. Forcing 3 / 4 / 6 blocks per SM with __launch_bounds__ (168 / 128 / 80
    // registers) was measured on the B200 and does not help at any batch size (16 k envs: 53 / 58 / 68 / 93 us,
    // 1 M envs: 1.82 / 1.82 / 1.94 / 2.51 ms): the kernel is bound by the dependent fp64 chain at small batches and by
    // the L1 / L2 traffic of the per-thread scratch at large ones, not by occupancy.
    if (ms->env_params) b2::k_task_panda<T, true><<<grid, block, 0, s->stream>>>((const b2::ModelDev<T>*)ms->d_tables, a, topo, env);
    else b2::k_task_panda<T><<<grid, block, 0, s->stream>>>((const b2::ModelDev<T>*)ms->d_tables, a, topo, env);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

template <typename T>
int dispatch_task(b2sim* s, ModelState* ms, const void* actions, int traj_steps = 0, void* to = nullptr, void* tr = nullptr,
                  uint8_t* td = nullptr)
{
    if (ms->task == B2_TASK_PANDA_REACH) {
        if (traj_steps > 0) return fail(B2_ERR_UNSUPPORTED, "the reach task has no single-launch trajectory kernel");
        return launch_panda<T>(s, ms, actions, 0);
    }
    switch (ms->task) {
    case B2_TASK_PENDULUM_SWINGUP: return launch_task<B2_TASK_PENDULUM_SWINGUP, T>(s, ms, actions, traj_steps, to, tr, td);
    case B2_TASK_CARTPOLE_DISCRETE_BALANCING:
        return launch_task<B2_TASK_CARTPOLE_DISCRETE_BALANCING, T>(s, ms, actions, traj_steps, to, tr, td);
    case B2_TASK_CARTPOLE_CONTINUOUS_BALANCING:
        return launch_task<B2_TASK_CARTPOLE_CONTINUOUS_BALANCING, T>(s, ms, actions, traj_steps, to, tr, td);
    case B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP:
        return launch_task<B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP, T>(s, ms, actions, traj_steps, to, tr, td);
    default: return fail(B2_ERR_UNSUPPORTED, "task %d has no fused kernel", ms->task);
    }
}

template <int TASK, typename T>
int launch_reset_all(b2sim* s, ModelState* ms)
{
    const int block = 256, grid = grid_for(s->n, block);
    b2::k_task_reset_all<TASK, T><<<grid, block, 0, s->stream>>>(
        (T*)ms->buf[B2_BUF_STATE], (uint16_t*)ms->buf[B2_BUF_ELAPSED], s->n, ms->seed, ms->env_offset, 0,
        (T*)ms->buf[B2_BUF_RAND_PARAMS], ms->rand_mass_delta, ms->rand_gravity_sigma, s->gravity[2],
        ms->model->basis.mass[0], ms->model->basis.mass[1]);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

template <typename T>
int dispatch_reset_all(b2sim* s, ModelState* ms)
{
    switch (ms->task) {
    case B2_TASK_PENDULUM_SWINGUP: return launch_reset_all<B2_TASK_PENDULUM_SWINGUP, T>(s, ms);
    case B2_TASK_CARTPOLE_DISCRETE_BALANCING: return launch_reset_all<B2_TASK_CARTPOLE_DISCRETE_BALANCING, T>(s, ms);
    case B2_TASK_CARTPOLE_CONTINUOUS_BALANCING: return launch_reset_all<B2_TASK_CARTPOLE_CONTINUOUS_BALANCING, T>(s, ms);
    case B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP: return launch_reset_all<B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP, T>(s, ms);
    default: return fail(B2_ERR_UNSUPPORTED, "task %d has no fused kernel", ms->task);
    }
}

template <int TASK, typename T>
int launch_observe(b2sim* s, ModelState* ms)
{
    const int block = 256, grid = grid_for(s->n, block);
    b2::k_task_observe<TASK, T><<<grid, block, 0, s->stream>>>((const T*)ms->buf[B2_BUF_STATE], (T*)ms->buf[B2_BUF_OBS],
                                                               (T*)ms->buf[B2_BUF_REWARD], (uint8_t*)ms->buf[B2_BUF_DONE],
                                                               s->n);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

template <typename T>
int dispatch_observe(b2sim* s, ModelState* ms)
{
    if (ms->task == B2_TASK_PANDA_REACH) return launch_panda<T>(s, ms, nullptr, 1);
    switch (ms->task) {
    case B2_TASK_PENDULUM_SWINGUP: return launch_observe<B2_TASK_PENDULUM_SWINGUP, T>(s, ms);
    case B2_TASK_CARTPOLE_DISCRETE_BALANCING: return launch_observe<B2_TASK_CARTPOLE_DISCRETE_BALANCING, T>(s, ms);
    case B2_TASK_CARTPOLE_CONTINUOUS_BALANCING: return launch_observe<B2_TASK_CARTPOLE_CONTINUOUS_BALANCING, T>(s, ms);
    case B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP: return launch_observe<B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP, T>(s, ms);
    default: return fail(B2_ERR_UNSUPPORTED, "task %d has no fused kernel", ms->task);
    }
}

// element (env, col) of a [N, cols] buffer <-> host double
int read_elem(b2sim* s, const void* buf, int64_t cols, int64_t env, int col, double* out)
{
    if (s->dtype == B2_F64) {
        double v;
        B2_CUDA(cudaMemcpyAsync(&v, (const double*)buf + env * cols + col, 8, cudaMemcpyDeviceToHost, s->stream));
        B2_CUDA(cudaStreamSynchronize(s->stream));
        *out = v;
    } else {
        float v;
        B2_CUDA(cudaMemcpyAsync(&v, (const float*)buf + env * cols + col, 4, cudaMemcpyDeviceToHost, s->stream));
        B2_CUDA(cudaStreamSynchronize(s->stream));
        *out = v;
    }
    return B2_OK;
}
int write_elem(b2sim* s, void* buf, int64_t cols, int64_t env, int col, double value)
{
    if (s->dtype == B2_F64) {
        B2_CUDA(cudaMemcpyAsync((double*)buf + env * cols + col, &value, 8, cudaMemcpyHostToDevice, s->stream));
    } else {
        float v = (float)value;
        B2_CUDA(cudaMemcpyAsync((float*)buf + env * cols + col, &v, 4, cudaMemcpyHostToDevice, s->stream));
    }
    B2_CUDA(cudaStreamSynchronize(s->stream));  // the host value goes out of scope
    return B2_OK;
}

template <typename T>
int col_fill(b2sim* s, void* buf, int stride, int col, double value)
{
    b2::k_col_fill<T><<<grid_for(s->n, 256), 256, 0, s->stream>>>((T*)buf, s->n, stride, col, (T)value);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}
template <typename T>
int col_copy(b2sim* s, void* dst, int dstride, int dcol, const void* src, int sstride, int scol)
{
    b2::k_col_copy<T><<<grid_for(s->n, 256), 256, 0, s->stream>>>((T*)dst, dstride, dcol, (const T*)src, sstride, scol, s->n);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}
int col_fill_any(b2sim* s, void* buf, int stride, int col, double v)
{
    return s->dtype == B2_F64 ? col_fill<double>(s, buf, stride, col, v) : col_fill<float>(s, buf, stride, col, v);
}
int col_copy_any(b2sim* s, void* dst, int dstride, int dcol, const void* src, int sstride, int scol)
{
    return s->dtype == B2_F64 ? col_copy<double>(s, dst, dstride, dcol, src, sstride, scol)
                              : col_copy<float>(s, dst, dstride, dcol, src, sstride, scol);
}

template <typename T>
int launch_kinematics(b2sim* s, ModelState* ms)
{
    const int nq = ms->model->t.nq, block = 128, grid = grid_for(s->n, block);
    const b2::ModelDev<T>* tb = (const b2::ModelDev<T>*)ms->d_tables;
    const T* st = (const T*)ms->buf[B2_BUF_STATE];
    T* out = (T*)ms->buf[B2_BUF_LINK_POSE];
    if (nq <= 2) b2::k_kinematics<T, 2><<<grid, block, 0, s->stream>>>(tb, st, out, s->n);
    else if (nq <= 9) b2::k_kinematics<T, 9><<<grid, block, 0, s->stream>>>(tb, st, out, s->n);
    else b2::k_kinematics<T, 16><<<grid, block, 0, s->stream>>>(tb, st, out, s->n);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

template <typename T>
int launch_kindyn(b2sim* s, ModelState* ms, int link, void* M, void* h, void* J)
{
    const int nq = ms->model->t.nq, block = 128, grid = grid_for(s->n, block);
    const b2::ModelDev<T>* tb = (const b2::ModelDev<T>*)ms->d_tables;
    const T* st = (const T*)ms->buf[B2_BUF_STATE];
    if (nq <= 2) b2::k_kindyn<T, 2><<<grid, block, 0, s->stream>>>(tb, st, link, (T*)M, (T*)h, (T*)J, s->n);
    else if (nq <= 9) b2::k_kindyn<T, 9><<<grid, block, 0, s->stream>>>(tb, st, link, (T*)M, (T*)h, (T*)J, s->n);
    else b2::k_kindyn<T, 16><<<grid, block, 0, s->stream>>>(tb, st, link, (T*)M, (T*)h, (T*)J, s->n);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

template <typename T>
void fill_shape(b2::ShapeDev<T>& out, const b2_model_tables& t, int k, const b2::Pose& frame, int model, bool world_frame)
{
    out.type = t.shape_type[k];
    out.owner_model = model;
    out.owner_link = t.shape_link[k];
    b2::Pose sp;
    for (int a = 0; a < 9; ++a) sp.R.m[a] = t.shape_R[k][a];
    sp.p = {t.shape_p[k][0], t.shape_p[k][1], t.shape_p[k][2]};
    const int l = t.shape_link[k];
    b2::Pose lp;
    for (int a = 0; a < 9; ++a) lp.R.m[a] = t.link_R[l][a];
    lp.p = {t.link_p[l][0], t.link_p[l][1], t.link_p[l][2]};
    const b2::Pose full = b2::compose(frame, b2::compose(lp, sp));
    for (int a = 0; a < 9; ++a) out.R[a] = (T)full.R.m[a];
    out.p[0] = (T)full.p.x; out.p[1] = (T)full.p.y; out.p[2] = (T)full.p.z;
    if (out.type == B2_SHAPE_BOX) {
        for (int a = 0; a < 3; ++a) out.size[a] = (T)(0.5 * t.shape_size[k][a]);  // half extents
    } else if (out.type == B2_SHAPE_PLANE) {
        // unit normal in the world
        b2::V3<double> n{t.shape_size[k][0], t.shape_size[k][1], t.shape_size[k][2]};
        n = b2::mul(full.R, n);
        const double len = sqrt(b2::dot(n, n));
        out.size[0] = (T)(n.x / len); out.size[1] = (T)(n.y / len); out.size[2] = (T)(n.z / len);
    } else {
        for (int a = 0; a < 3; ++a) out.size[a] = (T)t.shape_size[k][a];
    }
    out.mu = (T)t.shape_mu[k];
    (void)world_frame;
}

// External wrenches on free bodies (Link::applyWorldWrench, Physics.cpp:1483-1532): the part of the device world
// description that changes while the world itself does not. `it` = physics iteration of the current run; a wrench acts
// on the iteration it was applied in and then for as long as the pre-step time is before its expiry (helpers.h:300-345).
template <typename T>
int upload_free_wrenches(b2sim* s, int it)
{
    struct { T ext[b2::kMaxFree][6]; long long env[b2::kMaxFree]; } host;
    memset(&host, 0, sizeof host);
    const int64_t t_pre = s->time_ns + (int64_t)it * s->dt_ns;
    for (size_t i = 0; i < s->free_models.size(); ++i) {
        host.env[i] = -2;
        for (const auto& w : s->models[s->free_models[i]]->wrenches) {
            if (it > 0 && t_pre >= w.expiry_ns) continue;
            for (int k = 0; k < 6; ++k) host.ext[i][k] = (T)w.w[k];
            host.env[i] = w.env;
        }
    }
    for (size_t i = s->free_models.size(); i < (size_t)b2::kMaxFree; ++i) host.env[i] = -2;
    B2_CUDA(cudaMemcpyAsync((char*)s->d_world + offsetof(b2::WorldDev<T>, ext), host.ext, sizeof host.ext, cudaMemcpyHostToDevice,
                            s->stream));
    B2_CUDA(cudaMemcpyAsync((char*)s->d_world + offsetof(b2::WorldDev<T>, ext_env), host.env, sizeof host.env,
                            cudaMemcpyHostToDevice, s->stream));
    B2_CUDA(cudaStreamSynchronize(s->stream));
    s->free_wrench_dirty = false;
    return B2_OK;
}

// (Re)builds the world description of the free bodies and static shapes and uploads it.
template <typename T>
int upload_world(b2sim* s)
{
    // large: kept off the stack, one per call (simulators on different threads must not share a staging copy)
    std::unique_ptr<b2::WorldDev<T>> staging(new b2::WorldDev<T>);
    b2::WorldDev<T>& W = *staging;
    memset(&W, 0, sizeof W);
    s->free_models.clear();
    s->static_shape_model.clear();
    s->static_shape_link.clear();
    s->robot_shape_link.clear();
    s->free_shape_col.clear();
    s->static_shape_col.clear();
    s->robot_shape_col.clear();
    s->robot_model = -1;
    W.iterations = s->contact_iterations;
    W.dt = (T)((double)s->dt_ns / 1e9);
    W.erp = (T)s->contact_erp;
    W.max_erv = (T)s->contact_max_erv;
    for (int k = 0; k < 3; ++k) W.g[k] = (T)s->gravity[k];
    for (size_t id = 0; id < s->models.size(); ++id) {
        ModelState* ms = s->models[id].get();
        if (ms->removed) continue;
        const b2_model_tables& t = ms->model->t;
        if (ms->kind == B2_KIND_FREE) {
            if (W.nfree >= b2::kMaxFree) return fail(B2_ERR_UNSUPPORTED, "more than %d free bodies in a world", b2::kMaxFree);
            b2::FreeBodyDev<T>& fb = W.body[W.nfree++];
            s->free_models.push_back((int)id);
            fb.mass = (T)t.body_mass;
            const double* I = t.body_Ic;
            const double det = I[0] * (I[4] * I[8] - I[5] * I[7]) - I[1] * (I[3] * I[8] - I[5] * I[6]) + I[2] * (I[3] * I[7] - I[4] * I[6]);
            if (!(t.body_mass > 0) || !(det > 0)) return fail(B2_ERR_INVALID, "free body '%s' needs a positive mass and inertia", ms->name.c_str());
            const double inv[9] = {(I[4] * I[8] - I[5] * I[7]) / det, (I[2] * I[7] - I[1] * I[8]) / det, (I[1] * I[5] - I[2] * I[4]) / det,
                                   (I[5] * I[6] - I[3] * I[8]) / det, (I[0] * I[8] - I[2] * I[6]) / det, (I[2] * I[3] - I[0] * I[5]) / det,
                                   (I[3] * I[7] - I[4] * I[6]) / det, (I[1] * I[6] - I[0] * I[7]) / det, (I[0] * I[4] - I[1] * I[3]) / det};
            for (int k = 0; k < 9; ++k) { fb.Ic[k] = (T)I[k]; fb.Ic_inv[k] = (T)inv[k]; }
            for (int k = 0; k < 3; ++k) fb.com[k] = (T)t.body_com[k];
            std::array<int, b2::kMaxBodyShapes> cols;
            cols.fill(-1);
            for (int k = 0; k < t.nshapes && fb.nshapes < b2::kMaxBodyShapes; ++k)
                if (t.shape_type[k] == B2_SHAPE_BOX || t.shape_type[k] == B2_SHAPE_SPHERE) {
                    cols[fb.nshapes] = k;
                    fill_shape(fb.shape[fb.nshapes++], t, k, b2::Pose(), (int)id, false);
                }
            s->free_shape_col.push_back(cols);
        } else if (ms->kind == B2_KIND_STATIC) {
            for (int k = 0; k < t.nshapes; ++k) {
                if (t.shape_type[k] != B2_SHAPE_BOX && t.shape_type[k] != B2_SHAPE_PLANE) continue;
                if (W.nstatic >= b2::kMaxStaticShapes) return fail(B2_ERR_UNSUPPORTED, "too many static collision shapes");
                fill_shape(W.stat[W.nstatic++], t, k, ms->base, (int)id, true);
                s->static_shape_model.push_back((int)id);
                s->static_shape_link.push_back(t.shape_link[k]);
                s->static_shape_col.push_back(k);
            }
        } else if (t.nq > 0 && s->robot_model < 0) {
            // articulated model: box / sphere shapes on its moving links collide with the free bodies and the static
            // shapes of the world (self-collisions stay off, Model.cpp:175-178). One such model per world.
            for (int k = 0; k < t.nshapes; ++k) {
                if (t.shape_type[k] != B2_SHAPE_BOX && t.shape_type[k] != B2_SHAPE_SPHERE) continue;
                const int body = t.link_body[t.shape_link[k]];
                if (body < 0 || W.nrobot >= b2::kMaxRobotShapes) continue;
                fill_shape(W.rshape[W.nrobot], t, k, b2::Pose(), (int)id, false);  // pose in the body frame
                W.rbody[W.nrobot++] = body;
                s->robot_shape_link.push_back(t.shape_link[k]);
                s->robot_shape_col.push_back(k);
            }
            if (W.nrobot > 0) s->robot_model = (int)id;
        }
    }
    W.robot_model = s->robot_model;
    for (int i = 0; i < b2::kMaxFree; ++i) W.ext_env[i] = -2;  // external wrenches are written by upload_free_wrenches
    s->free_wrench_dirty = true;
    if (!s->d_world) B2_CUDA(cudaMalloc(&s->d_world, sizeof(b2::WorldDev<double>)));
    B2_CUDA(cudaMemcpyAsync(s->d_world, &W, sizeof W, cudaMemcpyHostToDevice, s->stream));
    B2_CUDA(cudaStreamSynchronize(s->stream));
    if (W.nfree > 0 && !s->contact_count) {
        B2_CUDA(cudaMalloc(&s->contact_count, (size_t)s->n * sizeof(int32_t)));
        B2_CUDA(cudaMalloc(&s->contact_ids, (size_t)s->n * b2::kMaxContacts * 4 * sizeof(int32_t)));
        B2_CUDA(cudaMalloc(&s->contact_data, (size_t)s->n * b2::kMaxContacts * b2::kContactRec * sizeof(double)));
        B2_CUDA(cudaMemsetAsync(s->contact_count, 0, (size_t)s->n * sizeof(int32_t), s->stream));
    }
    // Warp-cooperative solver: lanes = generalized velocities of one world (joints of the coupled articulated model +
    // 6 per free body), 16 or 32 per env. Larger worlds, or row buffers beyond 8 GB, use the single-thread kernels.
    for (void** p : {&s->pgs_v, &s->pgs_J, &s->pgs_Y, &s->pgs_par, &s->pgs_lam, &s->pgs_aux})
        if (*p) { cudaFree(*p); *p = nullptr; }
    if (s->pgs_cnt) { cudaFree(s->pgs_cnt); s->pgs_cnt = nullptr; }
    s->pgs_nvp = 0;
    static const char* solver = getenv("B2_CONTACT_SOLVER");
    // Free bodies alone: the pipeline wins while the batch leaves schedulers idle (kWarpSolverMaxEnvs), the
    // single-thread kernel above that (launch_world).
    if (W.nfree > 0 && !(solver && !strcmp(solver, "thread")) &&
        (s->robot_model >= 0 || (solver && !strcmp(solver, "warp")) || s->n <= kWarpSolverMaxEnvs)) {
        const int rnq = s->robot_model >= 0 ? s->models[s->robot_model]->model->t.nq : 0;
        const int nv = rnq + 6 * W.nfree;
        const int nvp = nv <= 16 ? 16 : 32;
        const size_t row_bytes = (size_t)s->n * b2::kMaxPgsRows * nvp * sizeof(T);
        if (nv <= 32 && 2 * row_bytes <= ((size_t)8 << 30)) {
            B2_CUDA(cudaMalloc(&s->pgs_v, (size_t)s->n * nvp * sizeof(T)));
            B2_CUDA(cudaMalloc(&s->pgs_J, row_bytes));
            B2_CUDA(cudaMalloc(&s->pgs_Y, row_bytes));
            B2_CUDA(cudaMalloc(&s->pgs_par, (size_t)s->n * b2::kMaxPgsRows * 4 * sizeof(T)));
            B2_CUDA(cudaMalloc(&s->pgs_lam, (size_t)s->n * b2::kMaxPgsRows * sizeof(T)));
            B2_CUDA(cudaMalloc(&s->pgs_aux, (size_t)s->n * b2::pgs_aux_size(rnq, W.nfree) * sizeof(T)));
            B2_CUDA(cudaMemsetAsync(s->pgs_aux, 0, (size_t)s->n * b2::pgs_aux_size(rnq, W.nfree) * sizeof(T), s->stream));
            s->pgs_nq = rnq;
            s->pgs_nfree = W.nfree;
            B2_CUDA(cudaMalloc((void**)&s->pgs_cnt, (size_t)s->n * 2 * sizeof(int)));
            B2_CUDA(cudaMemsetAsync(s->pgs_cnt, 0, (size_t)s->n * 2 * sizeof(int), s->stream));
            s->pgs_nvp = nvp;
        }
    }
    s->world_dirty = false;
    return B2_OK;
}

template <typename T>
b2::PgsBuffers<T> pgs_buffers(b2sim* s)
{
    b2::PgsBuffers<T> g;
    g.v = (T*)s->pgs_v; g.J = (T*)s->pgs_J; g.Y = (T*)s->pgs_Y; g.par = (T*)s->pgs_par; g.lam = (T*)s->pgs_lam;
    g.aux = (T*)s->pgs_aux;
    g.cnt = s->pgs_cnt; g.nvp = s->pgs_nvp; g.nq = s->pgs_nq; g.nfree = s->pgs_nfree;
    g.aux_stride = b2::pgs_aux_size(s->pgs_nq, s->pgs_nfree);
    g.n = s->n;
    return g;
}

template <typename T>
b2::WorldBuffers<T> world_buffers(b2sim* s, int paused)
{
    b2::WorldBuffers<T> b;
    memset(&b, 0, sizeof b);
    for (size_t i = 0; i < s->free_models.size(); ++i) {
        ModelState* ms = s->models[s->free_models[i]].get();
        b.base_state[i] = (T*)ms->buf[B2_BUF_BASE_STATE];
        b.base_reset[i] = (T*)ms->buf[B2_BUF_BASE_RESET];
        b.reset_mask[i] = (uint32_t*)ms->buf[B2_BUF_RESET_MASK];
        b.base_accel[i] = (T*)ms->buf[B2_BUF_BASE_ACCEL];
    }
    b.contact_count = s->contact_count;
    b.contact_ids = s->contact_ids;
    b.contact_data = (T*)s->contact_data;
    b.n = s->n;
    b.paused = paused;
    return b;
}

// Per-env rows of the world's slots (b2sim_enable_free_body_params, b2sim_enable_shape_friction), resolved on every launch so
// that enabling or disabling rows needs no world rebuild. *any: some model of the world has rows (the ENV kernels run).
template <typename T>
b2::WorldRows<T> world_rows(const b2sim* s, bool* any)
{
    b2::WorldRows<T> r;
    memset(&r, 0, sizeof r);
    *any = false;
    for (const auto& ms : s->models)
        if (!ms->removed && (ms->body_rows || ms->mu_rows)) *any = true;
    if (!*any) return r;
    for (size_t i = 0; i < s->free_models.size(); ++i) {
        const ModelState* ms = s->models[s->free_models[i]].get();
        r.body[i] = (const T*)ms->body_rows;
        r.body_mu_stride[i] = ms->model->t.nshapes;
        for (int k = 0; k < b2::kMaxBodyShapes; ++k)
            if (ms->mu_rows && s->free_shape_col[i][k] >= 0) r.body_mu[i][k] = (const T*)ms->mu_rows + s->free_shape_col[i][k];
    }
    for (size_t k = 0; k < s->static_shape_col.size(); ++k) {
        const ModelState* ms = s->models[s->static_shape_model[k]].get();
        r.stat_mu_stride[k] = ms->model->t.nshapes;
        if (ms->mu_rows) r.stat_mu[k] = (const T*)ms->mu_rows + s->static_shape_col[k];
    }
    if (s->robot_model >= 0) {
        const ModelState* ms = s->models[s->robot_model].get();
        r.robot_mu_stride = ms->model->t.nshapes;
        for (size_t k = 0; k < s->robot_shape_col.size(); ++k)
            if (ms->mu_rows) r.robot_mu[k] = (const T*)ms->mu_rows + s->robot_shape_col[k];
    }
    return r;
}

// Solve + finish launches that follow a prepare kernel (not on paused runs).
template <typename T>
int launch_solve_finish(b2sim* s, ModelState* robot, bool clear_robot_mask = false)
{
    const b2::PgsBuffers<T> g = pgs_buffers<T>(s);
    // 64-thread blocks, NVP lanes per env (4 or 2 envs per block); the lower block triangle of A = J M^-1 J^T of every
    // env in shared memory, seven blocks per SM
    if (g.nvp == 16) {
        constexpr int smem = 4 * b2::pgs_smem_per_env<T, 16>() * (int)sizeof(T);
        B2_CUDA(cudaFuncSetAttribute(b2::k_pgs_solve<T, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        b2::k_pgs_solve<T, 16><<<grid_for(s->n, 4), 64, smem, s->stream>>>(g, s->contact_iterations);
    } else {
        constexpr int smem = 2 * b2::pgs_smem_per_env<T, 32>() * (int)sizeof(T);
        B2_CUDA(cudaFuncSetAttribute(b2::k_pgs_solve<T, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        b2::k_pgs_solve<T, 32><<<grid_for(s->n, 2), 64, smem, s->stream>>>(g, s->contact_iterations);
    }
    B2_CUDA(cudaGetLastError());
    bool env = false;
    const b2::WorldRows<T> rows = world_rows<T>(s, &env);
    (env ? b2::k_world_finish<T, true> : b2::k_world_finish<T, false>)<<<grid_for(s->n * b2::kFinishLanes, 128), 128, 0, s->stream>>>(
        (const b2::WorldDev<T>*)s->d_world, world_buffers<T>(s, 0), g, robot ? (T*)robot->buf[B2_BUF_STATE] : nullptr,
        robot ? (T*)robot->buf[B2_BUF_ACCELERATION] : nullptr, robot ? robot->model->t.nq : 0,
        robot && clear_robot_mask ? (uint32_t*)robot->buf[B2_BUF_RESET_MASK] : nullptr, rows);
    B2_CUDA(cudaGetLastError());
    s->launches += 2;
    return B2_OK;
}

template <typename T>
int launch_world(b2sim* s, int paused)
{
    if (s->free_models.empty()) return B2_OK;
    // Free bodies alone, measured on the B200 (two stacked cubes, 8 contacts, 50 sweeps): the prepare / solve / finish
    // pipeline takes 182 / 269 / 853 / 3222 us per step at 1,024 / 4,096 / 16,384 / 65,536 envs, the single-thread kernel
    // (k_world_free) 341 / 344 / 601 / 1882 us: the pipeline spreads an env over a warp's lanes, which pays while the batch
    // leaves schedulers idle and costs instruction issue once it does not. B2_CONTACT_SOLVER=warp / thread overrides.
    static const char* solver = getenv("B2_CONTACT_SOLVER");
    const bool forced_thread = solver && !strcmp(solver, "thread");
    const bool forced_warp = solver && !strcmp(solver, "warp");
    bool env = false;
    const b2::WorldRows<T> rows = world_rows<T>(s, &env);
    if (s->pgs_nvp && !forced_thread && (forced_warp || s->n <= kWarpSolverMaxEnvs)) {
        const int block = s->n <= kWarpSolverMaxEnvs ? 32 : 64;  // small batches: one warp per SM
        (env ? b2::k_world_prepare<T, true> : b2::k_world_prepare<T, false>)<<<grid_for(s->n, block), block, 0, s->stream>>>(
            (const b2::WorldDev<T>*)s->d_world, world_buffers<T>(s, paused), pgs_buffers<T>(s), rows);
        ++s->launches;
        B2_CUDA(cudaGetLastError());
        return paused ? B2_OK : launch_solve_finish<T>(s, nullptr);
    }
    (env ? b2::k_world_free<T, true> : b2::k_world_free<T, false>)<<<grid_for(s->n, 64), 64, 0, s->stream>>>(
        (const b2::WorldDev<T>*)s->d_world, world_buffers<T>(s, paused), rows);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

// One iteration of a coupled world: the articulated model `ms` and every free body in one launch.
template <typename T>
int launch_coupled(b2sim* s, ModelState* ms, int paused, uint32_t compute_bit, uint32_t ct_bit, const int* wrench_iters)
{
    const b2::RunCfg<T> cfg = build_run_cfg<T>(s, ms, paused, 1, compute_bit, ct_bit, wrench_iters);
    b2::TreeTopo topo;
    int rc = tree_topology(ms, &topo);
    if (rc != B2_OK) return rc;
    const char* split_env = getenv("B2_COUPLED_SPLIT");  // read per launch: tests compare the two pipelines in one process
    bool env = false;
    const b2::WorldRows<T> rows = world_rows<T>(s, &env);
    if (s->pgs_nvp && !paused && !(split_env && !strcmp(split_env, "0"))) {
        // Unpaused step: the three independent parts of the prepare stage run concurrently on forked streams
        // (b2_kernels.cuh, "Split prepare"); the solve waits for all of them. 32-thread blocks: at the 4,096-env size of
        // this configuration every warp gets an SM (and its L1) of its own.
        if (!s->fork[0]) {
            for (int k = 0; k < 2; ++k) B2_CUDA(cudaStreamCreateWithFlags(&s->fork[k], cudaStreamNonBlocking));
            for (int k = 0; k < 3; ++k) B2_CUDA(cudaEventCreateWithFlags(&s->fork_ev[k], cudaEventDisableTiming));
            // The three kernels must be able to share an SM: each is one 32-thread block per SM at 4,096 envs. An SM is
            // configured with ONE shared-memory / L1 split at a time, and left to its own heuristic the driver picks a
            // different split for each of them (from the blocks per SM their registers would allow), so a kernel could only
            // start on SMs the others had left (measured: rows ended 360 us and M^-1 290 us after the fork instead of 94
            // and 65 us). The same explicit split for all three (64 KB shared, the rest L1 for their per-thread scratch).
            const int carve = b2::kCoupledCarveout;
            B2_CUDA(cudaFuncSetAttribute(b2::k_coupled_dynamics<T>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
            B2_CUDA(cudaFuncSetAttribute(b2::k_coupled_rows<T, false>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
            B2_CUDA(cudaFuncSetAttribute(b2::k_coupled_rows<T, true>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
            B2_CUDA(cudaFuncSetAttribute(b2::k_coupled_minv<T>, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
        }
        const b2::RunBuffers<T> rb = run_buffers<T>(s, ms);
        const b2::PgsBuffers<T> g = pgs_buffers<T>(s);
        const b2::ModelDev<T>* tb = (const b2::ModelDev<T>*)ms->d_tables;
        // B2_COUPLED_TRACE=1: device timeline of every 128th step on stderr (when each of the forked kernels ended,
        // relative to the fork point, and the end of the step)
        static const bool trace = getenv("B2_COUPLED_TRACE") != nullptr;
        static cudaEvent_t tev[5];
        static uint64_t tcount = 0;
        const bool tr = trace && (tcount++ % 128) == 127;
        if (tr && !tev[0]) for (auto& e : tev) cudaEventCreate(&e);
        if (tr) cudaEventRecord(tev[0], s->stream);
        B2_CUDA(cudaEventRecord(s->fork_ev[0], s->stream));
        B2_CUDA(cudaStreamWaitEvent(s->fork[0], s->fork_ev[0], 0));
        B2_CUDA(cudaStreamWaitEvent(s->fork[1], s->fork_ev[0], 0));
        // launch order = block dispatch order: the longest kernel (rows) first, the lane-parallel dynamics last
        (env ? b2::k_coupled_rows<T, true> : b2::k_coupled_rows<T, false>)<<<grid_for(s->n, 32), 32, 0, s->fork[0]>>>(
            tb, cfg, rb, (const b2::WorldDev<T>*)s->d_world, world_buffers<T>(s, 0), g, rows);
        if (tr) cudaEventRecord(tev[2], s->fork[0]);
        b2::k_coupled_minv<T><<<grid_for(s->n, 32), 32, 0, s->fork[1]>>>(tb, rb, g);
        if (tr) cudaEventRecord(tev[3], s->fork[1]);
        // the articulated model's controllers + forward dynamics: on lanes for the small batches of this configuration
        // (k_run_tree_lanes<COUPLED>), one thread per env otherwise; unlike launch_run, whatever the joint count
        if (run_on_lanes(s, ms, 0)) {
            B2_CUDA(b2::launch_run_tree_lanes<T>(tb, (const b2::LaneTable<T>*)ms->d_lane_table, cfg, rb, ms->model->t.parent,
                                                 ms->model->t.jtype, s->stream, g.v, g.nvp));
        } else {
            b2::k_coupled_dynamics<T><<<grid_for(s->n, 32), 32, 0, s->stream>>>(tb, cfg, rb, topo, g);
        }
        if (tr) cudaEventRecord(tev[1], s->stream);
        B2_CUDA(cudaGetLastError());
        B2_CUDA(cudaEventRecord(s->fork_ev[1], s->fork[0]));
        B2_CUDA(cudaEventRecord(s->fork_ev[2], s->fork[1]));
        B2_CUDA(cudaStreamWaitEvent(s->stream, s->fork_ev[1], 0));
        B2_CUDA(cudaStreamWaitEvent(s->stream, s->fork_ev[2], 0));
        s->launches += 3;
        rc = launch_solve_finish<T>(s, ms, true);
        if (tr) {
            cudaEventRecord(tev[4], s->stream);
            cudaEventSynchronize(tev[4]);
            float d[4];
            for (int k = 0; k < 4; ++k) cudaEventElapsedTime(&d[k], tev[0], tev[k + 1]);
            fprintf(stderr, "[b2sim trace] dynamics end %.1f us, rows end %.1f us, minv end %.1f us, step end %.1f us\n", d[0] * 1e3f,
                    d[1] * 1e3f, d[2] * 1e3f, d[3] * 1e3f);
        }
        return rc;
    }
    if (s->pgs_nvp) {
        // 32-thread blocks: at the 4,096-env size of this configuration every warp gets an SM (and its L1) of its own
        (env ? b2::k_coupled_prepare<T, true> : b2::k_coupled_prepare<T, false>)<<<grid_for(s->n, 32), 32, 0, s->stream>>>(
            (const b2::ModelDev<T>*)ms->d_tables, cfg, run_buffers<T>(s, ms), topo, (const b2::WorldDev<T>*)s->d_world,
            world_buffers<T>(s, paused), pgs_buffers<T>(s), rows);
        ++s->launches;
        B2_CUDA(cudaGetLastError());
        return paused ? B2_OK : launch_solve_finish<T>(s, ms);
    }
    (env ? b2::k_world_coupled<T, true> : b2::k_world_coupled<T, false>)<<<grid_for(s->n, 64), 64, 0, s->stream>>>(
        (const b2::ModelDev<T>*)ms->d_tables, cfg, run_buffers<T>(s, ms), topo, (const b2::WorldDev<T>*)s->d_world,
        world_buffers<T>(s, paused), rows);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

template <typename T>
int launch_link_motion(b2sim* s, ModelState* ms, int link, void* twist, void* accel)
{
    const int nq = ms->model->t.nq, block = 128, grid = grid_for(s->n, block);
    const b2::ModelDev<T>* tb = (const b2::ModelDev<T>*)ms->d_tables;
    const T* st = (const T*)ms->buf[B2_BUF_STATE];
    const T* ac = (const T*)ms->buf[B2_BUF_ACCELERATION];
    if (nq <= 2) b2::k_link_motion<T, 2><<<grid, block, 0, s->stream>>>(tb, st, ac, link, (T*)twist, (T*)accel, s->n);
    else if (nq <= 9) b2::k_link_motion<T, 9><<<grid, block, 0, s->stream>>>(tb, st, ac, link, (T*)twist, (T*)accel, s->n);
    else b2::k_link_motion<T, 16><<<grid, block, 0, s->stream>>>(tb, st, ac, link, (T*)twist, (T*)accel, s->n);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

void free_model_buffers(ModelState* ms)
{
    for (auto& b : ms->buf)
        if (b) { cudaFree(b); b = nullptr; }
    if (ms->force_read) { cudaFree(ms->force_read); ms->force_read = nullptr; }
    if (ms->body_rows) { cudaFree(ms->body_rows); ms->body_rows = nullptr; }
    if (ms->mu_rows) { cudaFree(ms->mu_rows); ms->mu_rows = nullptr; }
    if (ms->d_tables) { cudaFree(ms->d_tables); ms->d_tables = nullptr; }
    if (ms->d_step) { cudaFree(ms->d_step); ms->d_step = nullptr; }
    if (ms->d_ticket) { cudaFree(ms->d_ticket); ms->d_ticket = nullptr; }
    if (ms->d_ep_totals) { cudaFree(ms->d_ep_totals); ms->d_ep_totals = nullptr; }
    for (void** p : {&ms->pinned_actions, &ms->pinned_obs, &ms->pinned_reward, &ms->pinned_done})
        if (*p) { cudaFreeHost(*p); *p = nullptr; }
}

// Shared part of b2sim_enable_free_body_params / b2sim_enable_shape_friction: `rows` is the model's [N, cols] allocation,
// `init` its first row, copied into every env.
int enable_rows(b2sim* s, void*& rows, int enable, int cols, const double* init, b2_buffer* out)
{
    if (!enable) {
        if (rows) {
            B2_CUDA(cudaStreamSynchronize(s->stream));  // runs still queued read the rows
            cudaFree(rows);
            rows = nullptr;
        }
        return B2_OK;
    }
    if (!rows) {
        B2_CUDA(cudaMalloc(&rows, (size_t)s->n * cols * s->esize()));
        for (int k = 0; k < cols; ++k) {
            const int rc = col_fill_any(s, rows, cols, k, init[k]);
            if (rc != B2_OK) {
                cudaFree(rows);
                rows = nullptr;
                return rc;
            }
        }
    }
    if (out) *out = b2_buffer{rows, s->n, cols, s->dtype, (int32_t)s->esize()};
    return B2_OK;
}
}  // namespace

// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {

const char* b2sim_last_error(void) { return g_error.c_str(); }
int b2sim_version(void) { return 100; }

int b2sim_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// ---- model loader -----------------------------------------------------------------------------------
b2model* b2model_parse(const char* xml, size_t len)
{
    if (!xml) { fail(B2_ERR_INVALID, "null model description"); return nullptr; }
    try {
        b2model* m = b2::parse_model(xml, len);
        const double g[3] = {0, 0, -9.8};
        m->fit(b2::Pose(), g, 0.001);  // default classification; re-fitted on insertion
        return m;
    } catch (const std::exception& e) {
        fail(B2_ERR_PARSE, "%s", e.what());
        return nullptr;
    }
}
b2model* b2model_parse_file(const char* path)
{
    std::ifstream f(path ? path : "");
    if (!f) { fail(B2_ERR_NOT_FOUND, "cannot open model file '%s'", path ? path : ""); return nullptr; }
    std::stringstream ss;
    ss << f.rdbuf();
    const std::string xml = ss.str();
    return b2model_parse(xml.data(), xml.size());
}
void b2model_free(b2model* m) { delete m; }
const char* b2model_name(const b2model* m) { return m ? m->name.c_str() : ""; }
int b2model_kind(const b2model* m) { return m ? m->t.kind : B2_ERR_INVALID; }
int b2model_dofs(const b2model* m) { return m ? m->t.nq : B2_ERR_INVALID; }
int b2model_num_links(const b2model* m) { return m ? m->t.nlinks : B2_ERR_INVALID; }
int b2model_num_joints(const b2model* m) { return m ? (int)m->joint_names.size() : B2_ERR_INVALID; }
const char* b2model_joint_name(const b2model* m, int j)
{
    return (m && j >= 0 && j < (int)m->joint_names.size()) ? m->joint_names[j].c_str() : nullptr;
}
const char* b2model_link_name(const b2model* m, int l)
{
    return (m && l >= 0 && l < (int)m->link_names.size()) ? m->link_names[l].c_str() : nullptr;
}
int b2model_joint_index(const b2model* m, const char* name)
{
    if (!m || !name) return B2_ERR_INVALID;
    for (size_t j = 0; j < m->joint_names.size(); ++j)
        if (m->joint_names[j] == name) return (int)j;
    return fail(B2_ERR_NOT_FOUND, "joint '%s' not found in model '%s'", name, m->name.c_str());
}
int b2model_link_index(const b2model* m, const char* name)
{
    if (!m || !name) return B2_ERR_INVALID;
    for (size_t l = 0; l < m->link_names.size(); ++l)
        if (m->link_names[l] == name) return (int)l;
    return fail(B2_ERR_NOT_FOUND, "link '%s' not found in model '%s'", name, m->name.c_str());
}
int b2model_tables(const b2model* m, b2_model_tables* out)
{
    if (!m || !out) return fail(B2_ERR_INVALID, "null argument");
    *out = m->t;
    return B2_OK;
}

// ---- simulator ----------------------------------------------------------------------------------------
b2sim* b2sim_create(int device, int64_t num_envs, double step_size, int steps_per_run, int dtype)
{
    // GazeboSimulator::initialize rejects non-positive step size / iterations (GazeboSimulator.cpp:169-195)
    if (!(step_size > 0) || steps_per_run <= 0 || steps_per_run > 32 || num_envs <= 0 ||
        (dtype != B2_F64 && dtype != B2_F32)) {
        fail(B2_ERR_INVALID, "invalid simulator configuration");
        return nullptr;
    }
    int count = b2sim_device_count();
    if (count <= 0) {
        fail(B2_ERR_CUDA, "no CUDA device: the b2sim engine has no CPU execution path");
        return nullptr;
    }
    if (device < 0 || device >= count) {
        fail(B2_ERR_INVALID, "device %d out of range (%d visible)", device, count);
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) {
        fail(B2_ERR_CUDA, "cudaSetDevice(%d) failed", device);
        return nullptr;
    }
    auto* s = new b2sim();
    s->device = device;
    s->n = num_envs;
    s->step_size = step_size;
    s->dt_ns = to_ns(step_size);
    s->steps_per_run = steps_per_run;
    s->dtype = dtype;
    return s;
}

void b2sim_destroy(b2sim* s)
{
    if (!s) return;
    DeviceGuard guard__(s->device);
    cudaStreamSynchronize(s->stream);
    for (auto& ms : s->models) free_model_buffers(ms.get());
    for (void* p : {(void*)s->d_world, (void*)s->contact_count, (void*)s->contact_ids, s->contact_data, s->pgs_v, s->pgs_J,
                    s->pgs_Y, s->pgs_par, s->pgs_lam, s->pgs_aux, (void*)s->pgs_cnt})
        if (p) cudaFree(p);
    for (cudaEvent_t ev : s->events) cudaEventDestroy(ev);
    if (s->copy_in) cudaStreamDestroy(s->copy_in);
    for (int k = 0; k < 2; ++k) if (s->fork[k]) cudaStreamDestroy(s->fork[k]);
    for (int k = 0; k < 3; ++k) if (s->fork_ev[k]) cudaEventDestroy(s->fork_ev[k]);
    if (s->copy_out) cudaStreamDestroy(s->copy_out);
    delete s;
}

int64_t b2sim_num_envs(const b2sim* s) { return s ? s->n : 0; }
double b2sim_step_size(const b2sim* s) { return s ? s->step_size : 0; }
int b2sim_steps_per_run(const b2sim* s) { return s ? s->steps_per_run : 0; }
int b2sim_dtype(const b2sim* s) { return s ? s->dtype : B2_ERR_INVALID; }
int b2sim_set_stream(b2sim* s, void* stream)
{
    if (!s) return fail(B2_ERR_INVALID, "null simulator");
    DeviceGuard guard__(s->device);
    if ((cudaStream_t)stream != s->stream) {
        // work already queued on the old stream (buffer clears, resets, steps) is ordered before anything on the new one
        cudaEvent_t ev;
        B2_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        cudaError_t rc = cudaEventRecord(ev, s->stream);
        if (rc == cudaSuccess) rc = cudaStreamWaitEvent((cudaStream_t)stream, ev, 0);
        cudaEventDestroy(ev);
        B2_CUDA(rc);
    }
    s->stream = (cudaStream_t)stream;
    return B2_OK;
}
int b2sim_synchronize(b2sim* s)
{
    if (!s) return fail(B2_ERR_INVALID, "null simulator");
    DeviceGuard guard__(s->device);
    B2_CUDA(cudaStreamSynchronize(s->stream));
    return B2_OK;
}
double b2sim_time(const b2sim* s) { return s ? (double)s->time_ns / 1e9 : 0.0; }
uint64_t b2sim_launch_count(const b2sim* s) { return s ? s->launches : 0; }

int b2sim_set_gravity(b2sim* s, const double g[3])
{
    if (!s || !g) return fail(B2_ERR_INVALID, "null argument");
    if (s->time_ns != 0) return fail(B2_ERR_INVALID, "gravity can only be changed before the first step");
    DeviceGuard guard__(s->device);
    for (int k = 0; k < 3; ++k) s->gravity[k] = g[k];
    for (auto& ms : s->models)
        if (!ms->removed) {
            int rc = refresh_tables(s, ms.get());
            for (int k = 0; k < 3 && rc == B2_OK && ms->env_params; ++k) rc = col_fill_any(s, ms->buf[B2_BUF_GRAVITY], 3, k, g[k]);
            if (rc != B2_OK) return rc;
        }
    s->world_dirty = true;  // the free-body world description carries the gravity vector too
    return B2_OK;
}
int b2sim_gravity(const b2sim* s, double g[3])
{
    if (!s || !g) return fail(B2_ERR_INVALID, "null argument");
    for (int k = 0; k < 3; ++k) g[k] = s->gravity[k];
    return B2_OK;
}

int b2sim_insert_model(b2sim* s, const char* xml, size_t len, const double pose[7], const char* name)
{
    if (!s || !xml) return fail(B2_ERR_INVALID, "null argument");
    DeviceGuard guard__(s->device);
    std::unique_ptr<b2model> m;
    try {
        m.reset(b2::parse_model(xml, len));
    } catch (const std::exception& e) {
        return fail(B2_ERR_PARSE, "%s", e.what());
    }
    auto ms = std::make_unique<ModelState>();
    ms->name = (name && *name) ? name : m->name;
    for (auto& other : s->models)  // World.cpp:86-93: names are unique within a world
        if (!other->removed && other->name == ms->name)
            return fail(B2_ERR_INVALID, "a model named '%s' already exists", ms->name.c_str());
    if (pose) ms->base = b2::pose_from_xyz_quat(pose);
    ms->model = std::move(m);
    const int nq = ms->model->t.nq;
    for (int j = 0; j < B2_MAX_DOFS; ++j) {
        ms->mode[j] = B2_MODE_IDLE;                                   // Joint.cpp:126-127
        ms->pid[j] = b2_pid{1, 0.1, 0.01, -1, 0, -1, 0, 0};           // DefaultPID, Joint.cpp:63
        ms->has_force_cmd[j] = ms->has_vel_cmd[j] = ms->has_pos_target[j] = ms->has_vel_target[j] = false;
        ms->effort[j] = j < nq ? ms->model->t.effort[j] : 0.0;
    }
    int rc = refresh_tables(s, ms.get());
    if (rc != B2_OK) return rc;
    if (nq > 0) {
        for (int which : {B2_BUF_STATE, B2_BUF_ACCELERATION, B2_BUF_FORCE_CMD, B2_BUF_POS_TARGET, B2_BUF_VEL_TARGET,
                          B2_BUF_ACC_TARGET, B2_BUF_PID_STATE, B2_BUF_RESET_STATE, B2_BUF_RESET_MASK}) {
            rc = ensure_buffer(s, ms.get(), which);
            if (rc != B2_OK) { free_model_buffers(ms.get()); return rc; }
        }
        if (cudaMalloc(&ms->force_read, (size_t)s->n * nq * s->esize()) != cudaSuccess ||
            cudaMemsetAsync(ms->force_read, 0, (size_t)s->n * nq * s->esize(), s->stream) != cudaSuccess) {
            free_model_buffers(ms.get());
            return fail(B2_ERR_CUDA, "allocating the joint force readback failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
    }
    if (ms->kind == B2_KIND_FREE) {
        for (int which : {B2_BUF_BASE_STATE, B2_BUF_BASE_RESET, B2_BUF_RESET_MASK, B2_BUF_BASE_ACCEL}) {
            rc = ensure_buffer(s, ms.get(), which);
            if (rc != B2_OK) { free_model_buffers(ms.get()); return rc; }
        }
        // the insertion pose is the initial base pose of every env (World.cpp:169-177); velocity zero
        double q[7] = {0, 0, 0, 1, 0, 0, 0};
        if (pose) memcpy(q, pose, sizeof q);
        for (int k = 0; k < 13; ++k) {
            rc = col_fill_any(s, ms->buf[B2_BUF_BASE_STATE], 13, k, k < 7 ? q[k] : 0.0);
            if (rc != B2_OK) { free_model_buffers(ms.get()); return rc; }
        }
    }
    s->world_dirty = true;
    s->models.push_back(std::move(ms));
    return (int)s->models.size() - 1;
}

int b2sim_remove_model(b2sim* s, int model)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    DeviceGuard guard__(s->device);
    cudaStreamSynchronize(s->stream);
    free_model_buffers(ms);
    ms->removed = true;
    s->world_dirty = true;
    return B2_OK;
}
int b2sim_num_models(const b2sim* s)
{
    int c = 0;
    if (s)
        for (auto& ms : s->models) c += !ms->removed;
    return c;
}
int b2sim_model_id(const b2sim* s, const char* name)
{
    if (!s || !name) return fail(B2_ERR_INVALID, "null argument");
    for (size_t i = 0; i < s->models.size(); ++i)
        if (!s->models[i]->removed && s->models[i]->name == name) return (int)i;
    return fail(B2_ERR_NOT_FOUND, "model '%s' not found", name);
}
const char* b2sim_model_name(const b2sim* s, int model)
{
    ModelState* ms = get_model(s, model);
    return ms ? ms->name.c_str() : nullptr;
}
const b2model* b2sim_model(const b2sim* s, int model)
{
    ModelState* ms = get_model(s, model);
    return ms ? ms->model.get() : nullptr;
}

// ---- GazeboSimulator::run ----------------------------------------------------------------------------
int b2sim_run(b2sim* s, int paused)
{
    if (!s) return fail(B2_ERR_INVALID, "null simulator");
    DeviceGuard guard__(s->device);
    const int iterations = paused ? 1 : s->steps_per_run;
    if (s->world_dirty) {
        int rc = s->dtype == B2_F64 ? upload_world<double>(s) : upload_world<float>(s);
        if (rc != B2_OK) return rc;
    }
    if (!s->free_models.empty())  // a free body inserted after b2sim_enable_env_params
        for (auto& ms : s->models)
            if (!ms->removed && ms->env_params)
                return fail(B2_ERR_UNSUPPORTED, "model '%s' has per-env parameters and the world has free bodies",
                            ms->name.c_str());
    // An articulated model with link collision shapes shares its constraint solve with the free bodies of the world
    const int coupled = (s->robot_model >= 0 && !s->free_models.empty()) ? s->robot_model : -1;
    uint32_t c_bits = 0, c_ct_bits = 0;
    std::vector<int> c_wrench_iters(1, 0);
    for (size_t id = 0; id < s->models.size(); ++id) {
        ModelState* ms = s->models[id].get();
        if (ms->removed || ms->model->t.nq == 0) continue;
        // JointController rate gate, evaluated per iteration on the post-step time (JointController.cpp:128-169)
        uint32_t bits = 0;
        if (!paused && ms->controller_loaded) {
            int64_t t = s->time_ns;
            for (int it = 0; it < iterations; ++it) {
                t += s->dt_ns;
                double elapsed = (double)(t - ms->prev_update_ns) / 1e9;
                const double period = (double)ms->period_ns / 1e9;
                if (ms->prev_update_ns == 0) elapsed = period;
                if (elapsed >= period - DBL_EPSILON) {
                    ms->prev_update_ns = t;
                    bits |= 1u << it;
                }
            }
        }
        uint32_t ct_bits = 0;
        if (!paused && ms->ct_loaded) {  // ControllerRunner keeps its own update time (ControllerRunner.cpp:209-246)
            int64_t t = s->time_ns;
            for (int it = 0; it < iterations; ++it) {
                t += s->dt_ns;
                double elapsed = (double)(t - ms->ct_prev_update_ns) / 1e9;
                const double period = (double)ms->period_ns / 1e9;
                if (ms->ct_prev_update_ns == 0) elapsed = period;
                if (elapsed >= period - DBL_EPSILON) {
                    ms->ct_prev_update_ns = t;
                    ct_bits |= 1u << it;
                }
            }
        }
        // external wrenches: applied on every iteration until the post-step time reaches their expiry
        std::vector<int> wrench_iters(ms->wrenches.size() + 1, 0);
        if (!paused) {
            for (size_t k = 0; k < ms->wrenches.size(); ++k) {
                int64_t t = s->time_ns;
                for (int it = 0; it < iterations; ++it) {
                    t += s->dt_ns;
                    wrench_iters[k] = it + 1;
                    if (t >= ms->wrenches[k].expiry_ns) break;
                }
            }
        }
        if ((int)id == coupled) {
            // stepped below, one launch per iteration together with the free bodies
            c_bits = bits;
            c_ct_bits = ct_bits;
            c_wrench_iters = wrench_iters;
            continue;
        }
        int rc = s->dtype == B2_F64 ? launch_run<double>(s, ms, paused, iterations, bits, ct_bits, wrench_iters.data())
                                    : launch_run<float>(s, ms, paused, iterations, bits, ct_bits, wrench_iters.data());
        if (rc != B2_OK) return rc;
        if (!paused) {
            const int64_t t_end = s->time_ns + (int64_t)iterations * s->dt_ns;
            auto& ws = ms->wrenches;
            ws.erase(std::remove_if(ws.begin(), ws.end(), [t_end](const ModelState::LinkWrench& w) { return t_end >= w.expiry_ns; }),
                     ws.end());
        }
        if (!paused && ms->controller_loaded)
            for (int j = 0; j < ms->model->t.nq; ++j)
                if (ms->mode[j] == B2_MODE_POSITION || ms->mode[j] == B2_MODE_VELOCITY)
                    ms->has_force_cmd[j] = true;  // the PID wrote JointForceCmd (JointController.cpp:316)
                else if (ms->mode[j] == B2_MODE_VELOCITY_FOLLOWER_DART)
                    ms->has_vel_cmd[j] = true;
    }
    // free bodies and their contacts (and the coupled articulated model): one launch per physics iteration
    bool free_wrenches = false;
    for (int fm : s->free_models) free_wrenches = free_wrenches || !s->models[fm]->wrenches.empty();
    for (int it = 0; it < iterations; ++it) {
        int rc;
        if (!paused && s->d_world && (s->free_wrench_dirty || (free_wrenches && it > 0))) {
            rc = s->dtype == B2_F64 ? upload_free_wrenches<double>(s, it) : upload_free_wrenches<float>(s, it);
            if (rc != B2_OK) return rc;
        }
        if (coupled >= 0) {
            ModelState* ms = s->models[coupled].get();
            std::vector<int> wi(c_wrench_iters.size());
            for (size_t k = 0; k < wi.size(); ++k) wi[k] = c_wrench_iters[k] > it ? 1 : 0;
            const uint32_t cb = (c_bits >> it) & 1u, ctb = (c_ct_bits >> it) & 1u;
            rc = s->dtype == B2_F64 ? launch_coupled<double>(s, ms, paused, cb, ctb, wi.data())
                                    : launch_coupled<float>(s, ms, paused, cb, ctb, wi.data());
            if (!paused && ms->controller_loaded)
                for (int j = 0; j < ms->model->t.nq; ++j)
                    if (ms->mode[j] == B2_MODE_POSITION || ms->mode[j] == B2_MODE_VELOCITY) ms->has_force_cmd[j] = true;
                    else if (ms->mode[j] == B2_MODE_VELOCITY_FOLLOWER_DART) ms->has_vel_cmd[j] = true;
        } else {
            rc = s->dtype == B2_F64 ? launch_world<double>(s, paused) : launch_world<float>(s, paused);
        }
        if (rc != B2_OK) return rc;
    }
    if (coupled >= 0 && !paused) {
        const int64_t t_end = s->time_ns + (int64_t)iterations * s->dt_ns;
        auto& ws = s->models[coupled]->wrenches;
        ws.erase(std::remove_if(ws.begin(), ws.end(), [t_end](const ModelState::LinkWrench& w) { return t_end >= w.expiry_ns; }),
                 ws.end());
    }
    if (free_wrenches && !paused) {
        const int64_t t_end = s->time_ns + (int64_t)iterations * s->dt_ns;
        for (int fm : s->free_models) {
            auto& ws = s->models[fm]->wrenches;
            const size_t before = ws.size();
            ws.erase(std::remove_if(ws.begin(), ws.end(), [t_end](const ModelState::LinkWrench& w) { return t_end >= w.expiry_ns; }),
                     ws.end());
            if (ws.size() != before || !ws.empty()) s->free_wrench_dirty = true;
        }
    }
    if (!paused) s->time_ns += (int64_t)iterations * s->dt_ns;
    return B2_OK;
}

int b2sim_set_base(b2sim* s, int model, int64_t env, int velocity, const double* values)
{
    ModelState* ms = get_model(s, model);
    if (!ms || !values) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->kind != B2_KIND_FREE) return fail(B2_ERR_UNSUPPORTED, "model '%s' has a fixed base", ms->name.c_str());
    if (env < -1 || env >= s->n) return fail(B2_ERR_INVALID, "bad env index");
    DeviceGuard guard__(s->device);
    const int k0 = velocity ? 7 : 0, k1 = velocity ? 13 : 7;
    for (int k = k0; k < k1; ++k) {
        int rc = env < 0 ? col_fill_any(s, ms->buf[B2_BUF_BASE_RESET], 13, k, values[k - k0])
                         : write_elem(s, ms->buf[B2_BUF_BASE_RESET], 13, env, k, values[k - k0]);
        if (rc != B2_OK) return rc;
    }
    const uint32_t bit = velocity ? 2u : 1u;
    b2::k_or_mask<<<grid_for(env < 0 ? s->n : 1, 256), 256, 0, s->stream>>>((uint32_t*)ms->buf[B2_BUF_RESET_MASK], s->n, env, bit);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

int b2sim_base_state(b2sim* s, int model, int64_t env, double state[13])
{
    ModelState* ms = get_model(s, model);
    if (!ms || !state) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->kind != B2_KIND_FREE) return fail(B2_ERR_UNSUPPORTED, "model '%s' has a fixed base", ms->name.c_str());
    if (env < 0 || env >= s->n) return fail(B2_ERR_INVALID, "bad env index");
    DeviceGuard guard__(s->device);
    for (int k = 0; k < 13; ++k) {
        int rc = read_elem(s, ms->buf[B2_BUF_BASE_STATE], 13, env, k, &state[k]);
        if (rc != B2_OK) return rc;
    }
    return B2_OK;
}

int b2sim_contacts(b2sim* s, int64_t env, int max_contacts, int32_t* ids, double* data)
{
    if (!s) return fail(B2_ERR_INVALID, "null simulator");
    if (env < 0 || env >= s->n) return fail(B2_ERR_INVALID, "bad env index");
    if (!s->contact_count) return 0;
    DeviceGuard guard__(s->device);
    int32_t n = 0;
    B2_CUDA(cudaMemcpyAsync(&n, s->contact_count + env, sizeof n, cudaMemcpyDeviceToHost, s->stream));
    B2_CUDA(cudaStreamSynchronize(s->stream));
    if (n > max_contacts) n = max_contacts;
    if (n <= 0) return 0;
    std::vector<int32_t> raw((size_t)n * 4);
    B2_CUDA(cudaMemcpyAsync(raw.data(), s->contact_ids + (size_t)env * b2::kMaxContacts * 4, raw.size() * sizeof(int32_t),
                            cudaMemcpyDeviceToHost, s->stream));
    if (s->dtype == B2_F64) {
        B2_CUDA(cudaMemcpyAsync(data, (double*)s->contact_data + (size_t)env * b2::kMaxContacts * b2::kContactRec,
                                (size_t)n * b2::kContactRec * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
        B2_CUDA(cudaStreamSynchronize(s->stream));
    } else {
        std::vector<float> tmp((size_t)n * b2::kContactRec);
        B2_CUDA(cudaMemcpyAsync(tmp.data(), (float*)s->contact_data + (size_t)env * b2::kMaxContacts * b2::kContactRec,
                                tmp.size() * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
        B2_CUDA(cudaStreamSynchronize(s->stream));
        for (size_t k = 0; k < tmp.size(); ++k) data[k] = tmp[k];
    }
    B2_CUDA(cudaStreamSynchronize(s->stream));
    // translate world-level indices into (model, link) pairs: ids = model a, link a, model b, link b
    for (int k = 0; k < n; ++k) {
        const int a = raw[4 * k], sa = raw[4 * k + 1], b = raw[4 * k + 2];
        if (a <= b2::kRobotSide) {
            ids[4 * k] = s->robot_model;
            ids[4 * k + 1] = s->robot_shape_link[b2::kRobotSide - a];
        } else {
            const ModelState* ma = s->models[s->free_models[a]].get();
            int shape_seen = -1, link_a = 0;
            for (int q = 0; q < ma->model->t.nshapes; ++q)
                if (ma->model->t.shape_type[q] == B2_SHAPE_BOX || ma->model->t.shape_type[q] == B2_SHAPE_SPHERE)
                    if (++shape_seen == sa) link_a = ma->model->t.shape_link[q];
            ids[4 * k] = s->free_models[a];
            ids[4 * k + 1] = link_a;
        }
        if (b >= 0) {
            ids[4 * k + 2] = s->free_models[b];
            ids[4 * k + 3] = 0;
        } else if (b <= b2::kRobotSide) {
            ids[4 * k + 2] = s->robot_model;
            ids[4 * k + 3] = s->robot_shape_link[b2::kRobotSide - b];
        } else {
            ids[4 * k + 2] = s->static_shape_model[-1 - b];
            ids[4 * k + 3] = s->static_shape_link[-1 - b];
        }
    }
    return n;
}

// ---- shared joint configuration -------------------------------------------------------------------------
#define B2_JOINT_ARGS                                                                  \
    ModelState* ms = get_model(s, model);                                              \
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);               \
    if (joint < 0 || joint >= ms->model->t.nq) return fail(B2_ERR_NOT_FOUND, "joint %d not found", joint);

int b2sim_set_control_mode(b2sim* s, int model, int joint, int mode)
{
    B2_JOINT_ARGS
    DeviceGuard guard__(s->device);
    if (mode == B2_MODE_POSITION_INTERPOLATED) return fail(B2_ERR_INVALID, "PositionInterpolated not yet supported");
    if (mode <= B2_MODE_INVALID || mode > B2_MODE_POSITION_INTERPOLATED) return fail(B2_ERR_INVALID, "invalid control mode");
    if (mode == B2_MODE_POSITION || mode == B2_MODE_VELOCITY || mode == B2_MODE_VELOCITY_FOLLOWER_DART)
        ms->controller_loaded = true;  // JointController plugin inserted on demand (Joint.cpp:378-408)
    const int nq = ms->model->t.nq;
    ms->mode[joint] = mode;
    ms->has_pos_target[joint] = ms->has_vel_target[joint] = false;
    ms->has_acc_target[joint] = false;
    ms->has_vel_cmd[joint] = ms->has_force_cmd[joint] = false;
    int rc = B2_OK;
    switch (mode) {
    case B2_MODE_POSITION:
        ms->has_pos_target[joint] = true;  // target = current position (Joint.cpp:430-435)
        rc = col_copy_any(s, ms->buf[B2_BUF_POS_TARGET], nq, joint, ms->buf[B2_BUF_STATE], 2 * nq, joint);
        break;
    case B2_MODE_VELOCITY:
    case B2_MODE_VELOCITY_FOLLOWER_DART:
        ms->has_vel_target[joint] = true;
        rc = col_copy_any(s, ms->buf[B2_BUF_VEL_TARGET], nq, joint, ms->buf[B2_BUF_STATE], 2 * nq, nq + joint);
        break;
    default:
        ms->has_force_cmd[joint] = true;   // JointForceCmd = 0 (Joint.cpp:443-448)
        rc = col_fill_any(s, ms->buf[B2_BUF_FORCE_CMD], nq, joint, 0.0);
        break;
    }
    if (rc != B2_OK) return rc;
    for (int k = 0; k < 3; ++k) {  // pid.Reset() (Joint.cpp:454-457)
        rc = col_fill_any(s, ms->buf[B2_BUF_PID_STATE], 3 * nq, 3 * joint + k, 0.0);
        if (rc != B2_OK) return rc;
    }
    return B2_OK;
}
int b2sim_control_mode(const b2sim* s, int model, int joint)
{
    B2_JOINT_ARGS
    return ms->mode[joint];
}
int b2sim_set_pid(b2sim* s, int model, int joint, const b2_pid* pid)
{
    B2_JOINT_ARGS
    if (!pid) return fail(B2_ERR_INVALID, "null pid");
    b2_pid p = *pid;
    const double fmax = ms->effort[joint];
    if (p.cmd_min < -fmax || p.cmd_max > fmax) {  // Joint.cpp:503-513
        p.cmd_min = -fmax;
        p.cmd_max = fmax;
    }
    ms->pid[joint] = p;
    return B2_OK;
}
int b2sim_pid(const b2sim* s, int model, int joint, b2_pid* pid)
{
    B2_JOINT_ARGS
    if (!pid) return fail(B2_ERR_INVALID, "null pid");
    *pid = ms->pid[joint];
    return B2_OK;
}
int b2sim_set_controller_period(b2sim* s, int model, double period)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (!(period > 0)) return fail(B2_ERR_INVALID, "the controller period must be positive");
    ms->period_ns = to_ns(period);
    return B2_OK;
}
double b2sim_controller_period(const b2sim* s, int model)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return -1.0;
    return (double)ms->period_ns / 1e9;
}
int b2sim_set_max_generalized_force(b2sim* s, int model, int joint, double f)
{
    B2_JOINT_ARGS
    if (f < 0) return fail(B2_ERR_INVALID, "negative force limit");
    DeviceGuard guard__(s->device);
    ms->effort[joint] = f;
    return s->dtype == B2_F64 ? upload_tables<double>(s, ms) : upload_tables<float>(s, ms);
}

int b2sim_set_joint_friction(b2sim* s, int model, int joint, double coulomb, double viscous)
{
    B2_JOINT_ARGS
    DeviceGuard guard__(s->device);
    if (coulomb >= 0) ms->model->t.friction[joint] = coulomb;  // negative: leave unchanged
    if (viscous >= 0) ms->model->t.damping[joint] = viscous;
    if (ms->env_params) {  // "every env": the per-env rows follow
        int rc = B2_OK;
        if (viscous >= 0) rc = col_fill_any(s, ms->buf[B2_BUF_JOINT_DYNAMICS], b2::kEnvJointCols * ms->model->t.nq,
                                            b2::kEnvJointCols * joint, viscous);
        if (rc == B2_OK && coulomb >= 0)
            rc = col_fill_any(s, ms->buf[B2_BUF_JOINT_DYNAMICS], b2::kEnvJointCols * ms->model->t.nq, b2::kEnvJointCols * joint + 1,
                              coulomb);
        if (rc != B2_OK) return rc;
    }
    return refresh_tables(s, ms);  // the closed-form fit depends on the damping; Coulomb friction needs the tree path
}

int b2sim_set_computed_torque(b2sim* s, int model, const double* kp, const double* kd, const double gravity[3])
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    const int nq = ms->model->t.nq;
    if (nq == 0 || ms->kind == B2_KIND_FREE) return fail(B2_ERR_UNSUPPORTED, "the controller needs a fixed-base articulated model");
    if (!kp) {  // unload: ComputedTorqueFixedBase::terminate
        ms->ct_loaded = false;
        return B2_OK;
    }
    if (!kd) return fail(B2_ERR_INVALID, "null kd");
    for (int j = 0; j < nq; ++j) {
        ms->ct_kp[j] = kp[j];
        ms->ct_kd[j] = kd[j];
        int rc = b2sim_set_control_mode(s, model, j, B2_MODE_FORCE);  // ComputedTorqueFixedBase.cpp:180-188
        if (rc != B2_OK) return rc;
    }
    if (gravity)
        for (int k = 0; k < 3; ++k) ms->ct_gravity[k] = gravity[k];
    ms->ct_loaded = true;
    ms->ct_prev_update_ns = 0;
    // the applied torque lives in the PID command slot: clear it
    DeviceGuard guard__(s->device);
    B2_CUDA(cudaMemsetAsync(ms->buf[B2_BUF_PID_STATE], 0, (size_t)s->n * 3 * nq * s->esize(), s->stream));
    return B2_OK;
}

int b2sim_apply_link_wrench(b2sim* s, int model, int64_t env, int link, const double wrench[6], double duration)
{
    ModelState* ms = get_model(s, model);
    if (!ms || !wrench) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (link < 0 || link >= ms->model->t.nlinks) return fail(B2_ERR_NOT_FOUND, "link %d not found", link);
    if (env < -1 || env >= s->n || duration < 0) return fail(B2_ERR_INVALID, "bad env index or duration");
    if (ms->kind == B2_KIND_FREE) {
        // the force acts at the link origin: links lumped into the body at an offset would need the per-env orientation
        const double* lp = ms->model->t.link_p[link];
        if (lp[0] != 0 || lp[1] != 0 || lp[2] != 0)
            return fail(B2_ERR_UNSUPPORTED, "wrenches on free bodies are applied at the root link");
        if (!ms->wrenches.empty()) return fail(B2_ERR_UNSUPPORTED, "one external wrench per free body at a time");
        s->free_wrench_dirty = true;
    } else {
        if (ms->model->t.nq == 0) return fail(B2_ERR_UNSUPPORTED, "link wrenches need a free or an articulated model");
        if (ms->wrenches.size() >= 4) return fail(B2_ERR_UNSUPPORTED, "at most 4 concurrent link wrenches per model");
    }
    ModelState::LinkWrench w;
    w.link = link;
    w.env = env;
    for (int k = 0; k < 6; ++k) w.w[k] = wrench[k];
    w.expiry_ns = s->time_ns + to_ns(duration);
    ms->wrenches.push_back(w);
    return B2_OK;
}

// ---- per-env scalar access ---------------------------------------------------------------------------------
int b2sim_get_joint(b2sim* s, int model, int field, int64_t env, int joint, double* value)
{
    B2_JOINT_ARGS
    if (!value || env < 0 || env >= s->n) return fail(B2_ERR_INVALID, "bad env index or null output");
    DeviceGuard guard__(s->device);
    const int nq = ms->model->t.nq;
    switch (field) {
    case B2_FIELD_POSITION: return read_elem(s, ms->buf[B2_BUF_STATE], 2 * nq, env, joint, value);
    case B2_FIELD_VELOCITY: return read_elem(s, ms->buf[B2_BUF_STATE], 2 * nq, env, nq + joint, value);
    case B2_FIELD_ACCELERATION: return read_elem(s, ms->buf[B2_BUF_ACCELERATION], nq, env, joint, value);
    case B2_FIELD_FORCE: return read_elem(s, ms->force_read, nq, env, joint, value);
    case B2_FIELD_FORCE_TARGET:
        if (!ms->has_force_cmd[joint]) return fail(B2_ERR_UNSET, "no force target was set");
        return read_elem(s, ms->buf[B2_BUF_FORCE_CMD], nq, env, joint, value);
    case B2_FIELD_POSITION_TARGET:
        if (!ms->has_pos_target[joint]) return fail(B2_ERR_UNSET, "no position target was set");
        return read_elem(s, ms->buf[B2_BUF_POS_TARGET], nq, env, joint, value);
    case B2_FIELD_VELOCITY_TARGET:
        if (!ms->has_vel_target[joint]) return fail(B2_ERR_UNSET, "no velocity target was set");
        return read_elem(s, ms->buf[B2_BUF_VEL_TARGET], nq, env, joint, value);
    case B2_FIELD_ACCELERATION_TARGET:
        if (!ms->has_acc_target[joint]) return fail(B2_ERR_UNSET, "no acceleration target was set");
        return read_elem(s, ms->buf[B2_BUF_ACC_TARGET], nq, env, joint, value);
    default: return fail(B2_ERR_INVALID, "field %d is not readable", field);
    }
}

int b2sim_set_joint(b2sim* s, int model, int field, int64_t env, int joint, double value)
{
    B2_JOINT_ARGS
    if (env < -1 || env >= s->n) return fail(B2_ERR_INVALID, "bad env index");  // -1 = every env
    DeviceGuard guard__(s->device);
    const int nq = ms->model->t.nq;
    const int md = ms->mode[joint];
    switch (field) {
    case B2_FIELD_FORCE_TARGET:  // Joint.cpp:774-815
        if (!(md == B2_MODE_FORCE || md == B2_MODE_POSITION || md == B2_MODE_POSITION_INTERPOLATED ||
              md == B2_MODE_VELOCITY))
            return fail(B2_ERR_INVALID, "the active joint control mode does not accept a force target");
        ms->has_force_cmd[joint] = true;
        return env < 0 ? col_fill_any(s, ms->buf[B2_BUF_FORCE_CMD], nq, joint, value)
                       : write_elem(s, ms->buf[B2_BUF_FORCE_CMD], nq, env, joint, value);
    case B2_FIELD_POSITION_TARGET:  // Joint.cpp:683-729
        if (!(md == B2_MODE_POSITION || md == B2_MODE_POSITION_INTERPOLATED || md == B2_MODE_IDLE ||
              md == B2_MODE_FORCE))
            return fail(B2_ERR_INVALID, "the active joint control mode does not accept a position target");
        if (!ms->has_pos_target[joint] && env >= 0) {  // component created for every env: seed the rest with 0
            int rc = col_fill_any(s, ms->buf[B2_BUF_POS_TARGET], nq, joint, 0.0);
            if (rc != B2_OK) return rc;
        }
        ms->has_pos_target[joint] = true;
        return env < 0 ? col_fill_any(s, ms->buf[B2_BUF_POS_TARGET], nq, joint, value)
                       : write_elem(s, ms->buf[B2_BUF_POS_TARGET], nq, env, joint, value);
    case B2_FIELD_VELOCITY_TARGET:  // Joint.cpp:731-772
        if (!(md == B2_MODE_POSITION_INTERPOLATED || md == B2_MODE_VELOCITY ||
              md == B2_MODE_VELOCITY_FOLLOWER_DART || md == B2_MODE_IDLE || md == B2_MODE_FORCE))
            return fail(B2_ERR_INVALID, "the active joint control mode does not accept a velocity target");
        if (!ms->has_vel_target[joint] && env >= 0) {
            int rc = col_fill_any(s, ms->buf[B2_BUF_VEL_TARGET], nq, joint, 0.0);
            if (rc != B2_OK) return rc;
        }
        ms->has_vel_target[joint] = true;
        return env < 0 ? col_fill_any(s, ms->buf[B2_BUF_VEL_TARGET], nq, joint, value)
                       : write_elem(s, ms->buf[B2_BUF_VEL_TARGET], nq, env, joint, value);
    case B2_FIELD_ACCELERATION_TARGET:  // Joint.cpp:731-772
        if (!(md == B2_MODE_POSITION_INTERPOLATED || md == B2_MODE_IDLE || md == B2_MODE_FORCE))
            return fail(B2_ERR_INVALID, "the active joint control mode does not accept an acceleration target");
        if (!ms->has_acc_target[joint] && env >= 0) {
            int rc = col_fill_any(s, ms->buf[B2_BUF_ACC_TARGET], nq, joint, 0.0);
            if (rc != B2_OK) return rc;
        }
        ms->has_acc_target[joint] = true;
        return env < 0 ? col_fill_any(s, ms->buf[B2_BUF_ACC_TARGET], nq, joint, value)
                       : write_elem(s, ms->buf[B2_BUF_ACC_TARGET], nq, env, joint, value);
    case B2_FIELD_POSITION_RESET:
    case B2_FIELD_VELOCITY_RESET: {
        const int is_vel = field == B2_FIELD_VELOCITY_RESET;
        const int64_t count = env < 0 ? s->n : 1;
        if (s->dtype == B2_F64)
            b2::k_set_reset<double><<<grid_for(count, 256), 256, 0, s->stream>>>(
                (double*)ms->buf[B2_BUF_RESET_STATE], (uint32_t*)ms->buf[B2_BUF_RESET_MASK],
                (double*)ms->buf[B2_BUF_PID_STATE], s->n, nq, env, joint, is_vel, value);
        else
            b2::k_set_reset<float><<<grid_for(count, 256), 256, 0, s->stream>>>(
                (float*)ms->buf[B2_BUF_RESET_STATE], (uint32_t*)ms->buf[B2_BUF_RESET_MASK],
                (float*)ms->buf[B2_BUF_PID_STATE], s->n, nq, env, joint, is_vel, (float)value);
        ++s->launches;
        B2_CUDA(cudaGetLastError());
        return B2_OK;
    }
    default: return fail(B2_ERR_INVALID, "field %d is not writable", field);
    }
}

// ---- kinematics ----------------------------------------------------------------------------------------------
int b2sim_update_kinematics(b2sim* s, int model)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->model->t.nq == 0) return fail(B2_ERR_UNSUPPORTED, "static models have no per-env kinematics");
    DeviceGuard guard__(s->device);
    int rc = ensure_buffer(s, ms, B2_BUF_LINK_POSE);
    if (rc != B2_OK) return rc;
    return s->dtype == B2_F64 ? launch_kinematics<double>(s, ms) : launch_kinematics<float>(s, ms);
}

int b2sim_link_pose(b2sim* s, int model, int64_t env, int link, double pose[7])
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (link < 0 || link >= ms->model->t.nlinks || !pose || env < 0 || env >= s->n)
        return fail(B2_ERR_NOT_FOUND, "link %d not found", link);
    if (ms->model->t.nq == 0) {
        // static model: every link sits at base * offset; free body: at its per-env base pose * offset
        const b2_model_tables& t = ms->model->t;
        b2::Pose base = ms->base;
        if (ms->kind == B2_KIND_FREE) {
            double st[13];
            int rc = b2sim_base_state(s, model, env, st);
            if (rc != B2_OK) return rc;
            base = b2::pose_from_xyz_quat(st);
        }
        b2::Pose off;
        for (int k = 0; k < 9; ++k) off.R.m[k] = t.link_R[link][k];
        off.p = {t.link_p[link][0], t.link_p[link][1], t.link_p[link][2]};
        b2::Pose w = b2::compose(base, off);
        pose[0] = w.p.x; pose[1] = w.p.y; pose[2] = w.p.z;
        b2::rot_to_quat(w.R, pose + 3);
        return B2_OK;
    }
    int rc = b2sim_update_kinematics(s, model);
    if (rc != B2_OK) return rc;
    const int64_t cols = 7 * ms->model->t.nlinks;
    for (int k = 0; k < 7; ++k) {
        rc = read_elem(s, ms->buf[B2_BUF_LINK_POSE], cols, env, 7 * link + k, &pose[k]);
        if (rc != B2_OK) return rc;
    }
    return B2_OK;
}

int b2sim_kindyn(b2sim* s, int model, int link, void* mass_matrix, void* bias_forces, void* jacobian)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->model->t.nq == 0) return fail(B2_ERR_UNSUPPORTED, "static model");
    if (jacobian && (link < 0 || link >= ms->model->t.nlinks)) return fail(B2_ERR_NOT_FOUND, "link %d not found", link);
    DeviceGuard guard__(s->device);
    return s->dtype == B2_F64 ? launch_kindyn<double>(s, ms, link, mass_matrix, bias_forces, jacobian)
                              : launch_kindyn<float>(s, ms, link, mass_matrix, bias_forces, jacobian);
}

int b2sim_link_motion(b2sim* s, int model, int link, void* twist, void* acceleration)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->model->t.nq == 0) return fail(B2_ERR_UNSUPPORTED, "link motion queries need an articulated fixed-base model");
    if (link < 0 || link >= ms->model->t.nlinks) return fail(B2_ERR_NOT_FOUND, "link %d not found", link);
    DeviceGuard guard__(s->device);
    return s->dtype == B2_F64 ? launch_link_motion<double>(s, ms, link, twist, acceleration)
                              : launch_link_motion<float>(s, ms, link, twist, acceleration);
}

int b2sim_centroidal(b2sim* s, int model, void* com, void* com_velocity, void* momentum, void* com_jacobian)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    const int nq = ms->model->t.nq;
    if (nq == 0) return fail(B2_ERR_UNSUPPORTED, "model '%s' has no joints", ms->name.c_str());
    DeviceGuard guard__(s->device);
    const int block = 128, grid = grid_for(s->n, block);
    if (s->dtype == B2_F64)
        b2::k_centroidal<double, b2::kMaxDofs><<<grid, block, 0, s->stream>>>(
            (const b2::ModelDev<double>*)ms->d_tables, (const double*)ms->buf[B2_BUF_STATE], (double*)com,
            (double*)com_velocity, (double*)momentum, (double*)com_jacobian, s->n);
    else
        b2::k_centroidal<float, b2::kMaxDofs><<<grid, block, 0, s->stream>>>(
            (const b2::ModelDev<float>*)ms->d_tables, (const float*)ms->buf[B2_BUF_STATE], (float*)com,
            (float*)com_velocity, (float*)momentum, (float*)com_jacobian, s->n);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

int b2sim_momentum_jacobian(b2sim* s, int model, void* momentum_jacobian, void* locked_inertia)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    const int nq = ms->model->t.nq;
    if (nq == 0) return fail(B2_ERR_UNSUPPORTED, "model '%s' has no joints", ms->name.c_str());
    DeviceGuard guard__(s->device);
    const int block = 128, grid = grid_for(s->n, block);
    if (s->dtype == B2_F64)
        b2::k_momentum<double, b2::kMaxDofs><<<grid, block, 0, s->stream>>>(
            (const b2::ModelDev<double>*)ms->d_tables, (const double*)ms->buf[B2_BUF_STATE], (double*)momentum_jacobian,
            (double*)locked_inertia, s->n);
    else
        b2::k_momentum<float, b2::kMaxDofs><<<grid, block, 0, s->stream>>>(
            (const b2::ModelDev<float>*)ms->d_tables, (const float*)ms->buf[B2_BUF_STATE], (float*)momentum_jacobian,
            (float*)locked_inertia, s->n);
    ++s->launches;
    B2_CUDA(cudaGetLastError());
    return B2_OK;
}

// ---- per-env physical parameters ----------------------------------------------------------------------------------
int b2sim_enable_env_params(b2sim* s, int model, int enable)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    DeviceGuard guard__(s->device);
    const int bufs[3] = {B2_BUF_BODY_INERTIA, B2_BUF_JOINT_DYNAMICS, B2_BUF_GRAVITY};
    if (!enable) {
        if (ms->env_params) B2_CUDA(cudaStreamSynchronize(s->stream));  // runs still queued read the rows
        for (int which : bufs)
            if (ms->buf[which]) { cudaFree(ms->buf[which]); ms->buf[which] = nullptr; }
        ms->env_params = false;
        return B2_OK;
    }
    const b2_model_tables& t = ms->model->t;
    const int nq = t.nq;
    if (nq == 0 || ms->kind == B2_KIND_FREE || ms->kind == B2_KIND_STATIC)
        return fail(B2_ERR_UNSUPPORTED, "model '%s' is not a fixed-base articulated model", ms->name.c_str());
    if (ms->task != B2_TASK_NONE && ms->task != B2_TASK_PANDA_REACH)
        return fail(B2_ERR_UNSUPPORTED, "model '%s' has a pendulum / cart-pole task, whose kernels read the shared tables only",
                    ms->name.c_str());
    for (auto& other : s->models)
        if (!other->removed && other->kind == B2_KIND_FREE)
            return fail(B2_ERR_UNSUPPORTED, "the world has free bodies: the coupled contact pipeline has no per-env parameters");
    if (ms->env_params) return B2_OK;
    ms->env_params = true;
    int rc = B2_OK;
    for (int which : bufs)
        if (rc == B2_OK) rc = ensure_buffer(s, ms, which);
    // every row starts from the model's current values: loader tables, set_joint_friction edits, world gravity
    const int sym[6] = {0, 1, 2, 4, 5, 8};
    for (int b = 0; b < nq && rc == B2_OK; ++b) {
        double v[b2::kEnvInertiaCols] = {t.mass[b], t.com[b][0], t.com[b][1], t.com[b][2]};
        for (int k = 0; k < 6; ++k) v[4 + k] = t.Ic[b][sym[k]];
        for (int k = 0; k < b2::kEnvInertiaCols && rc == B2_OK; ++k)
            rc = col_fill_any(s, ms->buf[B2_BUF_BODY_INERTIA], b2::kEnvInertiaCols * nq, b2::kEnvInertiaCols * b + k, v[k]);
        if (rc == B2_OK) rc = col_fill_any(s, ms->buf[B2_BUF_JOINT_DYNAMICS], b2::kEnvJointCols * nq, b2::kEnvJointCols * b, t.damping[b]);
        if (rc == B2_OK)
            rc = col_fill_any(s, ms->buf[B2_BUF_JOINT_DYNAMICS], b2::kEnvJointCols * nq, b2::kEnvJointCols * b + 1, t.friction[b]);
    }
    for (int k = 0; k < 3 && rc == B2_OK; ++k) rc = col_fill_any(s, ms->buf[B2_BUF_GRAVITY], 3, k, s->gravity[k]);
    if (rc != B2_OK) {
        std::string msg = g_error;
        b2sim_enable_env_params(s, model, 0);
        return fail(rc, "%s", msg.c_str());
    }
    return B2_OK;
}

int b2sim_enable_free_body_params(b2sim* s, int model, int enable, b2_buffer* out)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    DeviceGuard guard__(s->device);
    if (enable && ms->kind != B2_KIND_FREE)
        return fail(B2_ERR_UNSUPPORTED, "model '%s' is not a free-floating body", ms->name.c_str());
    const b2_model_tables& t = ms->model->t;
    double init[b2::kFreeBodyCols] = {t.body_mass, t.body_com[0], t.body_com[1], t.body_com[2]};
    const int sym[6] = {0, 1, 2, 4, 5, 8};
    for (int k = 0; k < 6; ++k) init[4 + k] = t.body_Ic[sym[k]];
    return enable_rows(s, ms->body_rows, enable, b2::kFreeBodyCols, init, out);
}

int b2sim_enable_shape_friction(b2sim* s, int model, int enable, b2_buffer* out)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    DeviceGuard guard__(s->device);
    const b2_model_tables& t = ms->model->t;
    if (enable && t.nshapes == 0) return fail(B2_ERR_UNSUPPORTED, "model '%s' has no collision shape", ms->name.c_str());
    return enable_rows(s, ms->mu_rows, enable, t.nshapes, t.shape_mu, out);
}

// ---- zero-copy view --------------------------------------------------------------------------------------------
int b2sim_buffer(b2sim* s, int model, int which, b2_buffer* out)
{
    ModelState* ms = get_model(s, model);
    if (!ms || !out) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (which < 0 || which >= B2_BUF_COUNT) return fail(B2_ERR_INVALID, "unknown buffer %d", which);
    DeviceGuard guard__(s->device);
    int rc = ensure_buffer(s, ms, which);
    if (rc != B2_OK) return rc;
    int64_t cols;
    int dtype, itemsize;
    buffer_shape(s, ms, which, &cols, &dtype, &itemsize);
    if (!ms->buf[which]) return fail(B2_ERR_UNSET, "buffer %d is empty for this model (no task attached?)", which);
    out->ptr = ms->buf[which];
    out->rows = s->n;
    out->cols = cols;
    out->dtype = dtype;
    out->itemsize = itemsize;
    return B2_OK;
}

// ---- fused task path ----------------------------------------------------------------------------------------------
int b2sim_task_nobs(int task)
{
    switch (task) {
    case B2_TASK_PENDULUM_SWINGUP: return 3;
    case B2_TASK_CARTPOLE_DISCRETE_BALANCING:
    case B2_TASK_CARTPOLE_CONTINUOUS_BALANCING:
    case B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP: return 4;
    case B2_TASK_PANDA_REACH: return b2::panda_obs_size(9);
    default: return 0;
    }
}
int b2sim_task_nact(int task) { return task == B2_TASK_PANDA_REACH ? 9 : (b2sim_task_nobs(task) > 0 ? 1 : 0); }

int b2sim_set_task(b2sim* s, int model, int task, uint64_t seed, uint64_t env_offset, int max_episode_steps)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (b2sim_task_nobs(task) == 0) return fail(B2_ERR_UNSUPPORTED, "unknown task %d", task);
    if (max_episode_steps <= 0 || max_episode_steps > 65535) return fail(B2_ERR_INVALID, "max_episode_steps out of range");
    if (ms->env_params && task != B2_TASK_PANDA_REACH)
        return fail(B2_ERR_UNSUPPORTED, "model '%s' has per-env parameters: the pendulum / cart-pole task kernels read the shared "
                                        "tables only", ms->name.c_str());
    DeviceGuard guard__(s->device);
    const b2_model_tables& t = ms->model->t;
    if (task == B2_TASK_PANDA_REACH) {
        if (t.nq < 1) return fail(B2_ERR_UNSUPPORTED, "the reach task needs an articulated model");
        b2::TreeTopo topo;
        int rc = tree_topology(ms, &topo);
        if (rc != B2_OK) return rc;
        ms->task = task;
        ms->seed = seed;
        ms->env_offset = env_offset;
        ms->max_episode_steps = max_episode_steps;
        ms->task_steps = 0;
        ms->task_ee_link = t.nlinks - 1;
        for (size_t l = 0; l < ms->model->link_names.size(); ++l)
            if (ms->model->link_names[l] == "end_effector_frame") ms->task_ee_link = (int)l;
        for (int which : {B2_BUF_OBS, B2_BUF_REWARD, B2_BUF_DONE, B2_BUF_ELAPSED, B2_BUF_ACTION}) {
            if (ms->buf[which]) { cudaFree(ms->buf[which]); ms->buf[which] = nullptr; }
            rc = ensure_buffer(s, ms, which);
            if (rc != B2_OK) return rc;
        }
        // position PID on every joint, controller period = physics step (test_pid_controllers.py:69)
        for (int j = 0; j < t.nq; ++j) {
            rc = b2sim_set_control_mode(s, model, j, B2_MODE_POSITION);
            if (rc != B2_OK) return rc;
        }
        ms->period_ns = s->dt_ns;
        return b2sim_task_reset_all(s, model);
    }
    const bool pendulum = task == B2_TASK_PENDULUM_SWINGUP;
    if (pendulum && ms->kind != B2_KIND_CHAIN1)
        return fail(B2_ERR_UNSUPPORTED, "the pendulum task needs a single-joint model");
    if (!pendulum && ms->kind != B2_KIND_CHAIN_PR)
        return fail(B2_ERR_UNSUPPORTED, "the cartpole tasks need a prismatic->revolute chain");
    // the closed forms skip the joint-limit constraint: the cart must terminate (|x| > 2.4) before the rail ends
    if (!pendulum && !(t.lower[0] < -2.5 && t.upper[0] > 2.5))
        return fail(B2_ERR_UNSUPPORTED, "cart travel limits must lie outside the task termination bound");
    if (!std::isinf(t.lower[pendulum ? 0 : 1]) || !std::isinf(t.upper[pendulum ? 0 : 1]))
        return fail(B2_ERR_UNSUPPORTED, "the pivot joint must be continuous");
    // the closed forms have no constraint stage: Coulomb friction (a JointCoulombFriction row in DART) cannot be honoured
    for (int j = 0; j < t.nq; ++j)
        if (t.friction[j] != 0.0)
            return fail(B2_ERR_UNSUPPORTED, "joint %d has Coulomb friction: the fused task kernels do not model it "
                                            "(step the model through b2sim_run instead)", j);
    ms->task = task;
    ms->seed = seed;
    ms->env_offset = env_offset;
    ms->max_episode_steps = max_episode_steps;
    ms->task_steps = 0;
    for (int which : {B2_BUF_OBS, B2_BUF_REWARD, B2_BUF_DONE, B2_BUF_ELAPSED, B2_BUF_ACTION}) {
        if (ms->buf[which]) { cudaFree(ms->buf[which]); ms->buf[which] = nullptr; }
        int rc = ensure_buffer(s, ms, which);
        if (rc != B2_OK) return rc;
    }
    if (!ms->d_step) {
        B2_CUDA(cudaMalloc(&ms->d_step, sizeof(unsigned long long)));
        B2_CUDA(cudaMalloc(&ms->d_ticket, b2::kTicketWords * sizeof(unsigned int)));
    }
    {
        const unsigned long long first = 1;  // Philox step index of the first step; 0 is the initial reset
        B2_CUDA(cudaMemcpyAsync(ms->d_step, &first, sizeof first, cudaMemcpyHostToDevice, s->stream));
        B2_CUDA(cudaMemsetAsync(ms->d_ticket, 0, b2::kTicketWords * sizeof(unsigned int), s->stream));
        B2_CUDA(cudaStreamSynchronize(s->stream));
    }
    // Task.reset_task puts the actuated joint in Force mode (cartpole_*.py:133-135)
    int rc = b2sim_set_control_mode(s, model, 0, B2_MODE_FORCE);
    if (rc != B2_OK) return rc;
    return b2sim_task_reset_all(s, model);
}

int b2sim_task_reset_all(b2sim* s, int model)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->task == B2_TASK_NONE) return fail(B2_ERR_UNSET, "no task attached");
    DeviceGuard guard__(s->device);
    if (ms->d_ep_totals)  // unfinished episodes are dropped from the statistics, the totals stay
        B2_CUDA(cudaMemsetAsync(ms->buf[B2_BUF_EP_RETURN], 0, (size_t)s->n * s->esize(), s->stream));
    if (ms->task == B2_TASK_PANDA_REACH) {
        // models/panda.py:42-44 initial configuration, zero velocity, PID reset, targets = q0
        const int nq = ms->model->t.nq;
        for (int j = 0; j < nq; ++j) {
            int rc = col_fill_any(s, ms->buf[B2_BUF_STATE], 2 * nq, j, ms->task_q0[j]);
            if (rc == B2_OK) rc = col_fill_any(s, ms->buf[B2_BUF_STATE], 2 * nq, nq + j, 0.0);
            if (rc == B2_OK) rc = col_fill_any(s, ms->buf[B2_BUF_POS_TARGET], nq, j, ms->task_q0[j]);
            if (rc != B2_OK) return rc;
        }
        B2_CUDA(cudaMemsetAsync(ms->buf[B2_BUF_PID_STATE], 0, (size_t)s->n * 3 * nq * s->esize(), s->stream));
        B2_CUDA(cudaMemsetAsync(ms->buf[B2_BUF_ELAPSED], 0, (size_t)s->n * 2, s->stream));
        return B2_OK;
    }
    return s->dtype == B2_F64 ? dispatch_reset_all<double>(s, ms) : dispatch_reset_all<float>(s, ms);
}

int b2sim_set_task_randomization(b2sim* s, int model, double mass_delta, double gravity_sigma)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->task == B2_TASK_NONE || ms->task == B2_TASK_PANDA_REACH)
        return fail(B2_ERR_UNSUPPORTED, "domain randomisation is available for the pendulum and cart-pole tasks");
    if (mass_delta < 0 || gravity_sigma < 0) return fail(B2_ERR_INVALID, "negative randomisation range");
    if (s->gravity[0] != 0 || s->gravity[1] != 0 || s->gravity[2] == 0)
        return fail(B2_ERR_UNSUPPORTED, "gravity randomisation needs a world gravity along z");
    DeviceGuard guard__(s->device);
    if (ms->buf[B2_BUF_RAND_PARAMS]) {
        B2_CUDA(cudaStreamSynchronize(s->stream));
        cudaFree(ms->buf[B2_BUF_RAND_PARAMS]);
        ms->buf[B2_BUF_RAND_PARAMS] = nullptr;
    }
    ms->rand_mass_delta = mass_delta;
    ms->rand_gravity_sigma = gravity_sigma;
    if (mass_delta != 0 || gravity_sigma != 0) {
        int rc = ensure_buffer(s, ms, B2_BUF_RAND_PARAMS);
        if (rc != B2_OK) return rc;
    }
    return b2sim_task_reset_all(s, model);
}

int b2sim_set_task_params(b2sim* s, int model, const double* goal, const double* q0, int ee_link)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (goal)
        for (int k = 0; k < 3; ++k) ms->task_goal[k] = goal[k];
    if (q0)
        for (int j = 0; j < ms->model->t.nq; ++j) ms->task_q0[j] = q0[j];
    if (ee_link >= 0) {
        if (ee_link >= ms->model->t.nlinks) return fail(B2_ERR_NOT_FOUND, "link %d not found", ee_link);
        ms->task_ee_link = ee_link;
    }
    return B2_OK;
}

int b2sim_task_observe(b2sim* s, int model)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->task == B2_TASK_NONE) return fail(B2_ERR_UNSET, "no task attached");
    DeviceGuard guard__(s->device);
    return s->dtype == B2_F64 ? dispatch_observe<double>(s, ms) : dispatch_observe<float>(s, ms);
}

int b2sim_task_step(b2sim* s, int model, const void* actions_dev)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->task == B2_TASK_NONE) return fail(B2_ERR_UNSET, "no task attached");
    if (!actions_dev) return fail(B2_ERR_INVALID, "null actions");
    DeviceGuard guard__(s->device);
    int rc = s->dtype == B2_F64 ? dispatch_task<double>(s, ms, actions_dev) : dispatch_task<float>(s, ms, actions_dev);
    if (rc != B2_OK) return rc;
    ms->task_steps += 1;
    s->time_ns += (int64_t)s->steps_per_run * s->dt_ns;
    return B2_OK;
}

int b2sim_task_rollout(b2sim* s, int model, const void* actions_dev, int steps, int64_t action_stride)
{
    if (steps <= 0) return fail(B2_ERR_INVALID, "steps must be positive");
    const size_t es = s ? s->esize() : 8;
    for (int t = 0; t < steps; ++t) {
        int rc = b2sim_task_step(s, model, (const char*)actions_dev + (size_t)t * (size_t)action_stride * es);
        if (rc != B2_OK) return rc;
    }
    return B2_OK;
}

int b2sim_task_trajectory(b2sim* s, int model, const void* actions_dev, int steps, void* obs_traj, void* reward_traj,
                          uint8_t* done_traj)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->task == B2_TASK_NONE) return fail(B2_ERR_UNSET, "no task attached");
    if (!actions_dev) return fail(B2_ERR_INVALID, "null actions");
    if (steps <= 0) return fail(B2_ERR_INVALID, "steps must be positive");
    if ((obs_traj != nullptr) != (reward_traj != nullptr) || (obs_traj != nullptr) != (done_traj != nullptr))
        return fail(B2_ERR_INVALID, "pass all three trajectory outputs or none");
    DeviceGuard guard__(s->device);
    int rc = s->dtype == B2_F64 ? dispatch_task<double>(s, ms, actions_dev, steps, obs_traj, reward_traj, done_traj)
                                : dispatch_task<float>(s, ms, actions_dev, steps, obs_traj, reward_traj, done_traj);
    if (rc != B2_OK) return rc;
    ms->task_steps += 1;
    s->time_ns += (int64_t)steps * s->steps_per_run * s->dt_ns;
    return B2_OK;
}

int b2sim_task_step_host(b2sim* s, int model, const void* actions_host, void* obs_host, void* reward_host,
                         uint8_t* done_host)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->task == B2_TASK_NONE) return fail(B2_ERR_UNSET, "no task attached");
    if (!actions_host) return fail(B2_ERR_INVALID, "null actions");
    DeviceGuard guard__(s->device);
    const bool panda = ms->task == B2_TASK_PANDA_REACH;
    const size_t es = s->esize();
    const size_t nobs = panda ? (size_t)b2::panda_obs_size(ms->model->t.nq) : (size_t)b2sim_task_nobs(ms->task);
    const size_t nact = panda ? (size_t)ms->model->t.nq : 1;
    // The env range is cut into chunks; chunk c's actions go host->device on one stream while chunk c-1 is stepped
    // and chunk c-2's outputs go device->host on another, so the two PCIe directions and the kernels overlap.
    // Measured at 4,194,304 envs: 2 / 4 / 8 / 16 / 32 chunks -> 1.18 / 1.24 / 1.23 / 1.19 / 1.11e9 env-steps/s.
    // Letting the kernel read the actions and write the outputs straight through mapped pinned memory instead of the copy
    // engines was measured too: 4.5e8 env-steps/s (22 GB/s on the link), so the copies stay.
    const int64_t min_chunk = 65536, max_chunks = 8;
    const int chunks = (int)std::max<int64_t>(1, std::min<int64_t>(max_chunks, s->n / min_chunk));
    if (!s->copy_in) {
        B2_CUDA(cudaStreamCreateWithFlags(&s->copy_in, cudaStreamNonBlocking));
        B2_CUDA(cudaStreamCreateWithFlags(&s->copy_out, cudaStreamNonBlocking));
    }
    while ((int)s->events.size() < 2 * chunks + 1) {
        cudaEvent_t ev;
        B2_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        s->events.push_back(ev);
    }
    char* act_dev = (char*)ms->buf[B2_BUF_ACTION];
    // earlier work on the simulator stream (resets, previous steps) must be visible to the copy streams
    B2_CUDA(cudaEventRecord(s->events[2 * chunks], s->stream));
    B2_CUDA(cudaStreamWaitEvent(s->copy_in, s->events[2 * chunks], 0));
    int rc = B2_OK;
    for (int c = 0; c < chunks && rc == B2_OK; ++c) {
        const int64_t b0 = s->n * c / chunks, b1 = s->n * (c + 1) / chunks, cnt = b1 - b0;
        B2_CUDA(cudaMemcpyAsync(act_dev + (size_t)b0 * nact * es, (const char*)actions_host + (size_t)b0 * nact * es,
                                (size_t)cnt * nact * es, cudaMemcpyHostToDevice, s->copy_in));
        B2_CUDA(cudaEventRecord(s->events[2 * c], s->copy_in));
        B2_CUDA(cudaStreamWaitEvent(s->stream, s->events[2 * c], 0));
        s->win_begin = b0;
        s->win_count = cnt;
        rc = s->dtype == B2_F64 ? dispatch_task<double>(s, ms, act_dev) : dispatch_task<float>(s, ms, act_dev);
        s->win_begin = 0;
        s->win_count = -1;
        if (rc != B2_OK) break;
        B2_CUDA(cudaEventRecord(s->events[2 * c + 1], s->stream));
        B2_CUDA(cudaStreamWaitEvent(s->copy_out, s->events[2 * c + 1], 0));
        if (obs_host)
            B2_CUDA(cudaMemcpyAsync((char*)obs_host + (size_t)b0 * nobs * es, (char*)ms->buf[B2_BUF_OBS] + (size_t)b0 * nobs * es,
                                    (size_t)cnt * nobs * es, cudaMemcpyDeviceToHost, s->copy_out));
        if (reward_host)
            B2_CUDA(cudaMemcpyAsync((char*)reward_host + (size_t)b0 * es, (char*)ms->buf[B2_BUF_REWARD] + (size_t)b0 * es,
                                    (size_t)cnt * es, cudaMemcpyDeviceToHost, s->copy_out));
        if (done_host)
            B2_CUDA(cudaMemcpyAsync(done_host + b0, (uint8_t*)ms->buf[B2_BUF_DONE] + b0, (size_t)cnt, cudaMemcpyDeviceToHost,
                                    s->copy_out));
    }
    if (rc != B2_OK) return rc;
    ms->task_steps += 1;
    s->time_ns += (int64_t)s->steps_per_run * s->dt_ns;
    B2_CUDA(cudaStreamSynchronize(s->copy_out));
    B2_CUDA(cudaStreamSynchronize(s->stream));
    return B2_OK;
}

int b2sim_episode_stats_enable(b2sim* s, int model, int enable)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (ms->task == B2_TASK_NONE) return fail(B2_ERR_UNSET, "no task attached");
    DeviceGuard guard__(s->device);
    B2_CUDA(cudaStreamSynchronize(s->stream));
    if (!enable) {
        if (ms->d_ep_totals) { cudaFree(ms->d_ep_totals); ms->d_ep_totals = nullptr; }
        if (ms->buf[B2_BUF_EP_RETURN]) { cudaFree(ms->buf[B2_BUF_EP_RETURN]); ms->buf[B2_BUF_EP_RETURN] = nullptr; }
        return B2_OK;
    }
    const size_t bytes = (size_t)B2_STAT_STRIPES * 4 * sizeof(double);
    static_assert(B2_STAT_STRIPES == b2::kStatStripes, "header and kernels disagree on the stripe count");
    if (!ms->d_ep_totals) B2_CUDA(cudaMalloc(&ms->d_ep_totals, bytes));
    B2_CUDA(cudaMemsetAsync(ms->d_ep_totals, 0, bytes, s->stream));
    int rc = ensure_buffer(s, ms, B2_BUF_EP_RETURN);
    if (rc != B2_OK) return rc;
    B2_CUDA(cudaMemsetAsync(ms->buf[B2_BUF_EP_RETURN], 0, (size_t)s->n * s->esize(), s->stream));
    return B2_OK;
}

int b2sim_episode_stats_device(b2sim* s, int model, void** totals_dev)
{
    ModelState* ms = get_model(s, model);
    if (!ms || !totals_dev) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (!ms->d_ep_totals) return fail(B2_ERR_UNSET, "episode statistics are not enabled");
    *totals_dev = ms->d_ep_totals;
    return B2_OK;
}

int b2sim_episode_stats(b2sim* s, int model, double totals[4], int clear)
{
    ModelState* ms = get_model(s, model);
    if (!ms || !totals) return fail(B2_ERR_NOT_FOUND, "model %d not found", model);
    if (!ms->d_ep_totals) return fail(B2_ERR_UNSET, "episode statistics are not enabled");
    DeviceGuard guard__(s->device);
    double host[B2_STAT_STRIPES * 4];
    B2_CUDA(cudaMemcpyAsync(host, ms->d_ep_totals, sizeof host, cudaMemcpyDeviceToHost, s->stream));
    if (clear) B2_CUDA(cudaMemsetAsync(ms->d_ep_totals, 0, sizeof host, s->stream));
    B2_CUDA(cudaStreamSynchronize(s->stream));
    for (int k = 0; k < 4; ++k) totals[k] = 0.0;
    for (int r = 0; r < B2_STAT_STRIPES; ++r)
        for (int k = 0; k < 4; ++k) totals[k] += host[4 * r + k];
    return B2_OK;
}

uint64_t b2sim_task_steps_done(const b2sim* s, int model)
{
    ModelState* ms = get_model(s, model);
    if (!ms) return 0;
    if (ms->d_step) {  // the device counter also sees steps replayed from a CUDA graph
        unsigned long long next = 0;
        DeviceGuard guard__(s->device);
        if (cudaMemcpyAsync(&next, ms->d_step, sizeof next, cudaMemcpyDeviceToHost, s->stream) == cudaSuccess &&
            cudaStreamSynchronize(s->stream) == cudaSuccess && next > 0)
            return next - 1;
    }
    return ms->task_steps;
}

}  // extern "C"
