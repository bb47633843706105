// Translation unit of the lane-parallel kernels (sm_100a). See b2_lanes.cuh.
#include "b2_lanes.hpp"

#include "b2_lanes.cuh"

namespace b2 {

namespace {
// Launches a lane kernel (LaneLayout<G>) over n envs: block geometry and dynamic shared memory. `pdl`: programmatic
// dependent launch (launch_pdl). `coupled`: the kernel runs beside k_coupled_rows / k_coupled_minv.
template <typename T, int G, typename... KArgs, typename... Args>
cudaError_t launch_lanes(void (*kernel)(KArgs...), int64_t n, bool pdl, bool coupled, cudaStream_t stream, Args... args)
{
    using L = LaneLayout<G>;
    // 64-thread blocks spread small batches over more SMs (4,096 envs: 14.4 us against 16.5 us), 128-thread blocks share
    // the staged model constants among more envs (16,384 envs: 39.0 us against 39.6 us)
    const int warps = n <= 8192 ? 2 : 4;
    const int64_t envs_per_block = (int64_t)warps * L::envs_per_warp;
    const int grid = (int)((n + envs_per_block - 1) / envs_per_block);
    const size_t smem = ((size_t)envs_per_block * L::stride + L::table + 12) * sizeof(T);
    cudaError_t rc = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc != cudaSuccess) return rc;
    if (coupled) {  // must share SMs with k_coupled_rows / k_coupled_minv: the same shared-memory carve-out
        rc = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, kCoupledCarveout);
        if (rc != cudaSuccess) return rc;
    }
    return launch_pdl(kernel, grid, 32 * warps, smem, stream, pdl, args...);
}

// Calls `launch` with the ENV flag of the kernel to instantiate: std::true_type (the per-env parameter variant) while the
// model has parameter rows, env.inertia != nullptr.
template <typename T, typename F>
cudaError_t with_env_flag(const EnvRows<T>& env, F launch)
{
    return env.inertia ? launch(std::true_type()) : launch(std::false_type());
}

template <typename T, int G, int NQ, unsigned P_LO = 0u, unsigned P_HI = 0u, unsigned REV = 0u>
cudaError_t launch_panda_g(const ModelDev<T>* tables, const LaneTable<T>* lane_table, const PandaArgs<T>& a, const TreeBits& tb,
                           cudaStream_t stream, const EnvRows<T>& env)
{
    return with_env_flag(env, [&](auto env_flag) {
        return launch_lanes<T, G>(k_task_panda_lanes<T, G, NQ, P_LO, P_HI, REV, decltype(env_flag)::value>, a.n, a.n > 8192, false,
                                  stream, tables, lane_table, a, tb, env);
    });
}

template <typename T, int G>
cudaError_t launch_run_v(const ModelDev<T>* tables, const LaneTable<T>* lane_table, const RunCfg<T>& cfg, const RunBuffers<T>& b,
                         const TreeBits& tb, cudaStream_t stream, T* v0, int nvp, const EnvRows<T>& env)
{
    const bool ct = cfg.ct_active && !cfg.paused;
    // a coupled step forks three kernels from one event: no programmatic overlap with the previous step's finish
    if (v0)
        return launch_lanes<T, G>(ct ? &k_run_tree_lanes<T, G, true, true> : &k_run_tree_lanes<T, G, false, true>, b.n, false, true,
                                  stream, tables, lane_table, cfg, b, tb, v0, nvp, env);
    return with_env_flag(env, [&](auto env_flag) {
        constexpr bool ENV = decltype(env_flag)::value;
        return launch_lanes<T, G>(ct ? &k_run_tree_lanes<T, G, true, false, ENV> : &k_run_tree_lanes<T, G, false, false, ENV>, b.n,
                                  b.n > 8192, false, stream, tables, lane_table, cfg, b, tb, v0, nvp, env);
    });
}
}  // namespace

template <typename T>
cudaError_t launch_task_panda_lanes(const ModelDev<T>* tables, const LaneTable<T>* lane_table, const PandaArgs<T>& a,
                                    const int* parent, const int* jtype, cudaStream_t stream, const EnvRows<T>& env)
{
    const TreeBits tb = make_tree_bits(a.nq, parent, jtype);
    if (a.nq <= 8) return launch_panda_g<T, 8, 0>(tables, lane_table, a, tb, stream, env);
    // the Panda (a chain of 7 revolute joints, two prismatic fingers on the last arm body): tree known at compile time
    constexpr unsigned kPandaLo = 0x76543210u, kPandaHi = 0x7u, kPandaRev = 0x7fu;
    if (a.nq == 9 && tb.p_lo == kPandaLo && tb.p_hi == kPandaHi && tb.rev_mask == kPandaRev)
        return launch_panda_g<T, 10, 9, kPandaLo, kPandaHi, kPandaRev>(tables, lane_table, a, tb, stream, env);
    if (a.nq <= 10) return launch_panda_g<T, 10, 0>(tables, lane_table, a, tb, stream, env);
    return launch_panda_g<T, 16, 0>(tables, lane_table, a, tb, stream, env);
}

template <typename T>
cudaError_t launch_run_tree_lanes(const ModelDev<T>* tables, const LaneTable<T>* lane_table, const RunCfg<T>& cfg,
                                  const RunBuffers<T>& b, const int* parent, const int* jtype, cudaStream_t stream, T* v0, int nvp,
                                  const EnvRows<T>& env)
{
    if (v0 && env.inertia) return cudaErrorInvalidValue;  // no coupled variant with per-env parameters
    const TreeBits tb = make_tree_bits(cfg.nq, parent, jtype);
    if (cfg.nq <= 8) return launch_run_v<T, 8>(tables, lane_table, cfg, b, tb, stream, v0, nvp, env);
    if (cfg.nq <= 10) return launch_run_v<T, 10>(tables, lane_table, cfg, b, tb, stream, v0, nvp, env);
    return launch_run_v<T, 16>(tables, lane_table, cfg, b, tb, stream, v0, nvp, env);
}

template cudaError_t launch_run_tree_lanes<double>(const ModelDev<double>*, const LaneTable<double>*, const RunCfg<double>&,
                                                   const RunBuffers<double>&, const int*, const int*, cudaStream_t, double*, int,
                                                   const EnvRows<double>&);
template cudaError_t launch_run_tree_lanes<float>(const ModelDev<float>*, const LaneTable<float>*, const RunCfg<float>&,
                                                  const RunBuffers<float>&, const int*, const int*, cudaStream_t, float*, int,
                                                  const EnvRows<float>&);

template cudaError_t launch_task_panda_lanes<double>(const ModelDev<double>*, const LaneTable<double>*, const PandaArgs<double>&,
                                                     const int*, const int*, cudaStream_t, const EnvRows<double>&);
template cudaError_t launch_task_panda_lanes<float>(const ModelDev<float>*, const LaneTable<float>*, const PandaArgs<float>&,
                                                    const int*, const int*, cudaStream_t, const EnvRows<float>&);

}  // namespace b2
