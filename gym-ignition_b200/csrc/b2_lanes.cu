// Translation unit of the lane-parallel kernels (sm_100a). See b2_lanes.cuh.
#include "b2_lanes.hpp"

#include "b2_lanes.cuh"

namespace b2 {

namespace {
// Launch with programmatic stream serialization: consecutive steps on a stream overlap the tail of one launch with the
// scheduling and model staging of the next (the kernels wait with griddepcontrol.wait before they touch per-env memory).
// Measured on the B200 (PandaReach): 39.1 -> 37.5 us per step at 16,384 envs, but 14.8 -> 15.6 us at 4,096 envs (less than one
// wave of blocks: the early blocks of the next step land on the SMs that free up first and unbalance it), so `allow` is set
// for batches above 8,192 envs only.
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t stream, bool allow, Args... args)
{
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)grid);
    lc.blockDim = dim3((unsigned)block);
    lc.dynamicSmemBytes = smem;
    lc.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = allow ? 1 : 0;
    lc.attrs = attr;
    lc.numAttrs = 1;
    return cudaLaunchKernelEx(&lc, kernel, KArgs(args)...);
}

template <typename T, int G, int NQ, unsigned P_LO = 0u, unsigned P_HI = 0u, unsigned REV = 0u, bool ENV = false>
cudaError_t launch_panda_g(const ModelDev<T>* tables, const LaneTable<T>* lane_table, const PandaArgs<T>& a, const TreeBits& tb,
                           cudaStream_t stream, const EnvRows<T>& env)
{
    using L = LaneLayout<G>;
    // 64-thread blocks spread small batches over more SMs (4,096 envs: 14.4 us against 16.5 us), 128-thread blocks share
    // the staged model constants among more envs (16,384 envs: 39.0 us against 39.6 us)
    const int warps = a.n <= 8192 ? 2 : 4;
    const int64_t envs_per_block = (int64_t)warps * L::envs_per_warp;
    const int grid = (int)((a.n + envs_per_block - 1) / envs_per_block);
    const size_t smem = ((size_t)envs_per_block * L::stride + L::table + 12) * sizeof(T);
    cudaError_t rc = cudaFuncSetAttribute(k_task_panda_lanes<T, G, NQ, P_LO, P_HI, REV, ENV>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem);
    if (rc != cudaSuccess) return rc;
    return launch_pdl(k_task_panda_lanes<T, G, NQ, P_LO, P_HI, REV, ENV>, grid, 32 * warps, smem, stream, a.n > 8192, tables, lane_table,
                      a, tb, env);
}
// env.inertia != nullptr selects the per-env parameter variant of the same specialisation
template <typename T, int G, int NQ, unsigned P_LO = 0u, unsigned P_HI = 0u, unsigned REV = 0u>
cudaError_t launch_panda_v(const ModelDev<T>* tables, const LaneTable<T>* lane_table, const PandaArgs<T>& a, const TreeBits& tb,
                           cudaStream_t stream, const EnvRows<T>& env)
{
    return env.inertia ? launch_panda_g<T, G, NQ, P_LO, P_HI, REV, true>(tables, lane_table, a, tb, stream, env)
                       : launch_panda_g<T, G, NQ, P_LO, P_HI, REV>(tables, lane_table, a, tb, stream, env);
}
}  // namespace

template <typename T>
cudaError_t launch_task_panda_lanes(const ModelDev<T>* tables, const LaneTable<T>* lane_table, const PandaArgs<T>& a,
                                    const int* parent, const int* jtype, cudaStream_t stream, const EnvRows<T>& env)
{
    const TreeBits tb = make_tree_bits(a.nq, parent, jtype);
    if (a.nq <= 8) return launch_panda_v<T, 8, 0>(tables, lane_table, a, tb, stream, env);
    // the Panda (a chain of 7 revolute joints, two prismatic fingers on the last arm body): tree known at compile time
    constexpr unsigned kPandaLo = 0x76543210u, kPandaHi = 0x7u, kPandaRev = 0x7fu;
    if (a.nq == 9 && tb.p_lo == kPandaLo && tb.p_hi == kPandaHi && tb.rev_mask == kPandaRev)
        return launch_panda_v<T, 10, 9, kPandaLo, kPandaHi, kPandaRev>(tables, lane_table, a, tb, stream, env);
    if (a.nq <= 10) return launch_panda_v<T, 10, 0>(tables, lane_table, a, tb, stream, env);
    return launch_panda_v<T, 16, 0>(tables, lane_table, a, tb, stream, env);
}

namespace {
template <typename T, int G, bool CT, bool COUPLED, bool ENV = false>
cudaError_t launch_run_g(const ModelDev<T>* tables, const LaneTable<T>* lane_table, const RunCfg<T>& cfg, const RunBuffers<T>& b,
                         const TreeBits& tb, cudaStream_t stream, T* v0, int nvp, const EnvRows<T>& env)
{
    using L = LaneLayout<G>;
    const int warps = b.n <= 8192 ? 2 : 4;
    const int64_t envs_per_block = (int64_t)warps * L::envs_per_warp;
    const int grid = (int)((b.n + envs_per_block - 1) / envs_per_block);
    const size_t smem = ((size_t)envs_per_block * L::stride + L::table + 12) * sizeof(T);
    cudaError_t rc = cudaFuncSetAttribute(k_run_tree_lanes<T, G, CT, COUPLED, ENV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc != cudaSuccess) return rc;
    if (COUPLED) {  // must share SMs with k_coupled_rows / k_coupled_minv: the same shared-memory carve-out
        rc = cudaFuncSetAttribute(k_run_tree_lanes<T, G, CT, COUPLED, ENV>, cudaFuncAttributePreferredSharedMemoryCarveout, kCoupledCarveout);
        if (rc != cudaSuccess) return rc;
    }
    // a coupled step forks three kernels from one event: no programmatic overlap with the previous step's finish
    return launch_pdl(k_run_tree_lanes<T, G, CT, COUPLED, ENV>, grid, 32 * warps, smem, stream, !COUPLED && b.n > 8192, tables, lane_table,
                      cfg, b, tb, v0, nvp, env);
}
template <typename T, int G>
cudaError_t launch_run_v(const ModelDev<T>* tables, const LaneTable<T>* lane_table, const RunCfg<T>& cfg, const RunBuffers<T>& b,
                         const TreeBits& tb, cudaStream_t stream, T* v0, int nvp, const EnvRows<T>& env)
{
    const bool ct = cfg.ct_active && !cfg.paused;
    if (v0) return ct ? launch_run_g<T, G, true, true>(tables, lane_table, cfg, b, tb, stream, v0, nvp, env)
                      : launch_run_g<T, G, false, true>(tables, lane_table, cfg, b, tb, stream, v0, nvp, env);
    if (env.inertia) return ct ? launch_run_g<T, G, true, false, true>(tables, lane_table, cfg, b, tb, stream, v0, nvp, env)
                               : launch_run_g<T, G, false, false, true>(tables, lane_table, cfg, b, tb, stream, v0, nvp, env);
    return ct ? launch_run_g<T, G, true, false>(tables, lane_table, cfg, b, tb, stream, v0, nvp, env)
              : launch_run_g<T, G, false, false>(tables, lane_table, cfg, b, tb, stream, v0, nvp, env);
}
}  // namespace

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
