// Host-side entry points of the lane-parallel kernels (b2_lanes.cuh), compiled in their own translation unit
// (b2_lanes.cu) so that the engine's two halves build side by side, and the launch helper they share with b2_sim.cu.
#pragma once

#include <cuda_runtime.h>

#include "b2_kernels.cuh"

namespace b2 {

// Launch with programmatic stream serialization: consecutive steps on a stream overlap the tail of one launch with the
// scheduling and model staging of the next (the kernels wait with griddepcontrol.wait before they touch per-env memory).
// Measured on the B200 (PandaReach): 39.1 -> 37.5 us per step at 16,384 envs, but 14.8 -> 15.6 us at 4,096 envs (less than one
// wave of blocks: the early blocks of the next step land on the SMs that free up first and unbalance it), so the lane
// kernels set `allow` for batches above 8,192 envs only.
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

// Fused Panda task, G lanes per env (G chosen from the number of joints). env.inertia != nullptr: the physics reads every
// env's own parameters (b2sim_enable_env_params).
template <typename T>
cudaError_t launch_task_panda_lanes(const ModelDev<T>* tables, const LaneTable<T>* lane_table, const PandaArgs<T>& a,
                                    const int* parent, const int* jtype, cudaStream_t stream, const EnvRows<T>& env);

// GazeboSimulator::run of a fixed-base tree on lanes (k_run_tree_lanes): PID / force / velocity-follower joints, the
// computed-torque controller, resets, external link wrenches. v0 != nullptr: the model belongs to a coupled world; the
// kernel stops after the unconstrained velocity update and writes the joint velocities into the solver's v0 rows
// ([N, nvp]), leaving constraint solve, integration and the pending-reset mask to k_pgs_solve / k_world_finish.
// env.inertia != nullptr: the physics reads every env's own parameters (b2sim_enable_env_params); not with v0.
template <typename T>
cudaError_t launch_run_tree_lanes(const ModelDev<T>* tables, const LaneTable<T>* lane_table, const RunCfg<T>& cfg,
                                  const RunBuffers<T>& b, const int* parent, const int* jtype, cudaStream_t stream,
                                  T* v0 = nullptr, int nvp = 0, const EnvRows<T>& env = EnvRows<T>());

}  // namespace b2
