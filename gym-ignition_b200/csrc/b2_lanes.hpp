// Host-side entry points of the lane-parallel kernels (b2_lanes.cuh), compiled in their own translation unit
// (b2_lanes.cu) so that the engine's two halves build side by side.
#pragma once

#include <cuda_runtime.h>

#include "b2_kernels.cuh"

namespace b2 {

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
