"""Batched task environment: N worlds stepped by one fused kernel launch per env.step.

Host-side mirror of the reference's GazeboRuntime.step / reset relay
(python/gym_ignition/runtimes/gazebo_runtime.py:91-140) for all envs at once. The per-env semantics are
those of the reference tasks (python/gym_ignition_environments/tasks/*.py); see csrc/b2_kernels.cuh.
"""
from typing import Optional, Tuple

import numpy as np

from . import _lib
from .engine import Simulator

TASKS = {
    "Pendulum-Gazebo-v0": (_lib.TASK_PENDULUM_SWINGUP, "pendulum"),
    "CartPoleDiscreteBalancing-Gazebo-v0": (_lib.TASK_CARTPOLE_DISCRETE_BALANCING, "cartpole"),
    "CartPoleContinuousBalancing-Gazebo-v0": (_lib.TASK_CARTPOLE_CONTINUOUS_BALANCING, "cartpole"),
    "CartPoleContinuousSwingup-Gazebo-v0": (_lib.TASK_CARTPOLE_CONTINUOUS_SWINGUP, "cartpole"),
    # not a registered id of the reference: BASELINE.json config 4 (Panda position PID + KinDyn observation)
    "PandaReach-Gazebo-v0": (_lib.TASK_PANDA_REACH, "panda"),
}

#: models/panda.py:42-44 initial arm configuration (+ closed fingers) and :48-58 PID gains at 1 kHz
PANDA_Q0 = [0, -0.785, 0, -2.356, 0, 1.571, 0.785, 0.0, 0.0]
PANDA_PID = [(50, 0, 20), (10000, 0, 500), (100, 0, 10), (1000, 0, 50), (100, 0, 10), (100, 0, 10), (10, 0.5, 0.1),
             (100, 0, 50), (100, 0, 50)]

# Algorithmic HBM bytes per env-step in fp64 (SURVEY.md §8d): read q,dq + action + reset flag,
# write q,dq + obs + reward + done.
ALGORITHMIC_BYTES = {
    _lib.TASK_PENDULUM_SWINGUP: {"float64": 74, "float32": 38},
    _lib.TASK_CARTPOLE_DISCRETE_BALANCING: {"float64": 114, "float32": 58},
    _lib.TASK_CARTPOLE_CONTINUOUS_BALANCING: {"float64": 114, "float32": 58},
    _lib.TASK_CARTPOLE_CONTINUOUS_SWINGUP: {"float64": 114, "float32": 58},
    # read q,dq 144 + targets 72 + PID state 216 + flag 1; write q,dq 144 + PID state 216 + obs 920 + reward 8 + done 1
    _lib.TASK_PANDA_REACH: {"float64": 1722, "float32": 862},
}


class BatchedTaskEnv:
    """``num_envs`` independent copies of a registered gym-ignition environment on one GPU."""

    def __init__(self, env_id: str, num_envs: int, dtype: str = "float64", device: int = 0, seed: int = 0,
                 env_offset: int = 0, max_episode_steps: int = 5000, physics_rate: float = 1000.0,
                 agent_rate: float = 1000.0, model_file: Optional[str] = None, **kwargs):
        import gym_ignition_models
        import torch

        if env_id not in TASKS:
            raise ValueError(f"unknown environment '{env_id}'")
        self.env_id = env_id
        self.task, model_name = TASKS[env_id]
        steps_per_run = int(physics_rate / agent_rate)
        self.sim = Simulator(num_envs, 1.0 / physics_rate, steps_per_run, dtype, device)
        # same world population as GazeboRuntime.world: ground plane + the robot
        self.ground = self.sim.insert_model_file(gym_ignition_models.get_model_file("ground_plane"))
        self.model = self.sim.insert_model_file(model_file or gym_ignition_models.get_model_file(model_name))
        if self.task == _lib.TASK_PANDA_REACH:
            dbl_max = float(np.finfo(np.float64).max)
            for j, (p, i, d) in enumerate(PANDA_PID):  # Joint.set_pid replaces the +-DBL_MAX limits by +-effort
                self.sim.set_pid(self.model, j, p, i, d, dbl_max, -dbl_max, dbl_max, -dbl_max, 0.0)
            self.sim.set_task_params(self.model, goal=kwargs.get("goal", (0.5, 0.0, 0.5)), q0=PANDA_Q0)
        self.sim.set_task(self.model, self.task, seed, env_offset, max_episode_steps)
        self.num_envs, self.dtype, self.device = num_envs, dtype, device
        self.torch_dtype = torch.float64 if dtype == "float64" else torch.float32
        self.state = self.sim.tensor(self.model, _lib.BUF_STATE)
        self.obs = self.sim.tensor(self.model, _lib.BUF_OBS)
        self.reward = self.sim.tensor(self.model, _lib.BUF_REWARD)
        self.done = self.sim.tensor(self.model, _lib.BUF_DONE)
        self.elapsed = self.sim.tensor(self.model, _lib.BUF_ELAPSED)
        self.nobs = self.obs.shape[1]
        self.nact = self.sim.buffer(self.model, _lib.BUF_ACTION).cols
        self.bytes_per_env_step = ALGORITHMIC_BYTES[self.task][dtype]
        self.rand_params = self.env_params = None
        self.episode_stats_enabled = False

    def randomize(self, mass_delta: float = 0.2, gravity_sigma: float = 0.2):
        """Per-env domain randomisation (randomizers/cartpole.py:51-56,100-135): at every reset an env draws link
        mass offsets U(-mass_delta, mass_delta) and gravity_z ~ N(g_z, gravity_sigma). Returns the [N, nq+1] tensor of
        (mass offsets, gravity scale) that the step kernel reads (+8 (nq+1) bytes of traffic per env-step)."""
        self.sim.set_task_randomization(self.model, mass_delta, gravity_sigma)
        if mass_delta == 0 and gravity_sigma == 0:
            self.rand_params = None
        else:
            self.rand_params = self.sim.tensor(self.model, _lib.BUF_RAND_PARAMS)
            self.bytes_per_env_step = ALGORITHMIC_BYTES[self.task][self.dtype] + \
                (8 if self.dtype == "float64" else 4) * self.rand_params.shape[1]
        return self.rand_params

    def enable_env_params(self, enable: bool = True):
        """Per-env body inertias, joint damping / Coulomb friction and gravity for the reach task
        (``Simulator.enable_env_params``; the pendulum and cart-pole tasks raise B2Error and have ``randomize``). Returns
        the views (body_inertia [N, nq, 10], joint_dynamics [N, nq, 2], gravity [N, 3]), or None when disabling. Every
        step reads them (+(12 nq + 3) scalars of traffic per env-step). For new parameters per episode, write the rows of
        the envs whose ``done`` is set (e.g. with torch.where on the done mask) after the step that reports it and before
        the next one: the terminal step ran with the old rows, the new episode runs with the new ones. The reach task
        ends at its TimeLimit only, so its envs finish together unless ``elapsed`` is staggered."""
        self.env_params = self.sim.enable_env_params(self.model, enable)
        self._count_bytes()
        return self.env_params

    def enable_episode_stats(self, enable: bool = True) -> None:
        """Let the step kernels accumulate [sum of returns, sum of lengths, finished episodes, non-finite rewards] on
        the device (two extra scalars of traffic per env-step). Read them with ``episode_stats()`` or hand them to
        ``b2sim.distributed.EpisodeStats`` for the end-of-rollout sum over ranks."""
        self.sim.episode_stats_enable(self.model, enable)
        self.episode_stats_enabled = enable
        self._count_bytes()

    def _count_bytes(self) -> None:
        """bytes_per_env_step: the task's traffic plus what the enabled per-env extras read or write per env-step."""
        es = 8 if self.dtype == "float64" else 4
        self.bytes_per_env_step = ALGORITHMIC_BYTES[self.task][self.dtype] + (2 * es if self.episode_stats_enabled else 0) + \
            (es * self.rand_params.shape[1] if self.rand_params is not None else 0) + \
            (es * sum(v[0].numel() for v in self.env_params) if self.env_params is not None else 0)

    def episode_stats(self, clear: bool = False):
        """Host copy of the four totals (synchronises the stream)."""
        return self.sim.episode_stats(self.model, clear)

    def use_stream(self, stream) -> None:
        """Enqueue the kernels on ``stream`` (a torch.cuda.Stream); default is the legacy default stream."""
        self.sim.set_stream(stream.cuda_stream if stream is not None else None)

    def reset(self):
        """Fresh episodes for every env (Task.reset_task + paused run); returns the initial observations."""
        self.sim.task_reset_all(self.model)
        return self.observe()

    def observe(self):
        """Recompute obs / reward / done from the current state without stepping."""
        self.sim.task_observe(self.model)
        return self.obs

    def step(self, actions) -> Tuple["torch.Tensor", "torch.Tensor", "torch.Tensor"]:
        """actions: device tensor [N] or [N, 1] in the simulator dtype. One kernel launch; no sync.

        Auto-reset contract: an env whose episode ends on this step (task termination or the TimeLimit) reports the
        terminal observation / reward / done = 1 and is reset inside the same launch, so its NEXT step already belongs to
        a fresh episode. ``obs`` keeps the terminal observation (what a serial GazeboRuntime user sees before calling
        ``reset()``); ``observe()`` recomputes the observations from the current states, i.e. the first observation of
        the new episode for the envs that just finished (one light launch, no stepping)."""
        if actions.dtype != self.torch_dtype or not actions.is_cuda or actions.numel() != self.num_envs * self.nact:
            raise ValueError("actions must be a CUDA tensor [num_envs, nact] in the simulator dtype")
        if not actions.is_contiguous():
            actions = actions.contiguous()
        self.sim.task_step(self.model, actions.data_ptr())
        return self.obs, self.reward, self.done

    def rollout(self, actions) -> None:
        """actions: CUDA tensor [T, N] (open-loop); T fused steps issued from C without returning to Python.
        obs / reward / done hold the outputs of the last step."""
        if actions.dtype != self.torch_dtype or not actions.is_cuda or actions.dim() < 2 \
                or actions[0].numel() != self.num_envs * self.nact or not actions.is_contiguous():
            raise ValueError("actions must be a contiguous CUDA tensor [T, num_envs(, nact)] in the simulator dtype")
        self.sim.task_rollout(self.model, actions.data_ptr(), actions.shape[0], actions[0].numel())

    def trajectory(self, actions, record: bool = True, out=None):
        """Open-loop rollout in ONE kernel launch (pendulum / cart-pole tasks): actions is a contiguous CUDA tensor
        [T, N]; every env keeps its state in registers over the T steps. Returns (obs [T, N, nobs], reward [T, N],
        done [T, N] uint8) when `record`, else None; obs / reward / done / state hold the last step either way.
        Same results as T calls of step() (done masks and resets exactly, states to rounding). `out` may pass preallocated output tensors."""
        import torch
        if actions.dtype != self.torch_dtype or not actions.is_cuda or actions.dim() < 2 \
                or actions[0].numel() != self.num_envs or not actions.is_contiguous():
            raise ValueError("actions must be a contiguous CUDA tensor [T, num_envs] in the simulator dtype")
        T = actions.shape[0]
        if not record:
            self.sim.task_trajectory(self.model, actions.data_ptr(), T)
            return None
        if out is None:
            out = (torch.empty((T, self.num_envs, self.nobs), dtype=self.torch_dtype, device=actions.device),
                   torch.empty((T, self.num_envs), dtype=self.torch_dtype, device=actions.device),
                   torch.empty((T, self.num_envs), dtype=torch.uint8, device=actions.device))
        o, r, d = out
        if o.shape != (T, self.num_envs, self.nobs) or r.shape != (T, self.num_envs) or d.shape != (T, self.num_envs) \
                or not (o.is_contiguous() and r.is_contiguous() and d.is_contiguous()) \
                or o.dtype != self.torch_dtype or r.dtype != self.torch_dtype or d.dtype != torch.uint8:
            raise ValueError("trajectory outputs have the wrong shape, dtype or layout")
        self.sim.task_trajectory(self.model, actions.data_ptr(), T, o.data_ptr(), r.data_ptr(), d.data_ptr())
        return out

    def step_host(self, actions: np.ndarray, obs: np.ndarray, reward: np.ndarray, done: np.ndarray) -> None:
        """Host-buffer variant: H2D actions, step, D2H obs/reward/done, synchronise."""
        self.sim.task_step_host(self.model, actions, obs, reward, done)

    def close(self):
        self.state = self.obs = self.reward = self.done = self.elapsed = None
        self.sim.close()
