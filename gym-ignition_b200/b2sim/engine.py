"""Python handle on the b2sim engine: simulator, model tables and zero-copy torch views.

This is plumbing over the C ABI (include/b2sim.h); all arithmetic happens in the CUDA kernels of
csrc/b2_kernels.cuh. PyTorch is used for device memory views and streams only.
"""
import ctypes as C
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import B2Error, check

_TYPESTR = {_lib.F64: "<f8", _lib.F32: "<f4", -8: "|u1", -16: "<u2", -32: "<u4"}


class DeviceArray:
    """A [rows, cols] device buffer owned by the simulator, exposed through ``__cuda_array_interface__``
    so that ``torch.as_tensor(arr, device='cuda')`` aliases it without a copy."""

    def __init__(self, owner, ptr: int, rows: int, cols: int, dtype: int, vector: bool = False):
        self._owner = owner  # keeps the simulator alive while views exist
        self.ptr, self.rows, self.cols, self.dtype = ptr, rows, cols, dtype
        shape = (rows,) if vector else (rows, cols)
        self.__cuda_array_interface__ = {
            "shape": shape, "typestr": _TYPESTR[dtype], "data": (ptr, False), "version": 3, "strides": None}

    def torch(self, device_index: int = 0):
        import torch
        return torch.as_tensor(self, device=torch.device("cuda", device_index))


class ModelInfo:
    """Host-side description of a parsed model (names, table, kind). No GPU needed."""

    def __init__(self, handle: int, owned: bool):
        self._h, self._owned = handle, owned
        lib = _lib.load()
        self.name = lib.b2model_name(handle).decode()
        self.kind = lib.b2model_kind(handle)
        self.dofs = lib.b2model_dofs(handle)
        self.joint_names: List[str] = [lib.b2model_joint_name(handle, j).decode()
                                       for j in range(lib.b2model_num_joints(handle))]
        self.link_names: List[str] = [lib.b2model_link_name(handle, l).decode()
                                      for l in range(lib.b2model_num_links(handle))]

    @classmethod
    def from_string(cls, xml: str) -> "ModelInfo":
        data = xml.encode()
        h = _lib.load().b2model_parse(data, len(data))
        if not h:
            raise B2Error(_lib.ERR_PARSE, _lib.load().b2sim_last_error().decode())
        return cls(h, True)

    @classmethod
    def from_file(cls, path: str) -> "ModelInfo":
        with open(path, "r") as f:
            return cls.from_string(f.read())

    def tables(self) -> Dict[str, np.ndarray]:
        t = _lib.ModelTables()
        check(_lib.load().b2model_tables(self._h, C.byref(t)))
        nq, nl = t.nq, t.nlinks
        arr = lambda name, n, *shape: np.array(getattr(t, name), dtype=float).reshape((-1,) + shape)[:n]
        return dict(
            kind=t.kind, nq=nq, nlinks=nl, fixed_base=t.fixed_base,
            parent=np.array(t.parent, np.int32)[:nq], jtype=np.array(t.jtype, np.int32)[:nq],
            axis=arr("axis", nq, 3), R=arr("R", nq, 3, 3), p=arr("p", nq, 3), mass=arr("mass", nq),
            com=arr("com", nq, 3), Ic=arr("Ic", nq, 3, 3), damping=arr("damping", nq),
            friction=arr("friction", nq), stiffness=arr("stiffness", nq), rest=arr("rest", nq),
            lower=arr("lower", nq), upper=arr("upper", nq), effort=arr("effort", nq), vmax=arr("vmax", nq),
            link_body=np.array(t.link_body, np.int32)[:nl], link_R=arr("link_R", nl, 3, 3),
            link_p=arr("link_p", nl, 3), link_mass=arr("link_mass", nl), total_mass=t.total_mass,
            nshapes=t.nshapes, shape_type=np.array(t.shape_type, np.int32)[:t.nshapes],
            shape_link=np.array(t.shape_link, np.int32)[:t.nshapes], shape_size=arr("shape_size", t.nshapes, 3),
            shape_R=arr("shape_R", t.nshapes, 3, 3), shape_p=arr("shape_p", t.nshapes, 3),
            shape_mu=arr("shape_mu", t.nshapes), body_mass=t.body_mass, body_com=np.array(t.body_com),
            body_Ic=np.array(t.body_Ic).reshape(3, 3), base_mass=t.base_mass, base_mc=np.array(t.base_mc), link_com=arr("link_com", nl, 3),
            base_Io=np.array(t.base_Io))

    def __del__(self):
        if getattr(self, "_owned", False) and getattr(self, "_h", None):
            _lib.load().b2model_free(self._h)
            self._h = None


class Simulator:
    """N independent worlds on one GPU (replaces scenario::gazebo::GazeboSimulator + Physics system)."""

    def __init__(self, num_envs: int = 1, step_size: float = 0.001, steps_per_run: int = 1,
                 dtype: str = "float64", device: int = 0):
        lib = _lib.load()
        code = {"float64": _lib.F64, "float32": _lib.F32}[dtype]
        self._h = lib.b2sim_create(device, num_envs, step_size, steps_per_run, code)
        if not self._h:
            raise B2Error(_lib.ERR_CUDA, lib.b2sim_last_error().decode())
        self.lib = lib
        self.num_envs, self.device, self.dtype = num_envs, device, dtype
        self.step_size, self.steps_per_run = step_size, steps_per_run
        self._infos: Dict[int, ModelInfo] = {}

    # ---- lifetime ----
    def close(self):
        if getattr(self, "_h", None):
            self.lib.b2sim_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self) -> int:
        if not self._h:
            raise RuntimeError("the simulator was closed")
        return self._h

    # ---- world ----
    def set_stream(self, cuda_stream: Optional[int]):
        check(self.lib.b2sim_set_stream(self.handle, C.c_void_p(cuda_stream or 0)))

    def synchronize(self):
        check(self.lib.b2sim_synchronize(self.handle))

    def run(self, paused: bool = False):
        self.run_count = getattr(self, "run_count", 0) + 1  # readers may cache what they fetched until the next run
        check(self.lib.b2sim_run(self.handle, int(paused)))

    def time(self) -> float:
        return self.lib.b2sim_time(self.handle)

    def gravity(self):
        g = (C.c_double * 3)()
        check(self.lib.b2sim_gravity(self.handle, g))
        return list(g)

    def set_gravity(self, g: Sequence[float]):
        check(self.lib.b2sim_set_gravity(self.handle, (C.c_double * 3)(*g)))

    def launch_count(self) -> int:
        return self.lib.b2sim_launch_count(self.handle)

    # ---- models ----
    def insert_model(self, xml: str, pose: Sequence[float] = (0, 0, 0, 1, 0, 0, 0), name: str = "") -> int:
        data = xml.encode()
        mid = check(self.lib.b2sim_insert_model(self.handle, data, len(data), (C.c_double * 7)(*pose),
                                                name.encode()))
        self._infos[mid] = ModelInfo(self.lib.b2sim_model(self.handle, mid), owned=False)
        return mid

    def insert_model_file(self, path: str, pose=(0, 0, 0, 1, 0, 0, 0), name: str = "") -> int:
        with open(path, "r") as f:
            return self.insert_model(f.read(), pose, name)

    def remove_model(self, model: int):
        check(self.lib.b2sim_remove_model(self.handle, model))
        self._infos.pop(model, None)

    def model_id(self, name: str) -> int:
        return check(self.lib.b2sim_model_id(self.handle, name.encode()))

    def model_names(self) -> List[str]:
        return [self.lib.b2sim_model_name(self.handle, m).decode() for m in sorted(self._infos)]

    def info(self, model: int) -> ModelInfo:
        return self._infos[model]

    # ---- joint configuration (shared by all envs) ----
    def set_control_mode(self, model, joint, mode):
        check(self.lib.b2sim_set_control_mode(self.handle, model, joint, mode))

    def control_mode(self, model, joint) -> int:
        return check(self.lib.b2sim_control_mode(self.handle, model, joint))

    def set_pid(self, model, joint, p, i, d, i_max, i_min, cmd_max, cmd_min, cmd_offset):
        pid = _lib.Pid(p, i, d, i_max, i_min, cmd_max, cmd_min, cmd_offset)
        check(self.lib.b2sim_set_pid(self.handle, model, joint, C.byref(pid)))

    def pid(self, model, joint):
        pid = _lib.Pid()
        check(self.lib.b2sim_pid(self.handle, model, joint, C.byref(pid)))
        return pid

    def set_controller_period(self, model, period: float):
        check(self.lib.b2sim_set_controller_period(self.handle, model, period))

    def controller_period(self, model) -> float:
        return self.lib.b2sim_controller_period(self.handle, model)

    # ---- custom controller / external wrenches ----
    def set_computed_torque(self, model, kp, kd, gravity=(0.0, 0.0, -9.80665)):
        arr = lambda v: (C.c_double * len(v))(*[float(x) for x in v]) if v is not None else None
        check(self.lib.b2sim_set_computed_torque(self.handle, model, arr(kp), arr(kd), arr(gravity)))

    def apply_link_wrench(self, model, env, link, wrench, duration: float):
        check(self.lib.b2sim_apply_link_wrench(self.handle, model, env, link, (C.c_double * 6)(*[float(v) for v in wrench]),
                                               float(duration)))

    # ---- per-env scalars ----
    def get_joint(self, model, field, env, joint) -> float:
        v = C.c_double(0)
        check(self.lib.b2sim_get_joint(self.handle, model, field, env, joint, C.byref(v)))
        return v.value

    def set_joint(self, model, field, env, joint, value: float):
        check(self.lib.b2sim_set_joint(self.handle, model, field, env, joint, float(value)))

    def link_pose(self, model, env, link):
        p = (C.c_double * 7)()
        check(self.lib.b2sim_link_pose(self.handle, model, env, link, p))
        return list(p)

    # ---- free bodies and contacts ----
    def base_state(self, model, env):
        st = (C.c_double * 13)()
        check(self.lib.b2sim_base_state(self.handle, model, env, st))
        return list(st)

    def set_base(self, model, env, values, velocity: bool):
        arr = (C.c_double * len(values))(*[float(v) for v in values])
        check(self.lib.b2sim_set_base(self.handle, model, env, int(velocity), arr))

    def contacts(self, env, max_contacts: int = 32):
        """[(model_a, link_a, model_b, link_b, position, normal_b_to_a, depth, force_on_a), ...] of the last step."""
        ids = (C.c_int32 * (4 * max_contacts))()
        data = (C.c_double * (10 * max_contacts))()
        n = check(self.lib.b2sim_contacts(self.handle, env, max_contacts, ids, data))
        out = []
        for k in range(n):
            d = data[10 * k:10 * k + 10]
            out.append((ids[4 * k], ids[4 * k + 1], ids[4 * k + 2], ids[4 * k + 3], tuple(d[0:3]), tuple(d[3:6]), d[6],
                        tuple(d[7:10])))
        return out

    # ---- batched views ----
    def buffer(self, model, which) -> DeviceArray:
        b = _lib.Buffer()
        check(self.lib.b2sim_buffer(self.handle, model, which, C.byref(b)))
        vector = which in (_lib.BUF_RESET_MASK, _lib.BUF_REWARD, _lib.BUF_DONE, _lib.BUF_ELAPSED, _lib.BUF_EP_RETURN)
        return DeviceArray(self, b.ptr, b.rows, b.cols, b.dtype, vector)

    def tensor(self, model, which):
        return self.buffer(model, which).torch(self.device)

    # ---- per-env physical parameters ----
    def enable_env_params(self, model, enable: bool = True):
        """Gives every env of `model` its own body inertias, joint damping / Coulomb friction and gravity, starting from
        the model's current values. Returns zero-copy views (body_inertia [N, nq, 10]: mass, centre of mass xyz, inertia
        about it xx xy xz yy yz zz in the body frame; joint_dynamics [N, nq, 2]: damping, friction; gravity [N, 3]) that
        the caller writes between runs, e.g. at its resets; every unpaused run reads them. enable=False returns the model
        to its shared tables and returns None. The views do not own their memory: disabling, removing the model or
        closing the simulator frees it, and a view kept from before must not be used afterwards (enable again for new
        views). The computed-torque controller, the KinDyn queries and the link-level inertial data (ModelInfo tables,
        the centre of mass used by the scenario module's wrench-at-CoM) stay nominal."""
        check(self.lib.b2sim_enable_env_params(self.handle, model, 1 if enable else 0))
        if not enable:
            return None
        nq = self.buffer(model, _lib.BUF_JOINT_DYNAMICS).cols // 2
        inertia = self.tensor(model, _lib.BUF_BODY_INERTIA).view(self.num_envs, nq, 10)
        dynamics = self.tensor(model, _lib.BUF_JOINT_DYNAMICS).view(self.num_envs, nq, 2)
        return inertia, dynamics, self.tensor(model, _lib.BUF_GRAVITY)

    def _enable_rows(self, fn, model, enable):
        b = _lib.Buffer()
        check(fn(self.handle, model, 1 if enable else 0, C.byref(b)))
        if not enable:
            return None
        return DeviceArray(self, b.ptr, b.rows, b.cols, b.dtype).torch(self.device)

    def enable_free_body_params(self, model, enable: bool = True):
        """Gives every env its own mass, centre of mass and inertia of the free-floating `model`, starting from the loader's
        values. Returns a zero-copy view [N, 10]: mass, centre of mass xyz in the root-link frame, inertia about it xx xy xz
        yy yz zz in root-link axes; the caller writes it between runs, and every unpaused run reads it. Enabling again
        returns the same rows unchanged. enable=False returns the body to its shared values and returns None. The view
        does not own its memory: disabling, removing the model or closing the simulator frees it, and a view kept from
        before must not be used afterwards (enable again for a new view). Gravity, the link-level inertial data (ModelInfo
        tables) and the dynamics of an articulated model in the same world stay nominal."""
        return self._enable_rows(self.lib.b2sim_enable_free_body_params, model, enable)

    def enable_shape_friction(self, model, enable: bool = True):
        """Gives every env its own Coulomb friction coefficient of each collision shape of `model` (free, static or
        articulated), starting from the loader's values. Returns a zero-copy view [N, nshapes] (column k: shape k of the
        ModelInfo tables); a contact uses the smaller of its two shapes' values in its env. Same lifetime as
        enable_free_body_params: enable=False frees the rows and returns None, and a view kept from before must not be
        used after disabling, removing the model or closing the simulator."""
        return self._enable_rows(self.lib.b2sim_enable_shape_friction, model, enable)

    # ---- fused task path ----
    def set_task(self, model, task, seed=0, env_offset=0, max_episode_steps=5000):
        self.run_count = getattr(self, "run_count", 0) + 1  # the per-object view drops what it cached
        check(self.lib.b2sim_set_task(self.handle, model, task, seed, env_offset, max_episode_steps))

    def set_task_params(self, model, goal=None, q0=None, ee_link: int = -1):
        arr = lambda v: (C.c_double * len(v))(*[float(x) for x in v]) if v is not None else None
        check(self.lib.b2sim_set_task_params(self.handle, model, arr(goal), arr(q0), ee_link))

    def set_task_randomization(self, model, mass_delta: float, gravity_sigma: float):
        self.run_count = getattr(self, "run_count", 0) + 1  # the per-object view drops what it cached
        check(self.lib.b2sim_set_task_randomization(self.handle, model, float(mass_delta), float(gravity_sigma)))

    def task_reset_all(self, model):
        self.run_count = getattr(self, "run_count", 0) + 1  # the per-object view drops what it cached
        check(self.lib.b2sim_task_reset_all(self.handle, model))

    def task_observe(self, model):
        check(self.lib.b2sim_task_observe(self.handle, model))

    def task_step(self, model, actions_ptr: int):
        self.run_count = getattr(self, "run_count", 0) + 1  # the per-object view drops what it cached
        check(self.lib.b2sim_task_step(self.handle, model, C.c_void_p(actions_ptr)))

    def task_rollout(self, model, actions_ptr: int, steps: int, action_stride: int):
        self.run_count = getattr(self, "run_count", 0) + 1  # the per-object view drops what it cached
        check(self.lib.b2sim_task_rollout(self.handle, model, C.c_void_p(actions_ptr), steps, action_stride))

    def task_trajectory(self, model, actions_ptr: int, steps: int, obs_ptr: int = 0, reward_ptr: int = 0, done_ptr: int = 0):
        self.run_count = getattr(self, "run_count", 0) + 1  # the per-object view drops what it cached
        check(self.lib.b2sim_task_trajectory(self.handle, model, C.c_void_p(actions_ptr), steps, C.c_void_p(obs_ptr or None),
                                             C.c_void_p(reward_ptr or None), C.c_void_p(done_ptr or None)))

    def task_step_host(self, model, actions: np.ndarray, obs: np.ndarray, reward: np.ndarray, done: np.ndarray):
        self.run_count = getattr(self, "run_count", 0) + 1  # the per-object view drops what it cached
        # the C side copies n * nact / n * nobs / n elements of the simulator's scalar type: refuse anything else
        ftype = np.float64 if self.dtype == "float64" else np.float32
        nact = self.buffer(model, _lib.BUF_ACTION).cols
        nobs = self.buffer(model, _lib.BUF_OBS).cols
        for name, arr, dt, size, out in (("actions", actions, ftype, self.num_envs * nact, False),
                                         ("obs", obs, ftype, self.num_envs * nobs, True),
                                         ("reward", reward, ftype, self.num_envs, True),
                                         ("done", done, np.uint8, self.num_envs, True)):
            if not isinstance(arr, np.ndarray) or arr.dtype != dt or arr.size != size or not arr.flags.c_contiguous \
                    or (out and not arr.flags.writeable):
                raise ValueError(f"{name} must be a C-contiguous{' writeable' if out else ''} numpy array of "
                                 f"{np.dtype(dt).name} with {size} elements")
        check(self.lib.b2sim_task_step_host(self.handle, model, actions.ctypes.data, obs.ctypes.data,
                                            reward.ctypes.data, done.ctypes.data))

    # ---- episode statistics accumulated by the step kernels ----
    def episode_stats_enable(self, model, enable: bool = True):
        check(self.lib.b2sim_episode_stats_enable(self.handle, model, 1 if enable else 0))

    def episode_stats_tensor(self, model):
        """[STAT_STRIPES, 4] float64 device view of the striped totals (sum the rows)."""
        p = C.c_void_p()
        check(self.lib.b2sim_episode_stats_device(self.handle, model, C.byref(p)))
        return DeviceArray(self, p.value, _lib.STAT_STRIPES, 4, _lib.F64).torch(self.device)

    def episode_stats(self, model, clear: bool = False):
        out = (C.c_double * 4)()
        check(self.lib.b2sim_episode_stats(self.handle, model, out, 1 if clear else 0))
        return [float(v) for v in out]

    # ---- KinDyn ----
    def update_kinematics(self, model):
        check(self.lib.b2sim_update_kinematics(self.handle, model))

    def link_motion(self, model, link, twist=None, acceleration=None):
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        check(self.lib.b2sim_link_motion(self.handle, model, link, ptr(twist), ptr(acceleration)))

    def centroidal(self, model, com=None, com_velocity=None, momentum=None, com_jacobian=None):
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        check(self.lib.b2sim_centroidal(self.handle, model, ptr(com), ptr(com_velocity), ptr(momentum), ptr(com_jacobian)))

    def momentum_jacobian(self, model, momentum_jacobian=None, locked_inertia=None):
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        check(self.lib.b2sim_momentum_jacobian(self.handle, model, ptr(momentum_jacobian), ptr(locked_inertia)))

    def kindyn(self, model, link=0, mass_matrix=None, bias_forces=None, jacobian=None):
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        check(self.lib.b2sim_kindyn(self.handle, model, link, ptr(mass_matrix), ptr(bias_forces), ptr(jacobian)))
