"""ctypes declarations for libb2sim.so (include/b2sim.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``csrc/Makefile``. Importing this module
fails loudly when the shared object is missing: there is no Python or CPU stand-in for the engine.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2SIM_LIBRARY") or os.path.normpath(os.path.join(_HERE, "..", "lib", "libb2sim.so"))

B2_MAX_DOFS = 16
B2_MAX_LINKS = 32
B2_MAX_SHAPES = 16

OK, ERR_INVALID, ERR_NOT_FOUND, ERR_PARSE, ERR_CUDA, ERR_UNSET, ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
F64, F32 = 0, 1
KIND_STATIC, KIND_CHAIN1, KIND_CHAIN_PR, KIND_TREE, KIND_FREE = 0, 1, 2, 3, 4
SHAPE_BOX, SHAPE_SPHERE, SHAPE_CYLINDER, SHAPE_PLANE = 0, 1, 2, 3

(BUF_STATE, BUF_ACCELERATION, BUF_FORCE_CMD, BUF_POS_TARGET, BUF_VEL_TARGET, BUF_PID_STATE,
 BUF_RESET_STATE, BUF_RESET_MASK, BUF_OBS, BUF_REWARD, BUF_DONE, BUF_ELAPSED, BUF_ACTION,
 BUF_LINK_POSE, BUF_BASE_STATE, BUF_BASE_RESET, BUF_ACC_TARGET, BUF_RAND_PARAMS, BUF_EP_RETURN,
 BUF_BASE_ACCEL, BUF_BODY_INERTIA, BUF_JOINT_DYNAMICS, BUF_GRAVITY) = range(23)
STAT_STRIPES = 32  # B2_STAT_STRIPES

(FIELD_POSITION, FIELD_VELOCITY, FIELD_ACCELERATION, FIELD_FORCE, FIELD_FORCE_TARGET,
 FIELD_POSITION_TARGET, FIELD_VELOCITY_TARGET, FIELD_POSITION_RESET, FIELD_VELOCITY_RESET,
 FIELD_ACCELERATION_TARGET) = range(10)

TASK_NONE = 0
TASK_PENDULUM_SWINGUP = 1
TASK_CARTPOLE_DISCRETE_BALANCING = 2
TASK_CARTPOLE_CONTINUOUS_BALANCING = 3
TASK_CARTPOLE_CONTINUOUS_SWINGUP = 4
TASK_PANDA_REACH = 5


class Buffer(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("rows", C.c_int64), ("cols", C.c_int64),
                ("dtype", C.c_int32), ("itemsize", C.c_int32)]


class ModelTables(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("nq", C.c_int32), ("nlinks", C.c_int32), ("fixed_base", C.c_int32),
        ("parent", C.c_int32 * B2_MAX_DOFS), ("jtype", C.c_int32 * B2_MAX_DOFS),
        ("axis", C.c_double * (B2_MAX_DOFS * 3)), ("R", C.c_double * (B2_MAX_DOFS * 9)),
        ("p", C.c_double * (B2_MAX_DOFS * 3)), ("mass", C.c_double * B2_MAX_DOFS),
        ("com", C.c_double * (B2_MAX_DOFS * 3)), ("Ic", C.c_double * (B2_MAX_DOFS * 9)),
        ("damping", C.c_double * B2_MAX_DOFS), ("friction", C.c_double * B2_MAX_DOFS),
        ("stiffness", C.c_double * B2_MAX_DOFS), ("rest", C.c_double * B2_MAX_DOFS),
        ("lower", C.c_double * B2_MAX_DOFS), ("upper", C.c_double * B2_MAX_DOFS),
        ("effort", C.c_double * B2_MAX_DOFS), ("vmax", C.c_double * B2_MAX_DOFS),
        ("link_body", C.c_int32 * B2_MAX_LINKS), ("link_R", C.c_double * (B2_MAX_LINKS * 9)),
        ("link_p", C.c_double * (B2_MAX_LINKS * 3)), ("link_mass", C.c_double * B2_MAX_LINKS),
        ("total_mass", C.c_double),
        ("nshapes", C.c_int32), ("shape_type", C.c_int32 * B2_MAX_SHAPES), ("shape_link", C.c_int32 * B2_MAX_SHAPES),
        ("shape_size", C.c_double * (B2_MAX_SHAPES * 3)), ("shape_R", C.c_double * (B2_MAX_SHAPES * 9)),
        ("shape_p", C.c_double * (B2_MAX_SHAPES * 3)), ("shape_mu", C.c_double * B2_MAX_SHAPES),
        ("body_mass", C.c_double), ("body_com", C.c_double * 3), ("body_Ic", C.c_double * 9),
        ("base_mass", C.c_double), ("base_mc", C.c_double * 3),
        ("link_com", C.c_double * (B2_MAX_LINKS * 3)),
        ("base_Io", C.c_double * 6),
    ]


class Pid(C.Structure):
    _fields_ = [(n, C.c_double) for n in
                ("p", "i", "d", "i_max", "i_min", "cmd_max", "cmd_min", "cmd_offset")]


# every symbol include/b2sim.h declares: name -> (restype, argtypes)
_vp, _i, _i64, _u64, _d, _cp = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_double, C.c_char_p
_dp = C.POINTER(C.c_double)
SYMBOLS = {
    "b2sim_last_error": (_cp, []),
    "b2sim_version": (_i, []),
    "b2sim_device_count": (_i, []),
    "b2model_parse": (_vp, [_cp, C.c_size_t]),
    "b2model_parse_file": (_vp, [_cp]),
    "b2model_free": (None, [_vp]),
    "b2model_name": (_cp, [_vp]),
    "b2model_kind": (_i, [_vp]),
    "b2model_dofs": (_i, [_vp]),
    "b2model_num_links": (_i, [_vp]),
    "b2model_num_joints": (_i, [_vp]),
    "b2model_joint_name": (_cp, [_vp, _i]),
    "b2model_link_name": (_cp, [_vp, _i]),
    "b2model_joint_index": (_i, [_vp, _cp]),
    "b2model_link_index": (_i, [_vp, _cp]),
    "b2model_tables": (_i, [_vp, C.POINTER(ModelTables)]),
    "b2sim_create": (_vp, [_i, _i64, _d, _i, _i]),
    "b2sim_destroy": (None, [_vp]),
    "b2sim_num_envs": (_i64, [_vp]),
    "b2sim_step_size": (_d, [_vp]),
    "b2sim_steps_per_run": (_i, [_vp]),
    "b2sim_dtype": (_i, [_vp]),
    "b2sim_set_stream": (_i, [_vp, _vp]),
    "b2sim_synchronize": (_i, [_vp]),
    "b2sim_run": (_i, [_vp, _i]),
    "b2sim_time": (_d, [_vp]),
    "b2sim_set_gravity": (_i, [_vp, _dp]),
    "b2sim_gravity": (_i, [_vp, _dp]),
    "b2sim_insert_model": (_i, [_vp, _cp, C.c_size_t, _dp, _cp]),
    "b2sim_remove_model": (_i, [_vp, _i]),
    "b2sim_num_models": (_i, [_vp]),
    "b2sim_model_id": (_i, [_vp, _cp]),
    "b2sim_model_name": (_cp, [_vp, _i]),
    "b2sim_model": (_vp, [_vp, _i]),
    "b2sim_set_control_mode": (_i, [_vp, _i, _i, _i]),
    "b2sim_control_mode": (_i, [_vp, _i, _i]),
    "b2sim_set_pid": (_i, [_vp, _i, _i, C.POINTER(Pid)]),
    "b2sim_pid": (_i, [_vp, _i, _i, C.POINTER(Pid)]),
    "b2sim_set_controller_period": (_i, [_vp, _i, _d]),
    "b2sim_controller_period": (_d, [_vp, _i]),
    "b2sim_set_max_generalized_force": (_i, [_vp, _i, _i, _d]),
    "b2sim_set_joint_friction": (_i, [_vp, _i, _i, _d, _d]),
    "b2sim_enable_env_params": (_i, [_vp, _i, _i]),
    "b2sim_enable_free_body_params": (_i, [_vp, _i, _i, C.POINTER(Buffer)]),
    "b2sim_enable_shape_friction": (_i, [_vp, _i, _i, C.POINTER(Buffer)]),
    "b2sim_set_computed_torque": (_i, [_vp, _i, _dp, _dp, _dp]),
    "b2sim_apply_link_wrench": (_i, [_vp, _i, _i64, _i, _dp, _d]),
    "b2sim_get_joint": (_i, [_vp, _i, _i, _i64, _i, _dp]),
    "b2sim_set_joint": (_i, [_vp, _i, _i, _i64, _i, _d]),
    "b2sim_link_pose": (_i, [_vp, _i, _i64, _i, _dp]),
    "b2sim_set_base": (_i, [_vp, _i, _i64, _i, _dp]),
    "b2sim_base_state": (_i, [_vp, _i, _i64, _dp]),
    "b2sim_contacts": (_i, [_vp, _i64, _i, C.POINTER(C.c_int32), _dp]),
    "b2sim_buffer": (_i, [_vp, _i, _i, C.POINTER(Buffer)]),
    "b2sim_set_task": (_i, [_vp, _i, _i, _u64, _u64, _i]),
    "b2sim_set_task_params": (_i, [_vp, _i, _dp, _dp, _i]),
    "b2sim_set_task_randomization": (_i, [_vp, _i, _d, _d]),
    "b2sim_task_reset_all": (_i, [_vp, _i]),
    "b2sim_task_observe": (_i, [_vp, _i]),
    "b2sim_task_step": (_i, [_vp, _i, _vp]),
    "b2sim_task_rollout": (_i, [_vp, _i, _vp, _i, _i64]),
    "b2sim_task_trajectory": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp]),
    "b2sim_task_step_host": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "b2sim_task_nobs": (_i, [_i]),
    "b2sim_task_nact": (_i, [_i]),
    "b2sim_task_steps_done": (_u64, [_vp, _i]),
    "b2sim_episode_stats_enable": (_i, [_vp, _i, _i]),
    "b2sim_episode_stats_device": (_i, [_vp, _i, C.POINTER(C.c_void_p)]),
    "b2sim_episode_stats": (_i, [_vp, _i, _dp, _i]),
    "b2sim_launch_count": (_u64, [_vp]),
    "b2sim_update_kinematics": (_i, [_vp, _i]),
    "b2sim_kindyn": (_i, [_vp, _i, _i, _vp, _vp, _vp]),
    "b2sim_link_motion": (_i, [_vp, _i, _i, _vp, _vp]),
    "b2sim_centroidal": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "b2sim_momentum_jacobian": (_i, [_vp, _i, _vp, _vp]),
}

_lib = None


def load():
    """Load libb2sim.so and bind every exported symbol. Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA engine first (python -c 'import __graft_entry__ as g; "
            "g.build()' or make -C gym-ignition_b200/csrc). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class B2Error(RuntimeError):
    """Raised for negative status codes; the reference maps every C++ exception to RuntimeError
    (bindings/core/core.i:14-22)."""

    def __init__(self, code, message):
        super().__init__(f"b2sim error {code}: {message}")
        self.code = code


def check(code):
    if code is None or code < 0:
        raise B2Error(code, load().b2sim_last_error().decode())
    return code
