/* b2sim — C ABI of the B200-native batched physics-and-observation engine.
 *
 * This is the drop-in boundary for gym-ignition's env.step hot path: the entry points below are what a
 * binding for the Python module `scenario` (SWIG in the reference: bindings/core/core.i,
 * bindings/gazebo/gazebo.i) binds instead of ScenarI/O's C++ classes. Plain pointers and sizes only;
 * no torch / C++ types. Every function returns 0 on success (or a non-negative id / count) and a
 * negative B2_ERR_* code on failure; b2sim_last_error() gives the message (the reference logs with
 * sError and returns false: e.g. cpp/scenario/gazebo/src/Joint.cpp:134-138).
 *
 * One simulator = N independent worlds ("envs") on one GPU, all holding the same models
 * (the reference: one process = one world = one robot, docs/sphinx/info/limitations.rst:19-20).
 * Per-env state is struct-of-arrays in HBM, env-major: q/dq live in state[N][2*nq].
 *
 * The library has no CPU fallback: anything that touches per-env state needs a CUDA device and fails
 * with B2_ERR_CUDA otherwise. Model parsing (b2model_*) is host-only and works without a GPU.
 */
#ifndef B2SIM_H
#define B2SIM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_MAX_DOFS 16
#define B2_MAX_LINKS 32
#define B2_MAX_SHAPES 16

/* ---- status codes ------------------------------------------------------------------------- */
enum {
    B2_OK = 0,
    B2_ERR_INVALID = -1,   /* bad argument / wrong control mode (reference: returns false) */
    B2_ERR_NOT_FOUND = -2, /* unknown model / joint / link (reference: ModelNotFound, JointNotFound) */
    B2_ERR_PARSE = -3,     /* malformed URDF / SDF */
    B2_ERR_CUDA = -4,      /* no device, or a CUDA call failed */
    B2_ERR_UNSET = -5,     /* reading a target that was never set (reference: ComponentNotFound) */
    B2_ERR_UNSUPPORTED = -6
};

/* cpp/scenario/core/include/scenario/core/Joint.h:25-45 */
enum { B2_JOINT_INVALID = 0, B2_JOINT_FIXED = 1, B2_JOINT_REVOLUTE = 2, B2_JOINT_PRISMATIC = 3, B2_JOINT_BALL = 4 };
enum {
    B2_MODE_INVALID = 0,
    B2_MODE_IDLE = 1,
    B2_MODE_FORCE = 2,
    B2_MODE_VELOCITY = 3,
    B2_MODE_VELOCITY_FOLLOWER_DART = 4,
    B2_MODE_POSITION = 5,
    B2_MODE_POSITION_INTERPOLATED = 6
};

enum { B2_F64 = 0, B2_F32 = 1 };

/* How the dynamics of a model are evaluated on the device. */
enum {
    B2_KIND_STATIC = 0,  /* no degrees of freedom (ground plane, fixtures) */
    B2_KIND_CHAIN1 = 1,  /* one 1-DoF joint: closed form  I q'' = tau - g(q)            (pendulum) */
    B2_KIND_CHAIN_PR = 2,/* prismatic -> revolute chain: closed-form 2x2                 (cartpole) */
    B2_KIND_TREE = 3,    /* general fixed-base tree of 1-DoF joints: articulated-body algorithm    */
    B2_KIND_FREE = 4     /* one free-floating rigid body (all links welded together): contact dynamics */
};

/* Collision primitives kept by the loader (size: box = full extents xyz, sphere = radius, cylinder = radius,
 * length, plane = normal). */
enum { B2_SHAPE_BOX = 0, B2_SHAPE_SPHERE = 1, B2_SHAPE_CYLINDER = 2, B2_SHAPE_PLANE = 3 };

/* Tasks of python/gym_ignition_environments/tasks/ (fused observation / reward / done / reset). */
enum {
    B2_TASK_NONE = 0,
    B2_TASK_PENDULUM_SWINGUP = 1,               /* pendulum_swingup.py:29-130 */
    B2_TASK_CARTPOLE_DISCRETE_BALANCING = 2,    /* cartpole_discrete_balancing.py:41-144 */
    B2_TASK_CARTPOLE_CONTINUOUS_BALANCING = 3,  /* cartpole_continuous_balancing.py:40-146 */
    B2_TASK_CARTPOLE_CONTINUOUS_SWINGUP = 4,    /* cartpole_continuous_swingup.py:40-153 */
    B2_TASK_PANDA_REACH = 5                     /* Panda PID tracking + KinDyn FK/Jacobian observation */
};

/* Per-env buffers that can be viewed zero-copy (b2sim_buffer). Shapes are [num_envs, cols]. */
enum {
    B2_BUF_STATE = 0,        /* [N, 2*nq]  q then dq                      (JointPosition, JointVelocity) */
    B2_BUF_ACCELERATION = 1, /* [N, nq]                                  (JointAcceleration) */
    B2_BUF_FORCE_CMD = 2,    /* [N, nq]  one-shot force command          (JointForceCmd) */
    B2_BUF_POS_TARGET = 3,   /* [N, nq]                                  (JointPositionTarget) */
    B2_BUF_VEL_TARGET = 4,   /* [N, nq]                                  (JointVelocityTarget) */
    B2_BUF_PID_STATE = 5,    /* [N, 3*nq] iErr, pErrLast, cmd per joint  (JointPID state) */
    B2_BUF_RESET_STATE = 6,  /* [N, 2*nq] pending reset values           (Joint{Position,Velocity}Reset) */
    B2_BUF_RESET_MASK = 7,   /* [N] uint32: bit j = position reset of dof j, bit 16+j = velocity reset */
    B2_BUF_OBS = 8,          /* [N, nobs] task observation */
    B2_BUF_REWARD = 9,       /* [N] */
    B2_BUF_DONE = 10,        /* [N] uint8 */
    B2_BUF_ELAPSED = 11,     /* [N] uint16 steps since the episode started (gym TimeLimit) */
    B2_BUF_ACTION = 12,      /* [N, nact] staging buffer used by b2sim_task_step_host */
    B2_BUF_LINK_POSE = 13,   /* [N, 7*nlinks] world pose (xyz, quat wxyz) after b2sim_update_kinematics */
    B2_BUF_BASE_STATE = 14,  /* [N, 13] B2_KIND_FREE: base position xyz, quaternion wxyz, world linear and angular velocity */
    B2_BUF_BASE_RESET = 15,  /* [N, 13] pending WorldPoseCmd / WorldVelocityCmd values (Model::resetBase*) */
    B2_BUF_ACC_TARGET = 16,  /* [N, nq]                                  (JointAccelerationTarget) */
    B2_BUF_RAND_PARAMS = 17, /* [N, nq+1] per-env body mass offsets and gravity scale (domain randomisation) */
    B2_BUF_EP_RETURN = 18,   /* [N] running return of the current episode (b2sim_episode_stats_enable) */
    B2_BUF_BASE_ACCEL = 19,  /* [N, 6] B2_KIND_FREE: world linear acceleration of the base frame origin and angular acceleration
                              * over the last step, constraint impulses included (Link::world{Linear,Angular}Acceleration,
                              * Link.cpp:240-294; DART adds the velocity change of the constraint stage / dt to the accelerations) */
    /* Per-env physical parameters (b2sim_enable_env_params), read by every unpaused b2sim_run of the model and every
     * step of its reach task: */
    B2_BUF_BODY_INERTIA = 20,   /* [N, 10*nq] per body j (child of joint j, welded links lumped in as in b2_model_tables):
                                 * mass, centre of mass xyz, inertia about it Ixx Ixy Ixz Iyy Iyz Izz, both in the body frame */
    B2_BUF_JOINT_DYNAMICS = 21, /* [N, 2*nq] per joint: viscous damping, Coulomb friction */
    B2_BUF_GRAVITY = 22,        /* [N, 3] gravity this model's dynamics sees in the env, world frame */
    B2_BUF_COUNT = 23
};

typedef struct {
    void* ptr;        /* device pointer */
    int64_t rows;     /* num_envs */
    int64_t cols;
    int32_t dtype;    /* B2_F64 / B2_F32, or -8 for uint8, -16 for uint16, -32 for uint32 */
    int32_t itemsize;
} b2_buffer;

/* Flattened model tables (what the loader produces; SURVEY.md §7 step 1). */
typedef struct {
    int32_t kind;
    int32_t nq;                         /* moving 1-DoF joints = bodies, parents first */
    int32_t nlinks;                     /* all links except "world" */
    int32_t fixed_base;
    int32_t parent[B2_MAX_DOFS];        /* parent body, -1 = base */
    int32_t jtype[B2_MAX_DOFS];         /* B2_JOINT_REVOLUTE / B2_JOINT_PRISMATIC */
    double axis[B2_MAX_DOFS][3];
    double R[B2_MAX_DOFS][9];           /* child frame in parent body frame at q = 0 */
    double p[B2_MAX_DOFS][3];
    double mass[B2_MAX_DOFS];
    double com[B2_MAX_DOFS][3];
    double Ic[B2_MAX_DOFS][9];
    double damping[B2_MAX_DOFS], friction[B2_MAX_DOFS], stiffness[B2_MAX_DOFS], rest[B2_MAX_DOFS];
    double lower[B2_MAX_DOFS], upper[B2_MAX_DOFS], effort[B2_MAX_DOFS], vmax[B2_MAX_DOFS];
    int32_t link_body[B2_MAX_LINKS];    /* body a link is rigidly attached to, -1 = base */
    double link_R[B2_MAX_LINKS][9];     /* link frame in its body frame */
    double link_p[B2_MAX_LINKS][3];
    double link_mass[B2_MAX_LINKS];
    double total_mass;
    /* collision shapes, pose given in the frame of the link they belong to */
    int32_t nshapes;
    int32_t shape_type[B2_MAX_SHAPES];
    int32_t shape_link[B2_MAX_SHAPES];
    double shape_size[B2_MAX_SHAPES][3];
    double shape_R[B2_MAX_SHAPES][9];
    double shape_p[B2_MAX_SHAPES][3];
    double shape_mu[B2_MAX_SHAPES];
    /* B2_KIND_FREE: the lumped rigid body, in the frame of the root (base) link */
    double body_mass;
    double body_com[3];
    double body_Ic[9];
    /* links welded to the fixed base: total mass and first moment (mass * com) in the base frame; they do not
     * move but count in the centre of mass (KinDynComputations.get_com_position) */
    double base_mass;
    double base_mc[3];
    /* centre of mass of every link in its own frame (components::Inertial pose; Link::applyWorldWrenchToCoM,
     * Link.cpp:529-557) */
    double link_com[B2_MAX_LINKS][3];
    /* rotational inertia of the links welded to the fixed base about the base origin, base frame (xx, xy, xz, yy, yz, zz):
     * the base's share of the locked inertia (KinDynComputations average-velocity Jacobians) */
    double base_Io[6];
} b2_model_tables;

/* scenario::core::PID, cpp/scenario/core/include/scenario/core/Joint.h:505-523 */
typedef struct {
    double p, i, d, i_max, i_min, cmd_max, cmd_min, cmd_offset;
} b2_pid;

const char* b2sim_last_error(void);
int b2sim_version(void);
/* Number of CUDA devices visible (0 on a CPU-only host). */
int b2sim_device_count(void);

/* ---- model loader: replaces sdformat + SdfEntityCreator (World.cpp:70-180, helpers.cpp:48-88) ---- */
typedef struct b2model b2model;
b2model* b2model_parse(const char* xml, size_t len);          /* URDF, or an SDF <model> subset */
b2model* b2model_parse_file(const char* path);
void b2model_free(b2model* m);
const char* b2model_name(const b2model* m);
int b2model_kind(const b2model* m);
int b2model_dofs(const b2model* m);                           /* Model::dofs, Model.cpp:527-541 */
int b2model_num_links(const b2model* m);
int b2model_num_joints(const b2model* m);                     /* 1-DoF joints only, Model.cpp:555-559 */
const char* b2model_joint_name(const b2model* m, int j);
const char* b2model_link_name(const b2model* m, int l);
int b2model_joint_index(const b2model* m, const char* name);  /* B2_ERR_NOT_FOUND if absent */
int b2model_link_index(const b2model* m, const char* name);
int b2model_tables(const b2model* m, b2_model_tables* out);

/* ---- simulator: replaces scenario::gazebo::GazeboSimulator (GazeboSimulator.h:57-188) ------------ */
typedef struct b2sim b2sim;
b2sim* b2sim_create(int device, int64_t num_envs, double step_size, int steps_per_run, int dtype);
void b2sim_destroy(b2sim* s);
int64_t b2sim_num_envs(const b2sim* s);
double b2sim_step_size(const b2sim* s);
int b2sim_steps_per_run(const b2sim* s);
int b2sim_dtype(const b2sim* s);
/* Kernels are enqueued on this stream (a cudaStream_t; NULL = the legacy default stream). */
int b2sim_set_stream(b2sim* s, void* cuda_stream);
int b2sim_synchronize(b2sim* s);
/* GazeboSimulator::run(paused), GazeboSimulator.cpp:202-251: steps_per_run iterations of
 * JointController::PreUpdate + Physics::Update for every env; a paused run applies pending resets
 * and refreshes readbacks without advancing time. */
int b2sim_run(b2sim* s, int paused);
double b2sim_time(const b2sim* s);                            /* World::time, World.cpp:293-299 */
int b2sim_set_gravity(b2sim* s, const double g[3]);           /* World.cpp:301-319: only at time 0 */
int b2sim_gravity(const b2sim* s, double g[3]);

/* World::insertModel (World.cpp:394-429). pose = xyz + quaternion wxyz. Returns the model id. */
int b2sim_insert_model(b2sim* s, const char* xml, size_t len, const double pose[7], const char* name);
int b2sim_remove_model(b2sim* s, int model);                  /* World.cpp:431-453 */
int b2sim_num_models(const b2sim* s);
int b2sim_model_id(const b2sim* s, const char* name);         /* B2_ERR_NOT_FOUND if absent */
const char* b2sim_model_name(const b2sim* s, int model);
const b2model* b2sim_model(const b2sim* s, int model);

/* ---- per-model joint configuration (shared by all envs) ----------------------------------------- */
int b2sim_set_control_mode(b2sim* s, int model, int joint, int mode);     /* Joint.cpp:369-460 */
int b2sim_control_mode(const b2sim* s, int model, int joint);
int b2sim_set_pid(b2sim* s, int model, int joint, const b2_pid* pid);     /* Joint.cpp:479-525 */
int b2sim_pid(const b2sim* s, int model, int joint, b2_pid* pid);
int b2sim_set_controller_period(b2sim* s, int model, double period);      /* Model.cpp:589-602 */
double b2sim_controller_period(const b2sim* s, int model);
int b2sim_set_max_generalized_force(b2sim* s, int model, int joint, double f); /* Joint.cpp:908-940 */
/* Joint::setCoulombFriction / setViscousFriction (Joint.cpp:259-311): SDF <dynamics> friction and damping of one
 * joint, for every env; a negative value leaves that parameter unchanged. The caller enforces the reference's
 * "only while the model has just been created" rule (helpers.cpp:131-157). */
int b2sim_set_joint_friction(b2sim* s, int model, int joint, double coulomb, double viscous);
/* Per-env physical parameters (domain randomisation of articulated models: the batched counterpart of editing the SDF and
 * re-inserting the model at a reset, gym_ignition/randomizers/gazebo_env_randomizer.py). enable != 0 allocates
 * B2_BUF_BODY_INERTIA, B2_BUF_JOINT_DYNAMICS and B2_BUF_GRAVITY in the simulator dtype and fills every row with the
 * model's current values (loader tables, b2sim_set_joint_friction edits, world gravity). The caller owns the rows: a write
 * on the simulator stream between runs acts from the next run on. b2sim_set_joint_friction and b2sim_set_gravity keep
 * their "every env" meaning and overwrite their column in every row. enable = 0 frees the buffers and the model returns to
 * the shared tables; pointers from b2sim_buffer taken before are then invalid. What stays nominal: the computed-torque
 * controller (the reference's ComputedTorqueFixedBase loads its own copy of the model file), the KinDyn queries
 * (b2sim_kindyn, b2sim_centroidal, b2sim_momentum_jacobian, b2sim_update_kinematics, b2sim_link_motion:
 * KinDynComputations is built from the model file), and the per-link inertial data of the loader (b2model_tables:
 * link_mass, link_com, which a wrench applied at a link's centre of mass uses): the rows describe lumped bodies, not
 * links, so a per-link centre of mass cannot be derived from them. B2_TASK_PANDA_REACH reads the rows too, on every
 * step that runs physics (b2sim_task_step, b2sim_task_rollout, steps replayed from a CUDA graph, b2sim_task_step_host);
 * its observation is kinematic, so b2sim_task_observe and b2sim_task_reset_all do not read them. To draw new parameters
 * per episode, write the rows of the envs whose B2_BUF_DONE is set (or all of them: the reach task only ends at its
 * TimeLimit, so its envs finish together unless B2_BUF_ELAPSED is staggered) after that step and before the next: the
 * terminal step ran with the old rows, the new episode runs with the new ones. B2_ERR_UNSUPPORTED for a free-floating
 * or static model, a model with a pendulum / cart-pole task, and a world with free bodies (also from b2sim_run when a
 * free body is inserted later); b2sim_set_task refuses a pendulum / cart-pole task on a model with per-env parameters. */
int b2sim_enable_env_params(b2sim* s, int model, int enable);
/* Per-env parameters of a world's free bodies and contacts (domain randomisation of the objects a robot manipulates and of
 * the surfaces they touch). Both entry points follow b2sim_enable_env_params: enable != 0 allocates the rows in the
 * simulator dtype, fills every row with the model's current values and returns the view in `out` (which may be NULL);
 * enabling rows that exist returns the same view and does not refill it. The caller owns the rows: a write on the
 * simulator stream between runs acts from the next unpaused run on. Nothing checks them on the device: they must stay
 * physically valid (mass > 0, a symmetric positive-definite inertia, mu >= 0). enable = 0 synchronises the stream and
 * frees the rows, and the model returns to the shared values; removing the model or destroying the simulator frees them
 * too, and views taken before are then invalid. Rows may be enabled before a free body is inserted: they are read once
 * the world has a contact stage, and they survive the rebuilds of the world description when other models are inserted or
 * removed. What stays nominal: gravity (the world's), the dynamics of an articulated model that shares the world with free
 * bodies (b2sim_enable_env_params refuses such a world), and the link-level inertial data of the loader (b2model_tables:
 * link_com, which a wrench applied at a link's centre of mass uses, and total_mass).
 *
 * Free-body rows: [N, 10] for a B2_KIND_FREE model: mass, centre of mass xyz in the root-link frame, inertia about the
 * centre of mass in root-link axes (xx xy xz yy yz zz), the record of one body of B2_BUF_BODY_INERTIA; every row starts
 * from body_mass, body_com and body_Ic of b2model_tables. B2_ERR_UNSUPPORTED for any other kind of model. */
int b2sim_enable_free_body_params(b2sim* s, int model, int enable, b2_buffer* out);
/* Friction rows: [N, nshapes], column k = the Coulomb friction coefficient of collision shape k of b2model_tables in each
 * env, starting from shape_mu[k]; for a free, static (ground plane, table) or articulated model (the finger pads). A
 * contact's coefficient is the smaller of its two shapes' values in that env. Columns of shapes the contact stage does not
 * use (cylinders, shapes beyond the per-body / per-model limits, shapes on links welded to the base) are kept and never
 * read. B2_ERR_UNSUPPORTED for a model without collision shapes. */
int b2sim_enable_shape_friction(b2sim* s, int model, int enable, b2_buffer* out);

/* ---- custom controller: ComputedTorqueFixedBase run by ControllerRunner -------------------------------- */
/* Model::insertModelPlugin("ControllerRunner", ...) with a <controller name="ComputedTorqueFixedBase"> context
 * (cpp/scenario/plugins/ControllerRunner/ControllerRunner.cpp:102-282, controllers/src/ComputedTorqueFixedBase.cpp:125-271):
 * every joint goes to Force mode; at the controller period tau = M(q)(ddq_ref - kp (q - q_ref) - kd (dq - dq_ref)) + h(q, dq)
 * is computed from the position / velocity / acceleration targets (all three must have been set) with the controller's
 * own gravity, and re-applied on every iteration in between. kp = NULL unloads the controller. */
int b2sim_set_computed_torque(b2sim* s, int model, const double* kp, const double* kd, const double gravity[3]);
/* Link::applyWorldWrench (Link.cpp:496-527): force and torque in the world frame at the link origin, applied on every
 * physics iteration until the post-step simulated time reaches now + duration (helpers.h:300-345). env = -1: every env. */
int b2sim_apply_link_wrench(b2sim* s, int model, int64_t env, int link, const double wrench[6], double duration);

/* ---- per-env scalar access (the ScenarI/O per-object view; synchronises the stream) --------------- */
enum {
    B2_FIELD_POSITION = 0,        /* Joint::position, Joint.cpp:643-651 */
    B2_FIELD_VELOCITY = 1,
    B2_FIELD_ACCELERATION = 2,
    B2_FIELD_FORCE = 3,           /* Joint::generalizedForce */
    B2_FIELD_FORCE_TARGET = 4,    /* Joint::{set,}generalizedForceTarget, Joint.cpp:774-815,1105-1116 */
    B2_FIELD_POSITION_TARGET = 5, /* Joint.cpp:683-729 */
    B2_FIELD_VELOCITY_TARGET = 6, /* Joint.cpp:731-772 */
    B2_FIELD_POSITION_RESET = 7,  /* Joint::resetPosition, Joint.cpp:132-155 (write only) */
    B2_FIELD_VELOCITY_RESET = 8,  /* Joint::resetVelocity, Joint.cpp:157-180 (write only) */
    B2_FIELD_ACCELERATION_TARGET = 9 /* Joint::{set,}accelerationTarget, Joint.cpp:731-772,839-846 */
};
int b2sim_get_joint(b2sim* s, int model, int field, int64_t env, int joint, double* value);
int b2sim_set_joint(b2sim* s, int model, int field, int64_t env, int joint, double value);
/* Link world pose (xyz + quat wxyz) of one env, Link.cpp:71-103. */
int b2sim_link_pose(b2sim* s, int model, int64_t env, int link, double pose[7]);

/* ---- free-floating bodies and contacts (SURVEY §8f-1) -------------------------------------------------- */
/* Model::resetBasePose / resetBaseWorldVelocity (Model.cpp:256-377): pose = xyz + quaternion wxyz, velocity =
 * world linear + angular (6). Consumed by the next run, paused or not. env = -1 addresses every env. */
int b2sim_set_base(b2sim* s, int model, int64_t env, int velocity, const double* values);
/* Model::basePosition / baseOrientation / baseWorld{Linear,Angular}Velocity of one env: 13 values. */
int b2sim_base_state(b2sim* s, int model, int64_t env, double state[13]);
/* Contacts of the last physics step in one env (Physics.cpp:2351-2540, Link.cpp:360-482). Returns the count;
 * ids[4k..] = model a, link a, model b, link b; data[10k..] = position, normal (from b to a), depth, force on a. */
int b2sim_contacts(b2sim* s, int64_t env, int max_contacts, int32_t* ids, double* data);

/* ---- zero-copy batched view ------------------------------------------------------------------------ */
int b2sim_buffer(b2sim* s, int model, int which, b2_buffer* out);

/* ---- fused task path: the env.step hot path for all envs in one launch ----------------------------- */
/* Attaches a task to a model: allocates obs/reward/done, stores the Philox seed and the global index of
 * env 0 (multi-GPU sharding: env e on this device is global env env_offset + e). B2_TASK_PANDA_REACH may be attached to a
 * model with per-env parameters (b2sim_enable_env_params, before or after); the pendulum / cart-pole tasks may not. */
int b2sim_set_task(b2sim* s, int model, int task, uint64_t seed, uint64_t env_offset,
                   int max_episode_steps);
/* Parameters of B2_TASK_PANDA_REACH (any pointer may be NULL, ee_link < 0 keeps the current one): reach goal in the
 * world frame, initial joint configuration restored by resets (models/panda.py:42-44), observed link. Call
 * before b2sim_task_reset_all. */
int b2sim_set_task_params(b2sim* s, int model, const double* goal, const double* q0, int ee_link);
/* Per-env domain randomisation of the pendulum / cart-pole tasks, the batched counterpart of
 * python/gym_ignition_environments/randomizers/cartpole.py:51-56,100-135 (SDF mass + U(-mass_delta, mass_delta) for
 * every link, gravity_z ~ N(g_z, gravity_sigma)): every reset draws new parameters for the env. Adds 8 (nq + 1) bytes
 * of read traffic per env-step. Call after b2sim_set_task; 0, 0 switches it off. */
int b2sim_set_task_randomization(b2sim* s, int model, double mass_delta, double gravity_sigma);
/* Task.reset_task + paused run for every env: samples fresh episode states on the device. */
int b2sim_task_reset_all(b2sim* s, int model);
/* Task.get_observation / get_reward / is_done on the current state of every env, without stepping: fills
 * B2_BUF_OBS / REWARD / DONE (what GazeboRuntime.reset returns after its paused run, gazebo_runtime.py:122-140). */
int b2sim_task_observe(b2sim* s, int model);
/* One GazeboRuntime.step for every env (gazebo_runtime.py:91-120): set_action -> run -> observation,
 * reward, done -> masked auto-reset. `actions` is a device pointer [N, nact] in the simulator dtype.
 * One kernel launch on the simulator stream; returns without synchronising. */
int b2sim_task_step(b2sim* s, int model, const void* actions_dev);
/* `steps` consecutive b2sim_task_step launches issued from C (no per-step host round trip): step t reads its
 * actions at actions_dev + t * action_stride elements (stride 0 repeats one action buffer). The launches can
 * be captured in a CUDA graph by the caller (set the capturing stream with b2sim_set_stream). */
int b2sim_task_rollout(b2sim* s, int model, const void* actions_dev, int steps, int64_t action_stride);
/* The same `steps` GazeboRuntime.step calls in ONE kernel launch (pendulum / cart-pole tasks): every env keeps its
 * state in registers across the steps, reading actions_dev[t, env] ([steps, N], simulator dtype) and, when the three
 * trajectory outputs are given, writing obs_traj [steps, N, nobs], reward_traj [steps, N], done_traj [steps, N]
 * (device pointers). B2_BUF_OBS / REWARD / DONE receive the last step. Same results as `steps` b2sim_task_step calls
 * (done masks, resets and step indices exactly, states to rounding); meant for open-loop action sequences (synthetic rollouts, replay), where one launch per step is launch-bound at
 * small env counts. */
int b2sim_task_trajectory(b2sim* s, int model, const void* actions_dev, int steps, void* obs_traj, void* reward_traj,
                          uint8_t* done_traj);
/* Same, through host buffers: copies actions host->device, steps, copies obs/reward/done back, and
 * synchronises. Host pointers may be pageable or pinned. */
int b2sim_task_step_host(b2sim* s, int model, const void* actions_host, void* obs_host,
                         void* reward_host, uint8_t* done_host);
int b2sim_task_nobs(int task);
int b2sim_task_nact(int task);
uint64_t b2sim_task_steps_done(const b2sim* s, int model);

/* Episode statistics accumulated inside the fused step kernels: totals = [sum of episode returns, sum of episode
 * lengths, finished episodes, non-finite rewards]. This is the only quantity of the path that crosses GPUs: an RL loop
 * sums it over ranks at the end of a rollout (SURVEY.md 5, metrics row; no reference counterpart below the Python
 * logging of its users, e.g. the Monitor wrapper around examples/python/launch_cartpole.py:32-75).
 * enable != 0 allocates and clears the accumulators (+ 2 scalars of traffic per env-step); 0 releases them.
 * b2sim_episode_stats_device returns the device pointer of the striped accumulators, B2_STAT_STRIPES rows of 4
 * doubles (sum the rows; a collective may reduce the whole block in place). b2sim_episode_stats reads the four
 * totals to the host (synchronises the stream) and optionally clears them. */
#define B2_STAT_STRIPES 32
int b2sim_episode_stats_enable(b2sim* s, int model, int enable);
int b2sim_episode_stats_device(b2sim* s, int model, void** totals_dev);
int b2sim_episode_stats(b2sim* s, int model, double totals[4], int clear);
/* Kernel launches issued by this simulator so far (bench.py reports it as gpu_launches). */
uint64_t b2sim_launch_count(const b2sim* s);

/* ---- KinDyn queries: replaces iDynTree KinDynComputations (rbd/idyntree/kindyncomputations.py) ----- */
/* Refreshes B2_BUF_LINK_POSE for every env from the current joint positions. */
int b2sim_update_kinematics(b2sim* s, int model);
/* Batched, fixed base, MIXED representation. out pointers are device buffers in the simulator dtype:
 *   mass_matrix [N, nq*nq] (kindyncomputations.py:270-277, joint block),
 *   bias_forces [N, nq]    (:292-303, C(q,dq)dq + g(q)),
 *   jacobian    [N, 6*nq]  (:367-377, rows linear then angular, joint columns) of `link`.
 * Any out pointer may be NULL. */
int b2sim_kindyn(b2sim* s, int model, int link, void* mass_matrix, void* bias_forces, void* jacobian);
/* Link::world{Linear,Angular}Velocity and world{Linear,Angular}Acceleration for every env (Link.cpp:206-294): device
 * buffers [N, 6] = linear(3), angular(3) of the link frame origin in the world orientation; the acceleration is the
 * classical one, from the joint accelerations of the last step. Either pointer may be NULL. */
int b2sim_link_motion(b2sim* s, int model, int link, void* twist, void* acceleration);
/* Centre-of-mass and momentum queries of KinDynComputations for every env
 * (python/gym_ignition/rbd/idyntree/kindyncomputations.py:305-342), device buffers in the simulator's dtype:
 *   com          [N, 3]    get_com_position (world)
 *   com_velocity [N, 3]    get_com_velocity (MIXED: world orientation)
 *   momentum     [N, 12]   get_momentum (linear, angular about the world origin), then get_centroidal_momentum
 *                          (linear, angular about the centre of mass), world orientation
 *   com_jacobian [N, 3*nq] joint columns of the centre-of-mass Jacobian
 * Any out pointer may be NULL. */
int b2sim_centroidal(b2sim* s, int model, void* com, void* com_velocity, void* momentum, void* com_jacobian);
/* Momentum Jacobian and locked inertia of KinDynComputations for every env
 * (python/gym_ignition/rbd/idyntree/kindyncomputations.py:379-427: get_linear_angular_momentum_jacobian,
 * get_centroidal_total_momentum_jacobian, get_average_velocity_jacobian, get_centroidal_average_velocity_jacobian;
 * :351-363 get_average_velocity, get_centroidal_average_velocity), in the frame iDynTree's MIXED representation uses for
 * the momentum (world orientation, origin at the model's base), device buffers in the simulator's dtype:
 *   momentum_jacobian [N, 6*nq] joint columns, rows linear(3) then angular(3) about the base origin
 *   locked_inertia    [N, 10]   composite inertia of the whole model about the base origin: rotational xx, xy, xz, yy,
 *                               yz, zz, first moment m c (3), mass; the 6x6 base block and the average-velocity
 *                               Jacobians follow from it (gym_ignition/rbd/kindyn.py)
 * Either pointer may be NULL. */
int b2sim_momentum_jacobian(b2sim* s, int model, void* momentum_jacobian, void* locked_inertia);

#ifdef __cplusplus
}
#endif
#endif /* B2SIM_H */
