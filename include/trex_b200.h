/*
 * trex_b200.h -- C ABI of libtrex_b200.so: a batched, B200-native replacement for the
 * trex-gym hot path.  Plain pointers and sizes only; no torch / C++ types.
 *
 * The reference is pure Python over pybullet and has no FFI of its own for this path; each
 * entry point below names the reference interface (file:line under /root/reference) whose
 * work it replaces.  INTEGRATION.md shows the ctypes stub a maintainer would add.
 *
 * Buffers are ROW-MAJOR PER ENVIRONMENT ("one record per env"): action [N][25], obs [N][75],
 * reward [N], done [N], state [N][TREX_STATE_DIM].  One warp steps one environment, lane k
 * touches element k of the record, so a record is one coalesced burst.  Joint order of
 * action/obs is the reference's: revolute joints sorted by name (trex_robot.py:311-314).
 *
 * Ownership: the caller (PyTorch) owns action/obs/reward/done/state buffers and passes raw
 * device pointers; the library owns the uploaded model and its internal environment records
 * and never allocates, frees or retains caller memory.  All launches are asynchronous on the
 * caller's stream (a cudaStream_t passed as void*; NULL = default stream) -- one kernel per substep runs
 * on a library-owned side stream that is forked from and joined back into the caller's stream with events,
 * so stream order (and CUDA-graph capture, tests/test_gpu_parity.py::test_cuda_graph_capture_of_a_step) of the caller
 * is preserved; only trex_get_stats, trex_step_host, trex_host_wait and trex_reset_host synchronise.
 *
 * Errors: 0 = success, negative = error; trex_last_error() returns the thread-local message.
 * Calls on one handle are not re-entrant; different handles may be created and used from different threads.
 */
#ifndef TREX_B200_H
#define TREX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TREX_NUM_JOINTS 25   /* action width; trex_robot.py:413-422 */
#define TREX_OBS_DIM 75      /* q | qd | applied motor torque; trex_robot.py:359-365 */
#define TREX_STATE_DIM 160   /* floats per environment record, layout below */
#define TREX_AUX_DIM 8

/* environment record (float32), identical to the oracle's state vector for [0,152):
 *   [0:3]   base COM position (world)            getBasePositionAndOrientation, trex_robot.py:322-328
 *   [3:7]   base quaternion x,y,z,w (base->world)
 *   [7:10]  base angular velocity (world)   [10:13] base linear velocity (world)
 *   [13:38] joint position, pybullet link order  [38:63] joint velocity
 *   [63:88] applied motor torque of the last substep
 *   [88:152] cached normal impulse per contact candidate (solver warm start)
 *   [152] steps in the current episode  [153] episodes started  [154] NaN-guard resets
 *   [155:158] per-step accumulators (PGS iterations, contacts, contact overflow)
 *   [158] active-set signature of the last env step: a 24-bit hash (stored as an exact float) over, per physics substep, the
 *         contact candidates with rows, the limit rows / normal rows that ended with a positive impulse, the motors and
 *         friction pairs that ended on their bounds and the PGS iterations executed -- equal signatures of kernel and
 *         oracle mean both solved the same complementarity problem (tests/test_active_set_parity.py)  */

#define TREX_OK 0
#define TREX_ERR_INVALID (-1)
#define TREX_ERR_CUDA (-2)
#define TREX_ERR_MODEL (-3)

typedef struct trex_handle trex_handle;

#define TREX_SOLVE_DEFAULT 0
#define TREX_SOLVE_FRONT 1
#define TREX_SOLVE_FREE_ONLY 2
#define TREX_SOLVE_NO_HEAVY 3
#define TREX_HEAVY_BOTH 0
#define TREX_HEAVY_SHARED 1
#define TREX_HEAVY_TENSOR 2
#define TREX_CONTACT_TENSOR 0
#define TREX_CONTACT_SHARED 1
#define TREX_ACTUATION_POSITION 0
#define TREX_ACTUATION_TORQUE 1

typedef struct trex_config {
  int32_t num_substeps;      /* trex_env.py:18 NUM_SUBSTEPS (5); dt = 0.01/n, iterations = int(300/n)  (:71-73) */
  float distance_weight;     /* trex_env.py:42 */
  float energy_weight;       /* trex_env.py:43 */
  float drift_weight;        /* trex_env.py:44 */
  int32_t max_episode_steps; /* 0 = never terminate, the reference behaviour (trex_env.py:183-184) */
  int32_t enable_contacts;   /* 1 = floor contact on the derived candidate points; 0 = the literal
                                collision-less URDF of the reference (free fall) */
  int32_t reset_mode;        /* 0 = reference reset pose (trex_env.py:81-87,105-109); 1 = fallen-start sampler
                                (BASELINE configs[4]: base z U(0.3,3), uniform SO(3), joints U(limits); no
                                reference counterpart), Philox keyed by (seed, global env id, episode) */
  uint32_t seed;
  int64_t env_offset;        /* global id of environment 0 of this shard (multi-GPU: rank * n_envs); keys the reset sampler so
                                results do not depend on the number of GPUs */
  int32_t warps_per_block;   /* warps per CTA of the front / tail kernels: 1, 2 or 4; 0 = default (2).  With 4 the inward pass of
                                the CTA's four environments runs on one warp, eight lanes per environment (bit-identical) */
  int32_t solver_placement;  /* where a physics substep's constraint solve runs (results agree to FP32 round-off; diagnostics):
                                TREX_SOLVE_DEFAULT   contact-free substeps and substeps with <= 8 contacts: four environments per
                                                     warp (trex_solve_kernel); more contacts: trex_heavy_kernel
                                TREX_SOLVE_FRONT     everything inside the front kernel (one environment per warp)
                                TREX_SOLVE_FREE_ONLY only contact-free substeps are deferred
                                TREX_SOLVE_NO_HEAVY  as DEFAULT, but more than 8 contacts stay in the front kernel */
  int32_t heavy_share_div;   /* > 0: environments with 9-16 contacts go to trex_heavy_kernel only while at most
                                n_envs / heavy_share_div of the batch were in that class in the previous substep (1 = always);
                                0 = default: always (the routing then depends on the environment alone, never on its batch) */
  int32_t pipelines;         /* the batch is stepped as this many independent groups of environments, each a chain of kernels on
                                its own stream, so that one group's latency-bound solvers overlap another group's issue-bound
                                dynamics kernel (results do not depend on it): 1..8; 0 = default (2 from 8,192 environments) */
  int32_t heavy_memory;      /* where the many-contact solver (9-16 contacts, two environments per warp) keeps its 48 x 48 Delassus
                                matrices: TREX_HEAVY_BOTH (default) runs two kernel instances concurrently on one task list -- one with
                                the matrices in TENSOR MEMORY (tcgen05.st / tcgen05.ld as a per-lane scratchpad, 8 warps per SM), one
                                with them in shared memory (fills the shared memory left: 4 more warps per SM);
                                TREX_HEAVY_SHARED / TREX_HEAVY_TENSOR run one of them alone.  Results are bit-identical. */
  int32_t chunk_envs;        /* L2-resident work records: every group of `pipelines` walks its share of the batch in chunks of this many
                                environments (multiple of 4) -- all substeps of a chunk before the next one -- and reuses the same
                                work-record slots, so the 4.6-11.4 KB per environment and substep that the dynamics kernel hands to
                                the solvers stay in the 126 MB L2 instead of crossing HBM twice (results do not depend on it).
                                0 or -1 = off (default: one chunk per group; measured 6 % faster, HBM is at 7 % of its bandwidth either way) */
  int32_t contact_memory;    /* where the contact solver (1-8 contacts, four environments per warp) keeps its Delassus blocks and the
                                responses of each lane's own contact along the sweep: TREX_CONTACT_TENSOR (default) in TENSOR MEMORY
                                (persistent 4-warp CTAs, tcgen05.ld 32x32b as a lane-private scratchpad: the shared-memory instance
                                runs at 69 % of the shared-memory data pipe's wavefront peak), TREX_CONTACT_SHARED in shared memory.
                                Results are bit-identical. */
  int32_t env_params;        /* 0 (default): every environment simulates the model's own constants.  1: the handle owns a
                                per-environment parameter record (trex_set_env_params below) and runs the kernel instances that
                                read it; rows start as the model's constants, which reproduce the env_params = 0 results bit for bit */
  int32_t external_forces;   /* 0 (default): gravity is the only external load.  1: the handle owns a per-environment record of
                                external wrenches on the bodies (trex_set_external_forces below) and an optional push schedule, and
                                runs the dynamics-kernel instances that read them; the record starts at zero, which reproduces the
                                external_forces = 0 results bit for bit */
  int32_t actuation;         /* what an action is (any other value: TREX_ERR_INVALID):
                                TREX_ACTUATION_POSITION (0, default): a motor target, clipped to the joint limits (the reference's
                                  trex_robot.set_actions; the motors bound the impulse by max_torque * dt).
                                TREX_ACTUATION_TORQUE (1): joint torque control (pybullet's setJointMotorControlArray(TORQUE_CONTROL,
                                  forces=tau) after VELOCITY_CONTROL with forces 0; Isaac Gym's DOF actuation-force tensor).
                                  Action slot i (name-sorted) is the torque in N m on joint obs_dof[i], clipped to [-T, T] with T the
                                  model's motor_max_torque (env_params = 1: the environment's row element [29]; elements [27] and
                                  [28] are then ignored and the library keeps [30] at 0).  A NaN command is clipped to -T
                                  (as a NaN target becomes the lower joint limit in position mode): pass finite torques.  It acts in EVERY physics substep of the
                                  step, as an explicit joint torque next to pybullet's joint damping: Q = tau - d qd.  The motor
                                  rows stay with kp = kd = 0 and impulse bound 0 (as in a reset step); joint limits, contacts,
                                  damping, wrenches and pushes are unchanged.  Reset steps (trex_reset, the auto-reset) apply no
                                  torque, as in position mode.  The applied joint torque that record [63:88], observation [50:75]
                                  and the reward's energy term sum |qd tau| report is the CLIPPED COMMAND -- a deliberate
                                  difference from pybullet, whose getJointState reports the motor's impulse / dt, i.e. 0 in torque
                                  control (as far as we know), which would silently drop the reference's energy penalty.
                                  trex_get_action_limits gives the bounds; trex_fill_random_actions draws U(-T, T). */
  int32_t reserved[4];       /* must be zero */
} trex_config;

typedef struct trex_stats {
  int64_t env_steps;         /* environment steps executed since creation */
  int64_t episodes;          /* episodes started (resets) */
  int64_t nan_resets;        /* environments reset by the NaN guard */
  double mean_solver_iterations; /* PGS iterations per substep, last step */
  double mean_contacts;      /* active contact points per environment, last step */
  int64_t contact_overflow;  /* contact points dropped (more than the per-env capacity), last step */
} trex_stats;

/* Replaces TrexBulletEnv.__init__ + loadURDF (trex_env.py:39-96, trex_robot.py:47-56) for n_envs
 * environments on CUDA device `device`.  model_blob = bytes produced by
 * trex_gym_b200.model_compiler (URDF parsed by the reference's tools/urdf_parsing.py:237-239). */
int trex_create(const void* model_blob, size_t bytes, int32_t n_envs, int32_t device, const trex_config* cfg,
                trex_handle** out);
void trex_destroy(trex_handle* h);

/* TrexBulletEnv.reset (trex_env.py:98-122): reset pose, zero-gain motors, one physics step, obs.
 * mask_dev: optional uint8[N] on the device; only environments with mask != 0 are reset and have
 * their obs row written.  obs_dev may be NULL. */
int trex_reset(trex_handle* h, const uint8_t* mask_dev, float* obs_dev, void* stream);

/* TrexBulletEnv.step (trex_env.py:128-154) for all environments: clip, n substeps of
 * (set_actions; stepSimulation) (trex_robot.py:413-422), observations (trex_robot.py:359-365),
 * reward (trex_env.py:186-196), done (trex_env.py:183-184; plus optional horizon / NaN guard with
 * VecEnv-style auto-reset: a done environment is reset and its obs row is the reset observation). */
int trex_step(trex_handle* h, const float* action_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev,
              void* stream);

/* Same step with HOST buffers (the reference-facing call: numpy in, numpy out): copies the actions to the device, steps,
 * copies obs/reward/done back and synchronises.  Runs on library-owned non-blocking streams (not the legacy default stream);
 * a caller mixing it with device-pointer calls on its own stream must synchronise that stream first. */
int trex_step_host(trex_handle* h, const float* action_host, float* obs_host, float* reward_host,
                   uint8_t* done_host);
/* The same as a depth-1 pipeline, for callers that alternate between two sets of (pinned) host arrays: the host->device
 * copy runs on a second stream under the previous step's kernels and the device->host copies on a third stream, behind
 * events, under the next step's kernels (two internal sets of staging buffers).  Contract: when call k returns, the
 * outputs of call k-1 are complete in host memory; the arrays passed to call k (action included) must stay untouched
 * until call k+1 has returned or trex_host_wait() has.  trex_host_wait() drains everything outstanding. */
int trex_step_host_async(trex_handle* h, const float* action_host, float* obs_host, float* reward_host,
                         uint8_t* done_host);
int trex_host_wait(trex_handle* h);
int trex_reset_host(trex_handle* h, float* obs_host);

/* Simulator-state checkpoint / parity hooks: copy the environment records out / in (device pointers). */
int trex_get_state(trex_handle* h, float* state_dev, void* stream);
int trex_set_state(trex_handle* h, const float* state_dev, void* stream);
/* Per-environment dynamics parameters (handles created with trex_config.env_params = 1; TREX_ERR_INVALID otherwise).
 * The record is float32 [N][TREX_ENV_PARAM_DIM], one row per environment; each element replaces, for that environment only,
 * what a pybullet client sets with the call named beside it:
 *   [0:25]  mass scale of the body of joint k (pybullet link order, fixed links merged in)   changeDynamics(mass=, localInertiaDiagonal=)
 *   [25]    mass scale of the base body                                                        changeDynamics(-1, mass=, localInertiaDiagonal=)
 *           (uniform density scaling: mass, first moment, inertia, angular-damping tensor and link-damping masses; the COM stays)
 *   [26]    friction coefficient of the foot-floor contacts (the combined value)               changeDynamics(lateralFriction=)
 *   [27]    motor position gain kp, [28] velocity gain kd                                      setJointMotorControlArray(positionGains=, velocityGains=)
 *   [29]    motor max torque, N m                                                              setJointMotorControlArray(forces=)
 *   [30]    motor impulse bound = [29] * dt, computed in double by the library (the value passed is ignored)
 *   With TREX_ACTUATION_TORQUE: [27] and [28] are ignored, [29] is the bound the torque command is clipped to, and the library
 *   keeps [30] at 0 (the motors have no strength) on create, on a set and on every randomized reset.
 *   [31]    reserved, 0
 * Defaults (every row after trex_create): scales 1, then the model's friction, motor_kp, motor_kd, motor_max_torque.  Reset
 * steps keep zero motor gains, as with env_params = 0; mass scales and friction apply to them.
 * trex_get_state / trex_set_state do not carry the record: a checkpoint saves it with trex_get_env_params. */
#define TREX_ENV_PARAM_DIM 32
/* rows of params_dev [N][32] (device) -> the record: all rows, or (mask_dev uint8[N] on the device, optional) those with
 * mask != 0; element 30 is recomputed.  Stream ordered, capturable. */
int trex_set_env_params(trex_handle* h, const float* params_dev, const uint8_t* mask_dev, void* stream);
int trex_get_env_params(trex_handle* h, float* params_dev, void* stream);
/* Randomizer (domain randomization): while set, every reset of an environment -- trex_reset (masked too) and the auto-reset on
 * done -- first draws its row: element k = lo[k] + u (hi[k] - lo[k]), u in [0,1) from Philox4x32-10 keyed by the seed and
 * counted by (env_offset + env, episode, k / 4), so rows do not depend on the number of GPUs and lo == hi gives lo exactly;
 * element 30 follows from the drawn 29.  Host arrays of 32 floats: lo <= hi, finite, mass scales > 0, friction, gains and
 * torque >= 0, elements 30 and 31 zero.  NULL / NULL turns the randomizer off.  Synchronises the device (resets already
 * enqueued use the previous ranges); a CUDA graph keeps the setting it was captured with. */
int trex_set_env_param_ranges(trex_handle* h, const float* lo32_host, const float* hi32_host);

/* External forces and torques on the bodies (handles created with trex_config.external_forces = 1; TREX_ERR_INVALID
 * otherwise): what pybullet's applyExternalForce(robot, link, F, linkWorldCOM, WORLD_FRAME) and
 * applyExternalTorque(robot, link, T, WORLD_FRAME) do, summed over the links of a merged body.
 * The user layout is float32 [N][TREX_EXT_BODIES][6]: body k < 25 is the body moved by joint k (pybullet link order, fixed
 * links folded in), body 25 the base -- the order of an env-param row.  A wrench is [fx fy fz tx ty tz] in the world
 * frame (N, N m): the force acts at the body's centre of mass (the composite COM of the merged body; a mass scale leaves it
 * unchanged), the torque is a free vector.
 * PERSISTENCE DIFFERS FROM PYBULLET: pybullet clears external forces after every stepSimulation; here the record stays until
 * it is set again.  It acts in every physics substep of every trex_step / trex_step_host*, never in the physics step of a
 * reset (trex_reset and the auto-reset), and survives resets.  trex_get_state / trex_set_state do not carry it. */
#define TREX_EXT_BODIES 26
/* wrench_dev [N][26][6] (device) -> the record: all environments, or (mask_dev uint8[N] on the device, optional) those with
 * mask != 0; every wrench of such an environment is replaced.  Stream ordered, capturable. */
int trex_set_external_forces(trex_handle* h, const float* wrench_dev, const uint8_t* mask_dev, void* stream);
int trex_get_external_forces(trex_handle* h, float* wrench_dev, void* stream);
/* Push schedule: a horizontal push on one body, added to the record's force of that body while active.  Stateless: at env
 * step t of episode e (steps completed in the episode when the step starts) of environment gid = env_offset + env, window
 * w = t / interval draws u0..u3 from Philox4x32-10 keyed by the seed, counted by (gid, e, w), so pushes depend neither on
 * the number of GPUs nor on when the schedule was set.  The window holds a push iff u0 < probability; it starts
 * o = min(floor(u1 (interval - duration + 1)), interval - duration) steps into the window and lasts `duration` steps, and
 * no push acts before step first_step.  Magnitude force_min + u2 (force_max - force_min) N, direction one of 32 horizontal
 * unit vectors, index floor(32 u3), angle 2 pi index / 32 from the world x axis. */
typedef struct trex_push_schedule {
  int32_t body;              /* 0..25, numbered as above (25 = base) */
  int32_t interval;          /* >= 1 env steps per window */
  int32_t duration;          /* 1..interval env steps of a push */
  int32_t first_step;        /* >= 0: no push before this step of an episode */
  float probability;         /* [0, 1]: chance that a window holds a push */
  float force_min, force_max;  /* 0 <= force_min <= force_max, finite (N) */
  int32_t reserved[9];       /* must be zero */
} trex_push_schedule;
/* s_host NULL turns the schedule off.  The schedule is a kernel argument: it applies to the steps enqueued after the call,
 * and a CUDA graph keeps the schedule it was captured with. */
int trex_set_push_schedule(trex_handle* h, const trex_push_schedule* s_host);

/* World state of every body and the floor's contact force on it, computed on the device from the environment records (what
 * pybullet's getLinkState(robot, link, computeLinkVelocity=1) / getBasePositionAndOrientation / getBaseVelocity and the
 * summed getContactPoints(robot, floor)[9] give; Isaac Gym's rigid-body-state and net-contact-force tensors).  Works on every
 * handle; reads the records only (the step's results are unchanged); stream ordered, capturable.  Either output may be NULL,
 * not both (TREX_ERR_INVALID).  Bodies are numbered as in the wrench record: body k < 25 is the body moved by joint k
 * (pybullet link order, fixed links folded in), body 25 the base.
 *   states_dev [N][26][TREX_BODY_STATE_DIM] float32, all in the world frame:
 *     [0:3]   p: the body's centre of mass (the composite COM of the merged body, where an external force acts; a mass scale
 *             leaves it unchanged)
 *     [3:7]   q: body frame -> world rotation, x y z w.  The body frame of body k < 25 is its joint frame re-oriented so that
 *             the joint axis is +z (DESIGN.md section 2) -- NOT pybullet's link frame, which is the link's inertial frame;
 *             its quaternion comes from the rotation matrix with w >= 0.  The base's frame is the base link's inertial frame
 *             (pybullet's base pose); its row holds the record's [3:7] bit for bit, sign included
 *     [7:10]  v: linear velocity of the COM        [10:13] w: angular velocity (the base's: the record's [7:10] bit for bit)
 *   contact_force_dev [N][26] float32: the floor's NORMAL force on the body in the last physics substep (N): the sum over the
 *     body's contact candidates, in ascending candidate index, of record[88 + c] / dt_substep (sequential, unfused float32),
 *     i.e. pybullet's getContactPoints(robot, floor)[9] summed over the body's links after stepSimulation.  After a reset (or
 *     an auto-reset) it is that of the reset's physics step; 0 with enable_contacts = 0.  Friction forces are not kept in the
 *     record and are not reported. */
#define TREX_BODY_STATE_DIM 13
int trex_get_body_states(trex_handle* h, float* states_dev, float* contact_force_dev, void* stream);

/* Joint-space mass matrix, bias forces and body Jacobians, computed on the device from the environment records (pybullet's
 * calculateMassMatrix, calculateInverseDynamics with zero accelerations and calculateJacobian at every body's COM; Isaac
 * Gym's mass-matrix and Jacobian tensors).  Works on every handle; reads the records only (the step's results are
 * unchanged); stream ordered, capturable.  Any output may be NULL, not all three (TREX_ERR_INVALID); a NULL output is not
 * computed.  With trex_config.env_params = 1 the environment's mass scales apply (mass, first moment and inertia).
 *   Generalized velocity u [TREX_NUM_DOFS] -- the record's own velocity layout:
 *     u[0:3]  = record [7:10]:  base angular velocity, world frame
 *     u[3:6]  = record [10:13]: velocity of the base link's COM (the record's position [0:3], the origin of the base frame),
 *               world frame.  The merged base body (body 25 below) also holds the links fixed to the base, so its COM is
 *               elsewhere
 *     u[6:31] = record [38:63]: joint rates in pybullet link order (TrexBatchSim.dof_names()), NOT the name-sorted
 *               action / observation order: action slot i drives joint obs_dof[i] (model section obs_dof), whose rate is
 *               u[6 + obs_dof[i]]
 *   mass_matrix_dev [N][31][31] float32: M with kinetic energy = 1/2 u^T M u; stored full and exactly symmetric (one triangle
 *     is computed and mirrored)
 *   bias_dev [N][31] float32: b with M du/dt + b = tau, du/dt the time derivative of u in the coordinates above: gravity plus
 *     the Coriolis and centrifugal terms.  b does NOT contain link or joint damping, motors, joint limits, contacts or the
 *     external-wrench record.  In particular a torque-mode step (TREX_ACTUATION_TORQUE) adds the joint damping -d qd to the
 *     commanded torque, which b leaves out: a computed-torque controller adds d qd itself.  The generalized force tau of u[0:6] is the torque about the base link's COM, then the force
 *     (world).  Joint torques of given accelerations: tau = M du/dt + b, in torch (M @ udot[..., None])[..., 0] + b
 *   jacobian_dev [N][26][TREX_JACOBIAN_ROWS][31] float32: J_k of body k (numbered as in the wrench record and
 *     trex_get_body_states: body k < 25 is the body moved by joint k, body 25 the base), rows [v_COM (3); w (3)] in the world
 *     frame, linear first: J_k u = states[k][7:13] of trex_get_body_states.  The point is the body's COM as in the wrench
 *     record and the body states (the composite COM of the merged body), so sum_k J_k^T [f_k; t_k] is the generalized force
 *     of a wrench record.  A point p of body k moves with v_p = v_COM + w x (p - COM). */
#define TREX_NUM_DOFS 31
#define TREX_JACOBIAN_ROWS 6
int trex_get_dynamics(trex_handle* h, float* mass_matrix_dev, float* bias_dev, float* jacobian_dev, void* stream);

/* per-env diagnostics of the last step: head xyz (trex_robot.py:330-335), the three penalty terms
 * logged at trex_env.py:193-195 (lifting, station keeping, energy), PGS iterations, contacts. */
int trex_get_aux(trex_handle* h, float* aux_dev, void* stream);

/* action/observation limits in name-sorted joint order (trex_robot.py:337-357, 424-433); host pointers.  The observation
 * space uses them in either actuation mode. */
int trex_get_joint_limits(trex_handle* h, float* lower25_host, float* upper25_host);
/* the action space in name-sorted joint order: the joint limits with TREX_ACTUATION_POSITION, -T / +T with
 * TREX_ACTUATION_TORQUE (T = the model's motor_max_torque; per-environment bounds of env_params rows are not reflected);
 * host pointers */
int trex_get_action_limits(trex_handle* h, float* lo25_host, float* hi25_host);

/* Synthetic benchmark input: action[i][k] ~ U(lo_k, hi_k) of trex_get_action_limits, from a counter-based generator keyed by
 * (seed, env_offset + i, step), so streams do not depend on the number of GPUs. */
int trex_fill_random_actions(trex_handle* h, float* action_dev, uint32_t seed, uint64_t step, int64_t env_offset,
                             void* stream);

int trex_get_stats(trex_handle* h, trex_stats* out); /* synchronises the device */
/* Measurement aid (no reference counterpart): register-resident FFMA microbenchmark, best of 5, in
 * TFLOP/s -- the FP32 CUDA-core roofline denominator for this path.  Synchronises. */
int trex_measure_fp32_peak(int32_t device, double* tflops_out);
/* Rollout post-processing for the caller of the path (trex_train.py:49-61 -> baselines ppo2.Runner [RECALL]); buffers
 * are time-major [T][N] on the device.  done_dev[t] = episode-start flag of the state step t acted in, last_done closes it.
 *   A_t = delta_t + gamma*lam*(1-done_{t+1})*A_{t+1},  delta_t = r_t + gamma*V_{t+1}*(1-done_{t+1}) - V_t,  ret = A + V  */
int trex_gae(int32_t device, const float* reward_dev, const float* value_dev, const uint8_t* done_dev, const float* last_value_dev,
             const uint8_t* last_done_dev, float gamma, float lam, float* adv_dev, float* ret_dev, int32_t T, int32_t N, void* stream);
/* baselines VecNormalize (trex_train.py:45): out = clip((x - mean) / sqrt(var + eps), -clip, clip), x [n_rows][dim] */
int trex_normalize(int32_t device, const float* x_dev, const float* mean_dev, const float* var_dev, float eps, float clip,
                   float* out_dev, int64_t n_rows, int32_t dim, void* stream);
/* Fused policy / value forward of the rollout loop (SURVEY 8f; what baselines ppo2 evaluates per env step around
 * TrexBulletEnv.step, trex_train.py:48,107 [RECALL MlpPolicy]): observation filter (ob_mean/ob_var NULL = identity), two tanh
 * trunks 75 -> 64 -> 64, Gaussian-mean head (25) with state-independent log-std, value head (1);
 * action = mean + exp(logstd) * eps with eps ~ N(0,1) from Philox keyed by (seed, env_offset + row, step) (deterministic != 0:
 * action = mean), neglogp = 0.5 sum eps^2 + sum logstd + 0.5 D log(2 pi).  params_dev: trex_policy_param_count() floats,
 * row-major [in][out]:  pi W1[75][64] b1[64] W2[64][64] b2[64] Wo[64][25] bo[25] | vf W1 b1 W2 b2 Wo[64][1] bo[1] | logstd[25].
 * obs_dev [n_rows][75] is read in place; neglogp_dev, value_dev, mean_dev (the Gaussian means [n_rows][25]) may be NULL. */
int trex_policy_param_count(void);
int trex_policy_forward(int32_t device, const float* obs_dev, const float* ob_mean_dev, const float* ob_var_dev, float eps, float clip,
                        const float* params_dev, uint32_t seed, uint64_t step, int64_t env_offset, int32_t deterministic,
                        float* action_dev, float* neglogp_dev, float* value_dev, float* mean_dev, int64_t n_rows, void* stream);
int64_t trex_kernel_launches(const trex_handle* h);  /* kernels launched by this handle so far */
int32_t trex_num_envs(const trex_handle* h);
const char* trex_last_error(void);
const char* trex_version(void);

#ifdef __cplusplus
}
#endif
#endif
