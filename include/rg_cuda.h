/*
 * rg_cuda.h -- C ABI of the B200 (sm_100a) batched locomotion-controller library.
 *
 * This is the drop-in boundary for robot-gym's per-control-step MPC locomotion path.
 * The reference has NO native code of its own on this path; the only native boundaries
 * it crosses are third-party:
 *
 *   - pybind11 `mpc_osqp.ConvexMpc(mass, inertia[9], num_legs, horizon, dt, weights[13],
 *     alpha)` + `.compute_contact_forces(...)` of motion_imitation==0.0.5, reached from
 *     robot_gym/controllers/mpc/mpc_controller.py:47-56 (constructor arguments) and
 *     :102-106 (one solve per get_action());
 *   - PyBullet `calculateInverseKinematics` (robot_gym/controllers/mpc/kinematics.py:91-92)
 *     and `calculateJacobian` (robot_gym/controllers/mpc/kinematics.py:25-27).
 *
 * Each entry point below names the reference interface it replaces.  All data pointers
 * are DEVICE pointers owned by the caller (PyTorch in the bundled host code) unless the
 * name ends in `_host`.  Arrays are env-major, C-contiguous.  The library allocates no
 * persistent device memory, never synchronises the host (except rg_mpc_setup /
 * rg_robot_setup, which are one-time table uploads), launches on the given stream
 * (`stream` is a cudaStream_t passed as void*; NULL = legacy default stream) and is
 * re-entrant across streams as long as workspaces and outputs are disjoint.
 *
 * Every function returns 0 on success or a negative RG_ERR_* code; rg_last_error()
 * returns a thread-local description of the last failure.
 */
#ifndef RG_CUDA_H_
#define RG_CUDA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RG_NUM_LEGS 4
#define RG_MOTORS_PER_LEG 3
#define RG_NUM_MOTORS 12
#define RG_ACTION_DIM 60          /* 12 motors x (q, kp, qdot, kd, tau): simple_motor.py:15-22 */
#define RG_MAX_HORIZON 20
#define RG_VEL_WINDOW_MAX 64

enum {
  RG_OK = 0,
  RG_ERR_BAD_ARG = -1,        /* NULL pointer, negative size, bad enum */
  RG_ERR_UNSUPPORTED = -2,    /* horizon / num_legs / window the kernels are not built for */
  RG_ERR_SINGULAR = -3,       /* MPC weights leave a state channel unpenalised (K not SPD) */
  RG_ERR_WORKSPACE = -4,      /* workspace too small or not prepared by the setup call */
  RG_ERR_CUDA = -5            /* CUDA runtime / launch failure (message has the cuda string) */
};

/* LegState of motion_imitation's gait_generator (ghost/ctrl_constants.py:3,32-37). */
enum { RG_LEG_SWING = 0, RG_LEG_STANCE = 1, RG_LEG_EARLY_CONTACT = 2, RG_LEG_LOSE_CONTACT = 3 };

/* solve_info[n][0..3] */
enum { RG_INFO_IPM_ITERS = 0, RG_INFO_POLISH_ROUNDS = 1, RG_INFO_STATUS = 2, RG_INFO_NUM_ACTIVE = 3 };
/* status bits */
enum {
  RG_STATUS_POLISHED = 1,        /* active-set polish verified (exact KKT point of the QP) */
  RG_STATUS_IPM_CONVERGED = 2,   /* interior-point residual below tolerance */
  RG_STATUS_NO_STANCE = 4,       /* no foot in contact: all forces are zero by the bounds */
  RG_STATUS_NUMERIC = 8,         /* non-positive pivot met (result is the last good iterate) */
  RG_STATUS_ACTIVE_SET_ONLY = 16,/* the cold-start active-set iteration verified; no interior point ran */
  RG_STATUS_BAD_WORKSPACE = 32,  /* the workspace on the device is not the one rg_mpc_setup prepared for this horizon
                                    (freed / overwritten without rg_mpc_release): forces are zero, nothing was solved */
  RG_STATUS_BAD_MODEL = 64       /* this env's row of the rg_mpc_env_model fails the checks rg_mpc_setup makes (mass > 0
                                    and finite, inertia finite and invertible, friction coefficients > 0): forces and
                                    horizon outputs are zero, the warm-start set is reset, nothing was solved */
};
/* A row of an rg_gait_env_params (below) that is not valid has no status bit: the control step holds every leg of
 * that env in stance -- desired_leg_state = leg_state = RG_LEG_STANCE, mpc_contact_state = 1, normalized_phase = -1.0
 * (a value a valid row never produces: t >= 0 and the phase lies in [0, 1)), no swing target, last_leg_state = STANCE
 * -- so the env stands on the stance solve.  The other envs of the batch are not affected. */

/* ---- ConvexMpc constructor arguments + the constants compiled into mpc_osqp ------------
 * Replaces: mpc_osqp.ConvexMpc(...) as constructed by TorqueStanceLegController
 * (call site robot_gym/controllers/mpc/mpc_controller.py:47-56; mass/inertia from
 * robot_gym/model/robots/ghost/ctrl_constants.py:8-9).  State/weight order:
 * (roll,pitch,yaw, x,y,z, wx,wy,wz, vx,vy,vz, g). */
typedef struct rg_mpc_params {
  double mass;
  double inertia[9];           /* body-frame inertia, row major */
  int32_t num_legs;            /* must be 4 */
  int32_t horizon;             /* 5, 10 or 20 planning steps */
  double dt;                   /* planning time step [s] */
  double weights[13];
  double alpha;                /* force regulariser (1e-5) */
  double friction_coeffs[4];   /* indexed by pyramid ROW, as mpc_osqp does (see DESIGN.md) */
  double gravity;              /* 9.8 */
  double fz_max;               /* mass*g*10  */
  double fz_min;               /* mass*g*0.1 */
  double desired_body_height;  /* desired_com_position[2] */
  /* solver controls (not in the reference: OSQP eps/polish have no equivalent here) */
  double ipm_tol;              /* relative residual at which the interior point hands over (1e-6) */
  int32_t max_ipm_iters;       /* hard cap (40) */
  int32_t max_polish_rounds;   /* rounds per attempt (3); 0 disables the verified active-set rounds:
                                  the interior point alone leaves ~1e-3 relative in the alpha-directions */
  int32_t cold_start_rounds;   /* active-set rounds tried from the guessed / warm-started set BEFORE the interior
                                  point (12); 0 = always run the interior point first */
  int32_t cold_start_max_violations; /* > 0: hand over to the interior point at once when the first round finds
                                  more violated friction-cone rows than this; 0 (default) = no limit */
  int32_t two_kernel_solve;    /* 1 (default): a lean active-set-only kernel solves every env and queues the ones its
                                  rounds cannot verify; the complete solver (interior point, escalation) then runs on
                                  that list only (launched programmatically behind the first kernel, so that its
                                  launch latency hides behind the first grid's tail).  0: one kernel with the complete
                                  solver for every env.  Same results either way; needs cold_start_rounds > 0 and a
                                  workspace sized for n_env. */
  int32_t reserved_;
} rg_mpc_params;

/* Fill `p` with the motion_imitation defaults for the given mass/inertia/height. */
int rg_mpc_default_params(rg_mpc_params* p_host, double mass, const double* inertia9_host,
                          double desired_body_height, int horizon);

/* Bytes of device workspace rg_mpc_setup needs: parameter block + horizon tables, plus the fallback queue of the
 * two-kernel solve for batches of up to n_env envs (4 bytes per env).  A solve of more envs than the workspace was
 * sized for still works: it uses the single complete kernel. */
int rg_workspace_bytes(int n_env, int horizon, int num_legs, size_t* bytes_host);

/* One-time: validates params, computes the horizon tables on the host and uploads them plus
 * the parameters into `workspace` (256-byte aligned).  Synchronises `stream`.  A workspace serves one solve at a
 * time: concurrent solves on different streams need a workspace each (the queue lives in it). */
int rg_mpc_setup(const rg_mpc_params* p_host, void* workspace, size_t workspace_bytes, void* stream);

/* Forget a workspace prepared by rg_mpc_setup (call before freeing or reusing its memory). */
int rg_mpc_release(const void* workspace);

/* Replaces: ConvexMpc.compute_contact_forces(com_position=[0], com_velocity, rpy,
 * angular_velocity, foot_contact_states, foot_positions_base_frame, friction, desired...)
 * as called by TorqueStanceLegController.get_action (mpc_controller.py:47-56,105).
 * One QP per env: builds the condensed centroidal QP over the horizon and solves it.
 *   com_velocity_body  [N,3]  f32   state estimator body-frame COM velocity
 *   base_rpy           [N,3]  f32   roll, pitch, yaw.  The yaw is used AS GIVEN: TorqueStanceLegController passes a
 *                                   yaw-aligned attitude (yaw = 0); rg_control_step zeroes it itself, a direct caller
 *                                   of this entry point (or of robot_gym.cuda.mpc_build_solve) must do so too
 *   base_rpy_rate      [N,3]  f32   Robot.GetBaseRollPitchYawRate (robot.py:205-213)
 *   foot_contact_state [N,4]  u8    1 = planned stance (held over the horizon; see rg_mpc_build_solve_schedule for
 *                                   a per-step plan); 4-byte aligned
 *   foot_positions_base[N,12] f32   Robot.GetFootPositionsInBaseFrame (robot.py:389-397); 16-byte aligned
 *   command            [N,3]  f32   desired (vx, vy, wz) incl. per-robot offsets
 *   com_height         [N]    f32   or NULL -> EstimateCoMHeightSimple from the stance feet
 *   contact_forces     [N,12] f32   OUT  -(first-step QP solution): force applied ON the ground
 *   horizon_forces     [N,h,12] f32 OUT or NULL: -(full QP solution)
 *   solve_info         [N,4]  i32   OUT or NULL: see RG_INFO_*
 */
int rg_mpc_build_solve(const void* workspace, int n_env,
                       const float* com_velocity_body, const float* base_rpy,
                       const float* base_rpy_rate, const uint8_t* foot_contact_state,
                       const float* foot_positions_base, const float* command,
                       const float* com_height,
                       float* contact_forces, float* horizon_forces, int32_t* solve_info,
                       void* stream);

/* Same solve, warm-started: `active_set_io` [N, 4*horizon] u16 holds, per (step, leg) block, the bit mask of
 * the rows the previous solve of the same env verified active (bits 0-4: upper bounds of the five pyramid
 * rows, bits 5-9: lower bounds) or RG_ACTIVE_SET_UNKNOWN.  It seeds the active-set iteration and is
 * overwritten with this solve's verified set (UNKNOWN for swing blocks and unverified solves).  Consecutive
 * control steps of one env see almost the same QP, so the seed usually verifies in a single round.  The
 * result is the same unique optimum whatever the seed; initialise the buffer to 0xFF bytes.
 * (No counterpart in the reference: OSQP is re-created cold on every compute_contact_forces call.) */
#define RG_ACTIVE_SET_UNKNOWN 0xFFFFu
int rg_mpc_build_solve_warm(const void* workspace, int n_env, const float* com_velocity_body,
                            const float* base_rpy, const float* base_rpy_rate,
                            const uint8_t* foot_contact_state, const float* foot_positions_base,
                            const float* command, const float* com_height, float* contact_forces,
                            float* horizon_forces, int32_t* solve_info, uint16_t* active_set_io, void* stream);

/* The same solve with every argument in one struct (the two entry points above forward to it), plus two things
 * they do not expose:
 *   zero_yaw            != 0: the solve uses yaw = 0 whatever base_rpy[:,2] holds -- what TorqueStanceLegController
 *                       does before it calls compute_contact_forces ("yaw aligned world frame")
 *   horizon_forces_f64  [N,h,12] f64 OUT or NULL: the full solution in the precision it was computed in (the
 *                       reference's solver returns doubles; the f32 outputs round it to ~1e-7 relative). */
typedef struct rg_mpc_io {
  const float* com_velocity_body;      /* [N,3]  */
  const float* base_rpy;               /* [N,3]  */
  const float* base_rpy_rate;          /* [N,3]  */
  const uint8_t* foot_contact_state;   /* [N,4]  4-byte aligned */
  const float* foot_positions_base;    /* [N,12] */
  const float* command;                /* [N,3]  */
  const float* com_height;             /* [N] or NULL */
  float* contact_forces;               /* [N,12] OUT */
  float* horizon_forces;               /* [N,h,12] OUT or NULL */
  int32_t* solve_info;                 /* [N,4] OUT or NULL */
  uint16_t* active_set_io;             /* [N,4h] in/out or NULL */
  double* horizon_forces_f64;          /* [N,h,12] OUT or NULL */
  int32_t zero_yaw;
  int32_t reserved_;
} rg_mpc_io;
int rg_mpc_build_solve_io(const void* workspace, int n_env, const rg_mpc_io* io_host, void* stream);

/* Per-env body and ground: the values each reference process passes to its own ConvexMpc(mass, inertia, ...)
 * (mpc_controller.py:47-56) and as the `friction` argument of every compute_contact_forces call.  Float64 DEVICE
 * arrays, env-major, 8-byte aligned; each may be NULL (= the workspace's value for every env).  They are parameters,
 * not sensor inputs: float64 so that a model filled with the workspace's own values solves what the workspace does.
 *   mass             [N]    kg.  The force bounds follow it with the workspace's ratios:
 *                           fz_max_e = fz_max * (mass_e / mass), fz_min_e = fz_min * (mass_e / mass)
 *                           (mpc_osqp's kMaxScale m g / kMinScale m g)
 *   inertia          [N,9]  body-frame inertia, row major; inverted on the device per solve
 *   friction_coeffs  [N,4]  one per pyramid ROW, as rg_mpc_params.friction_coeffs
 * Weights, alpha, dt, horizon, gravity and the desired body height stay per workspace.  The kernels read the arrays
 * on every launch (a captured control-step graph included), so new values written in place take effect at the next
 * solve.  A row that fails the checks rg_mpc_setup makes gets RG_STATUS_BAD_MODEL; the other envs are unaffected. */
typedef struct rg_mpc_env_model {
  const double* mass;             /* [N]    or NULL */
  const double* inertia;          /* [N,9]  or NULL */
  const double* friction_coeffs;  /* [N,4]  or NULL */
} rg_mpc_env_model;

/* rg_mpc_build_solve_io with a per-env model.  model == NULL, or all three pointers NULL, is exactly
 * rg_mpc_build_solve_io (which forwards here with NULL). */
int rg_mpc_build_solve_model(const void* workspace, int n_env, const rg_mpc_io* io_host,
                             const rg_mpc_env_model* model_host, void* stream);

/* Contact schedule: the planned stance of every leg at every step of the MPC horizon (Di Carlo et al. 2018), instead of
 * one contact row held over the whole horizon.  A [N,h,4] uint8 DEVICE array, env-major, 4-byte aligned; row k is the
 * 4-byte planned-stance word of horizon step k in the format of foot_contact_state (nonzero = stance).
 *  - Block (k, leg) of the QP is a stance block iff its byte is nonzero; otherwise its forces are pinned to zero, as a
 *    swing leg's are without a schedule.
 *  - io->foot_contact_state is not read and may be NULL.
 *  - The com height (only when io->com_height is NULL) is the mean z of the stance feet of row 0, or of the first row
 *    that has a stance foot when row 0 has none.  The lever arms are the feet's current positions at every step (see
 *    rg_mpc_build_solve_footholds for per-step footholds).
 *  - An all-zero schedule gives zero forces and RG_STATUS_NO_STANCE | RG_STATUS_POLISHED, and resets the warm start.
 *  - A schedule whose rows all equal one contact row gives bit-identical forces, solve_info and warm-start words to the
 *    call without a schedule.
 * rg_mpc_build_solve_schedule with contact_schedule == NULL is exactly rg_mpc_build_solve_model; model may be NULL
 * (the workspace's body and ground).  A misaligned schedule returns RG_ERR_BAD_ARG before anything is launched. */
int rg_mpc_build_solve_schedule(const void* workspace, int n_env, const rg_mpc_io* io_host,
                                const rg_mpc_env_model* model_host, const uint8_t* contact_schedule, void* stream);

/* Foothold plan: the position of every foot at every step of the MPC horizon, so that the QP's lever arms follow the
 * feet through the plan (Di Carlo et al. 2018: one B per step from the predicted footholds) instead of holding the
 * current feet.  A [N,h,12] float32 DEVICE array, env-major, 16-byte aligned; row k holds the four feet (FR, FL, RR, RL;
 * x, y, z) at horizon step k, in the frame and convention of foot_positions_base (the base frame of the current step,
 * rotated by the solve's Rx Ry Rz of the yaw-zeroed attitude, as the current feet are).
 *  - Block (k, leg) takes row k's foot `leg` as its lever arm.  Entries of swing blocks (schedule byte 0) are not read:
 *    any value there, NaN included, changes nothing.
 *  - io->foot_positions_base is not read and may be NULL.  The com height (only when io->com_height is NULL) is the mean
 *    z of the stance feet of row r* of the plan, r* being the schedule row rg_mpc_build_solve_schedule takes it from
 *    (row 0, or the first row with a stance foot).
 *  - A plan whose rows all equal foot_positions_base gives bit-identical forces, solve_info and warm-start words to
 *    rg_mpc_build_solve_schedule.
 * A plan requires a contact schedule.  rg_mpc_build_solve_footholds with foothold_plan == NULL is exactly
 * rg_mpc_build_solve_schedule; a non-NULL plan with a NULL schedule, or a misaligned plan, returns RG_ERR_BAD_ARG before
 * anything is launched. */
int rg_mpc_build_solve_footholds(const void* workspace, int n_env, const rg_mpc_io* io_host,
                                 const rg_mpc_env_model* model_host, const uint8_t* contact_schedule,
                                 const float* foothold_plan, void* stream);

/* ---- robot model: leg chains + gait + gains ------------------------------------------------
 * Replaces the per-robot python constants the third-party stack reads through the robot
 * callbacks (robot.py:88-92,169-170; ghost/ctrl_constants.py:13,28-41;
 * ghost/motor_constants.py:9-15) and the URDF leg geometry PyBullet uses implicitly. */
typedef struct rg_leg_chain {
  /* foot = T0 * Rot(axis0,q0) * T1 * Rot(axis1,q1) * T2 * Rot(axis2,q2) * toe,  Ti = (Ri, pi) */
  double p[3][3];              /* joint origin translations (parent frame) */
  double r[3][9];              /* joint origin rotations, row major */
  double axis[3][3];           /* joint axes (joint frame) */
  double toe[3];               /* fixed toe offset in the lower-link frame */
  double ik_sign_hip;          /* +-1: branch of the abduction solution */
  double ik_sign_knee;         /* +-1: branch of the knee solution */
} rg_leg_chain;

typedef struct rg_robot_params {
  rg_leg_chain legs[RG_NUM_LEGS];          /* FR, FL, RR, RL */
  double hip_positions[RG_NUM_LEGS][3];    /* DEFAULT_HIP_POSITIONS (ghost/constants.py:31-36) */
  double motor_offset[RG_NUM_MOTORS];      /* MOTOR_OFFSET   (ghost/motor_constants.py:9) */
  double motor_direction[RG_NUM_MOTORS];   /* MOTOR_DIRECTION (ghost/motor_constants.py:11) */
  double motor_kp[RG_NUM_MOTORS];          /* MOTOR_POSITION_GAINS (:13) */
  double motor_kd[RG_NUM_MOTORS];          /* MOTOR_VELOCITY_GAINS (:15) */
  /* OpenloopGaitGenerator ctor args (mpc_controller.py:30-35) */
  double stance_duration[RG_NUM_LEGS];
  double duty_factor[RG_NUM_LEGS];
  double initial_leg_phase[RG_NUM_LEGS];
  int32_t initial_leg_state[RG_NUM_LEGS];
  double contact_detection_phase_threshold;   /* 0.1 */
  /* RaibertSwingLegController ctor args (mpc_controller.py:38-45) + module constants */
  double desired_height;                      /* MPC_BODY_HEIGHT */
  double foot_clearance;                      /* 0.01 */
  double swing_kp[3];                         /* _KP = (0.03, 0.03, 0.03) */
  double swing_max_clearance;                 /* 0.1 */
  int32_t velocity_window;                    /* COMVelocityEstimator window_size = 20 */
} rg_robot_params;

/* Host-only helper: picks ik_sign_hip / ik_sign_knee of every leg so that IK(FK(q)) == q at the
 * given reference pose (12 motor angles, e.g. INIT_MOTOR_ANGLES, ghost/constants.py:12-17). */
int rg_robot_calibrate_ik(rg_robot_params* p_host, const double* reference_motor_angles12_host);

int rg_robot_workspace_bytes(size_t* bytes_host);
int rg_robot_setup(const rg_robot_params* p_host, void* robot_workspace, size_t bytes, void* stream);

/* Replaces: OpenloopGaitGenerator.update(t) (+ .reset) -- call site mpc_controller.py:30-35,104.
 *   time_since_reset [N] f64; foot_contacts [N,4] u8 (Robot.GetFootContacts, robot.py:215-229)
 *   OUT desired_leg_state, leg_state [N,4] i32; normalized_phase [N,4] f64 (bit-exact vs CPython). */
int rg_gait_step(const void* robot_workspace, int n_env, const double* time_since_reset,
                 const uint8_t* foot_contacts, int32_t* desired_leg_state, int32_t* leg_state,
                 double* normalized_phase, void* stream);

/* Replaces: COMVelocityEstimator.update (window filter with Neumaier sums + rotation into the
 * body frame) -- call site mpc_controller.py:36,104.  State arrays are caller-owned:
 *   window [N,3,W] f64, window_sum/window_corr [N,3] f64, window_count/window_head [N] i32. */
int rg_com_velocity_update(const void* robot_workspace, int n_env, const float* base_velocity_world,
                           const float* base_orientation_xyzw, double* window, double* window_sum,
                           double* window_corr, int32_t* window_count, int32_t* window_head,
                           float* com_velocity_body, float* com_velocity_world, void* stream);

/* Replaces: RaibertSwingLegController.update/get_action up to (not including) IK --
 * call site mpc_controller.py:38-45,104-105.  Latches lift-off positions, computes the
 * Raibert foothold and the swing-trajectory point for every non-stance leg.
 *   last_leg_state [N,4] i32 in/out (-1 = "aliased after reset": first update never latches)
 *   phase_switch_foot_local_position [N,12] f32 in/out
 *   OUT swing_foot_target [N,12] f32 (base frame; untouched for stance legs) */
int rg_swing_targets(const void* robot_workspace, int n_env, const int32_t* desired_leg_state,
                     const int32_t* leg_state, const double* normalized_phase,
                     const float* foot_positions_base, const float* com_velocity_body,
                     const float* base_rpy_rate, const float* command,
                     int32_t* last_leg_state, float* phase_switch_foot_local_position,
                     float* swing_foot_target, void* stream);

/* Replaces: Kinematics.ComputeMotorAnglesFromFootLocalPosition -> pybullet.calculateInverseKinematics
 * (robot_gym/controllers/mpc/kinematics.py:98-133,90-92).  Closed-form 3-DoF leg IK per (env, leg):
 *   foot_local_position [N,12] f32 -> motor_angles [N,12] f32 ((joint - MOTOR_OFFSET)*MOTOR_DIRECTION);
 *   leg_mask [N,4] u8 or NULL (1 = compute this leg; others left untouched). */
int rg_leg_ik(const void* robot_workspace, int n_env, const float* foot_local_position,
              const uint8_t* leg_mask, float* motor_angles, void* stream);

/* State provider ("next" row f2 of SURVEY.md 8): the robot getters the controller stack pulls its inputs
 * from, for a simulator that exposes raw rigid-body state instead of PyBullet queries.  Replaces
 *   Robot.GetBaseRollPitchYaw          robot.py:79-86   (getEulerFromQuaternion of the base orientation)
 *   Robot.GetBaseRollPitchYawRate      robot.py:205-213 -> TransformAngularVelocityToLocalFrame :185-203
 *                                      (world angular velocity rotated by the inverse base orientation)
 *   Robot.GetMotorAngles               robot.py:231-236 ((joint - MOTOR_OFFSET) * MOTOR_DIRECTION)
 *   Robot.GetFootPositionsInBaseFrame  robot.py:389-397,367-383 (forward kinematics of the URDF chains
 *                                      instead of four getLinkState round trips)
 *   base_quat_xyzw [N,4] f32, base_ang_vel_world [N,3] f32 (may be NULL when base_rpy_rate is NULL),
 *   joint_angles [N,12] f32 (raw URDF joint angles)  ->  base_rpy [N,3], base_rpy_rate [N,3],
 *   motor_angles [N,12], foot_positions_base [N,4,3], all f32; any output may be NULL (skipped). */
int rg_state_from_sim(const void* robot_workspace, int n_env, const float* base_quat_xyzw,
                      const float* base_ang_vel_world, const float* joint_angles, float* base_rpy,
                      float* base_rpy_rate, float* motor_angles, float* foot_positions_base, void* stream);

/* Forward kinematics of the same chains (replaces Robot.GetFootPositionsInBaseFrame's
 * getLinkState round trips, robot.py:367-397, for a state provider without PyBullet). */
int rg_leg_fk(const void* robot_workspace, int n_env, const float* motor_angles,
              float* foot_positions_base, void* stream);

/* Replaces: Kinematics.MapContactForceToJointTorques -> pybullet.calculateJacobian
 * (robot_gym/controllers/mpc/kinematics.py:13-53): tau_j = (f . J[:,6+j]) * MOTOR_DIRECTION[j]
 * with J the base-frame translational foot Jacobian.  contact_forces [N,12], motor_angles [N,12]
 * -> motor_torques [N,12], all f32. */
int rg_force_to_torque(const void* robot_workspace, int n_env, const float* contact_forces,
                       const float* motor_angles, float* motor_torques, void* stream);

/* Replaces: LocomotionController.get_action's merge of swing and stance 5-tuples into the flat
 * 60-float hybrid command (consumer: simple_motor.py:128-137).  swing_joint_angles [N,12] holds
 * the persistent `_joint_angles` store; swing_joint_valid [N,4] u8 says whether a leg has one. */
int rg_pack_hybrid_action(const void* robot_workspace, int n_env, const int32_t* desired_leg_state,
                          const float* swing_joint_angles, const uint8_t* swing_joint_valid,
                          const float* motor_torques, float* action, void* stream);

/* One call = MPCController.get_action() (mpc_controller.py:102-106): gait update, velocity estimator, swing
 * latch/target/IK (prologue kernel), MPC stance solve (one kernel when the batch fits a wave, else the lean kernel plus
 * the fallback kernel on its queue), force->torque + action pack (+ optional motor model; epilogue kernel): three or
 * four launches, or ONE graph launch through rg_control_step_graph_* below.
 * All state in/out arrays as in the individual calls.  `controller_state` groups them. */
typedef struct rg_controller_state {
  /* inputs (robot callbacks) */
  const double* time_since_reset;        /* [N]    */
  const uint8_t* foot_contacts;          /* [N,4]  */
  const float* base_velocity_world;      /* [N,3]  */
  const float* base_orientation_xyzw;    /* [N,4]  */
  const float* base_rpy;                 /* [N,3]  */
  const float* base_rpy_rate;            /* [N,3]  */
  const float* foot_positions_base;      /* [N,12] */
  const float* motor_angles;             /* [N,12] (GetMotorAngles convention) */
  const float* command;                  /* [N,3]  */
  /* persistent controller state */
  double* vel_window; double* vel_window_sum; double* vel_window_corr;
  int32_t* vel_window_count; int32_t* vel_window_head;
  int32_t* last_leg_state;               /* [N,4]  */
  float* phase_switch_foot_local_position; /* [N,12] */
  float* swing_joint_angles;             /* [N,12] */
  uint8_t* swing_joint_valid;            /* [N,4]  */
  uint16_t* mpc_active_set;              /* [N,4*horizon] warm start of the stance QP (rg_mpc_build_solve_warm) or NULL */
  /* outputs */
  int32_t* desired_leg_state; int32_t* leg_state; double* normalized_phase;   /* [N,4] each */
  uint8_t* mpc_contact_state;            /* [N,4]  planned-stance flags handed to the MPC */
  float* swing_foot_target;              /* [N,12] */
  float* com_velocity_body;              /* [N,3]  */
  float* contact_forces;                 /* [N,12] */
  float* motor_torques;                  /* [N,12] */
  int32_t* solve_info;                   /* [N,4] or NULL */
  float* action;                         /* [N,60] */
  /* optional torque consumer (all three NULL = not attached): when applied_motor_torques is given, the epilogue
   * also evaluates the HYBRID motor model on the fresh command -- Robot.ApplyAction of the first of the
   * ACTION_REPEAT physics ticks (robot.py:276-307, simple_motor.py:128-140) -- so a GPU physics step can consume
   * torques without reading the [N,60] command back */
  const float* motor_velocities;         /* [N,12] GetMotorVelocities convention, required with the consumer */
  const float* motor_strength_ratios;    /* [N,12] RobotMotorModel._strength_ratios (simple_motor.py:52-60) or NULL = 1 */
  float* applied_motor_torques;          /* [N,12] OUT: strength * PD-plus-feed-forward torque * MOTOR_DIRECTION */
} rg_controller_state;

int rg_control_step(const void* mpc_workspace, const void* robot_workspace, int n_env,
                    const rg_controller_state* s_host, void* stream);

/* The same control step as ONE CUDA-graph launch (small batches are launch-bound: prologue + solve + epilogue are three
 * dependent kernels of a few microseconds each).  rg_control_step_graph_create captures rg_control_step with the pointers
 * of `s` baked in and -- to configure kernels and surface argument errors outside the capture -- EXECUTES ONE STEP while
 * doing so (on `stream`): call it in place of a control step, not before one; it synchronises `stream`.  rg_control_step_graph_launch replays the
 * step on `stream` without synchronising.  Re-create the graph when any buffer of `s` moves or n_env changes. */
int rg_control_step_graph_create(const void* mpc_workspace, const void* robot_workspace, int n_env,
                                 const rg_controller_state* s_host, void* stream, void** graph_out);
int rg_control_step_graph_launch(void* graph, void* stream);
int rg_control_step_graph_destroy(void* graph);

/* The control step and its graph with a per-env model in the stance solve (rg_mpc_env_model above; NULL = the two
 * calls before it, which forward here).  The graph bakes in the model POINTERS, not the values: writing new masses,
 * inertias or friction coefficients into the same arrays between replays needs no re-capture. */
int rg_control_step_model(const void* mpc_workspace, const void* robot_workspace, int n_env,
                          const rg_controller_state* s_host, const rg_mpc_env_model* model_host, void* stream);
int rg_control_step_graph_create_model(const void* mpc_workspace, const void* robot_workspace, int n_env,
                                       const rg_controller_state* s_host, const rg_mpc_env_model* model_host,
                                       void* stream, void** graph_out);

/* Per-env OpenloopGaitGenerator arguments (mpc_controller.py:30-35): what each reference process passes to its own
 * OpenloopGaitGenerator(stance_duration, duty_factor, initial_leg_phase, initial_leg_state).  DEVICE arrays, env-major,
 * each [N,4] (leg order FR, FL, RR, RL) and each may be NULL (= the robot workspace's value for every env).  Read on
 * every launch (a captured graph included), so values written in place between replays take effect at the next step,
 * at the env's current clock.  A row is valid when, for every leg, stance_duration > 0 and finite,
 * 0 < duty_factor <= 1, 0 <= initial_leg_phase < 1 and initial_leg_state is RG_LEG_SWING or RG_LEG_STANCE (the
 * workspace's value standing in for a NULL array).  The kernel decides validity from the values it loads (no host check); an invalid
 * row holds its env in stance (see the note after the status bits).  The stance duration also sets the Raibert
 * foothold of the swing legs (hv * stance_duration / 2). */
typedef struct rg_gait_env_params {
  const double*  stance_duration;    /* [N,4] f64, 8-byte aligned */
  const double*  duty_factor;        /* [N,4] f64, 8-byte aligned */
  const double*  initial_leg_phase;  /* [N,4] f64, 8-byte aligned */
  const int32_t* initial_leg_state;  /* [N,4] i32, 4-byte aligned */
} rg_gait_env_params;

/* The control step and its graph with a per-env model and a per-env gait (either may be NULL, or have all pointers
 * NULL: the _model calls above forward here with gait = NULL and launch exactly the gait-free kernels).  A misaligned
 * array returns RG_ERR_BAD_ARG before anything is launched.  As with the model, the graph bakes in the gait POINTERS. */
int rg_control_step_env(const void* mpc_workspace, const void* robot_workspace, int n_env,
                        const rg_controller_state* s_host, const rg_mpc_env_model* model_host,
                        const rg_gait_env_params* gait_host, void* stream);
int rg_control_step_graph_create_env(const void* mpc_workspace, const void* robot_workspace, int n_env,
                                     const rg_controller_state* s_host, const rg_mpc_env_model* model_host,
                                     const rg_gait_env_params* gait_host, void* stream, void** graph_out);

/* The control step with the stance solve planned over the gait's contact schedule (rg_mpc_build_solve_schedule).  The
 * prologue writes contact_schedule_out ([N,h,4] uint8 DEVICE array, 4-byte aligned, h = the MPC workspace's horizon)
 * and the solve reads it.  Row k is desired_leg_state == RG_LEG_STANCE of the env's OpenloopGaitGenerator (the
 * workspace's, or the env's row of `gait`) evaluated at t_k = t + k * dt, dt the MPC workspace's planning step, with
 * the separately rounded arithmetic of the gait update and no contact detection; row 0 therefore equals
 * mpc_contact_state.  An env whose gait row is not valid gets all-stance rows.  contact_schedule_out == NULL is exactly
 * rg_control_step_env / rg_control_step_graph_create_env.  A misaligned schedule returns RG_ERR_BAD_ARG before anything
 * is launched; the graph bakes in its pointer. */
int rg_control_step_plan(const void* mpc_workspace, const void* robot_workspace, int n_env,
                         const rg_controller_state* s_host, const rg_mpc_env_model* model_host,
                         const rg_gait_env_params* gait_host, uint8_t* contact_schedule_out, void* stream);
int rg_control_step_graph_create_plan(const void* mpc_workspace, const void* robot_workspace, int n_env,
                                      const rg_controller_state* s_host, const rg_mpc_env_model* model_host,
                                      const rg_gait_env_params* gait_host, uint8_t* contact_schedule_out, void* stream,
                                      void** graph_out);

/* The planned control step with predicted footholds (rg_mpc_build_solve_footholds).  The prologue writes
 * foothold_plan_out ([N,h,12] float32 DEVICE array, 16-byte aligned) next to contact_schedule_out, and the solve reads
 * both.  Per leg, with p its current foot (foot_positions_base) and v = (command[0], command[1], 0), in double and
 * stored as float32:
 *     anchor = p, k_a = 0
 *     for k in 0 .. h-1:
 *         if k >= 1 and schedule[k] is stance and schedule[k-1] is swing:   touchdown inside the horizon
 *             anchor = the Raibert foothold of the swing controller, k_a = k
 *         foothold[k] = anchor - (k - k_a) * dt * v                          the body walks over a planted foot
 * The Raibert foothold is exactly the end point of the leg's swing trajectory (the float32-rounded velocity estimate, yaw
 * rate, command, the env's stance duration, the hip offset and desired_height - foot_clearance).  The yaw rate is not
 * integrated into the footholds, as the QP's model holds the yaw in B.  An env whose gait row is not valid gets held
 * rows (foothold[k] = p).  foothold_plan_out == NULL is exactly rg_control_step_plan /
 * rg_control_step_graph_create_plan; a non-NULL plan with a NULL contact_schedule_out, or a misaligned plan, returns
 * RG_ERR_BAD_ARG before anything is launched; the graph bakes in its pointer. */
int rg_control_step_footholds(const void* mpc_workspace, const void* robot_workspace, int n_env,
                              const rg_controller_state* s_host, const rg_mpc_env_model* model_host,
                              const rg_gait_env_params* gait_host, uint8_t* contact_schedule_out,
                              float* foothold_plan_out, void* stream);
int rg_control_step_graph_create_footholds(const void* mpc_workspace, const void* robot_workspace, int n_env,
                                           const rg_controller_state* s_host, const rg_mpc_env_model* model_host,
                                           const rg_gait_env_params* gait_host, uint8_t* contact_schedule_out,
                                           float* foothold_plan_out, void* stream, void** graph_out);

/* ---- "next" row (SURVEY.md 8f rank 1): batched HYBRID motor model ----------------------------
 * Replaces RobotMotorModel.convert_to_torque HYBRID branch (simple_motor.py:128-139):
 * tau = -kp (q - q_des) - kd (qd - qd_des) + tau_ff ; no clipping (robot.py:40-45). */
int rg_hybrid_motor_torque(int n_env, const float* action, const float* motor_angles,
                           const float* motor_velocities, float* motor_torques, void* stream);
/* The same with the two factors Robot.ApplyAction applies around it (robot.py:276-307):
 *   observed = strength_ratios * tau      (simple_motor.py:140; strength_ratios [N,12] or NULL = 1)
 *   applied  = observed * MOTOR_DIRECTION (robot.py:291-292; from the robot workspace)
 * Either output may be NULL.  One call per physics tick of Simulation.ApplyStepAction (core/simulation.py:175-179). */
int rg_hybrid_motor_torque_ex(const void* robot_workspace, int n_env, const float* action, const float* motor_angles,
                              const float* motor_velocities, const float* strength_ratios,
                              float* observed_torques, float* applied_torques, void* stream);

/* Diagnostic (synchronises the device): best-of-4 CUDA-core FMA throughput in TFLOP/s, fp32 or fp64,
 * the roofline denominator for the solve kernel (MEASURED_PEAKS.json has no CUDA-core peak). */
int rg_measure_fma_peak(int use_fp64, int iters, double* tflops_host);

/* Counters for bench.py's gpu_launches claim: number of kernels this library launched since load. */
uint64_t rg_launch_count(void);
const char* rg_last_error(void);
const char* rg_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RG_CUDA_H_ */
