// Shared device/host definitions for the batched locomotion-controller kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "rg_cuda.h"

#define RG_WS_MAGIC_MPC 0x52474d50u   // "RGMP"
#define RG_WS_MAGIC_ROBOT 0x5247524fu // "RGRO"

// Device image of rg_mpc_params + the horizon tables, as laid out in the MPC workspace.
struct RgMpcDev {
  uint32_t magic;
  int32_t horizon;
  int32_t max_ipm_iters;
  int32_t max_polish_rounds;
  int32_t cold_start_rounds;
  int32_t cold_start_max_violations;
  double inv_mass;
  double inv_inertia[9];   // body frame
  double dt;
  double w_rho[6];         // weights of (roll,pitch,yaw,x,y,z)
  double w_nu[6];          // weights of (wx,wy,wz,vx,vy,vz)
  double alpha;
  double mu[4];
  double gravity;
  double fz_max, fz_min;
  double height;
  double ipm_tol;
  // Generalised eigen-decomposition of the horizon coupling tables (see DESIGN.md 3.2):
  //   c1(j,k) = h - max(j,k), c2(j,k) = sum_{i>max(j,k)}^{h} (i-j-1/2)(i-k-1/2)
  //   U^T c1 U = I,  U^T c2 U = diag(gamma);  eig_u is row-major [j][t].
  double eig_u[RG_MAX_HORIZON * RG_MAX_HORIZON];
  double eig_gamma[RG_MAX_HORIZON];
  // eig_uu[(j(j+1)/2 + k) * h + t] = U[j][t] U[k][t], k <= j: the rank-h weights of K^-1's (j,k) time block
  double eig_uu[RG_MAX_HORIZON * (RG_MAX_HORIZON + 1) / 2 * RG_MAX_HORIZON];
  // env-independent tables (host-computed, read through the L1/L2-cached uniform path):
  double c2tab[RG_MAX_HORIZON * RG_MAX_HORIZON];                        // c2(j,k), row-major h x h
  double kinv_lin[3][RG_MAX_HORIZON * (RG_MAX_HORIZON + 1) / 2];        // K^-1 of the x/y/z channels, packed
  // mass of the parameter set: a per-env model (rg_mpc_env_model) scales fz_max / fz_min by mass_e / mass.  Last, so
  // that the offsets the model-free kernels read are the ones they were tuned with.
  double mass;
};

// Per-workspace scratch behind the parameter block (rg_workspace_bytes(n_env, ...) sizes it for n_env envs):
// the fallback queue of the two-kernel solve.  The lean kernel appends the envs its active-set rounds could
// not verify; the full kernel then runs on that list and its last CTA re-arms the counters, so no memset
// sits between launches.  One solve at a time per workspace (concurrent streams need their own workspace).
struct RgMpcScratch {
  int32_t queue_tail;      // number of queued envs (atomicAdd by the lean kernel)
  int32_t done_ctas;       // ticket counter of the fallback kernel's CTAs
  int32_t capacity;        // entries of queue[] (written by rg_mpc_setup, read-only afterwards)
  int32_t reserved[61];
  int32_t queue[1];        // [capacity]
};
#define RG_MPC_SCRATCH_OFFSET ((sizeof(RgMpcDev) + 255) & ~size_t(255))

// Device image of rg_robot_params with the IK constants derived on the host.
struct RgLegDev {
  double p[3][3];
  double r[3][9];
  double axis[3][3];
  double toe[3];
  // closed-form IK constants (hip-joint frame), see rg_kinematics.cuh
  double e0[3], e1[3], e2[3];   // orthonormal basis in the hip-link frame: e0 = hip axis, e1 = upper axis
  double t1e0, t1e2, dconst;    // upper-joint offset along e0/e2 and the constant lateral offset D along e1
  double l1, l2, phi2, psi;     // planar two-link lengths, phase of link 2, phase of the plane basis
  double s2;                    // +1/-1: lower axis parallel/antiparallel to the upper axis
  double sign_hip, sign_knee;
};

struct RgRobotDev {
  uint32_t magic;
  int32_t velocity_window;
  RgLegDev legs[RG_NUM_LEGS];
  double hip_positions[RG_NUM_LEGS][3];
  double motor_offset[RG_NUM_MOTORS];
  double motor_direction[RG_NUM_MOTORS];
  double motor_kp[RG_NUM_MOTORS];
  double motor_kd[RG_NUM_MOTORS];
  double stance_duration[RG_NUM_LEGS];
  double duty_factor[RG_NUM_LEGS];
  double initial_leg_phase[RG_NUM_LEGS];
  int32_t initial_leg_state[RG_NUM_LEGS];
  int32_t next_leg_state[RG_NUM_LEGS];
  double initial_state_ratio[RG_NUM_LEGS];
  double contact_detection_phase_threshold;
  double desired_height;
  double foot_clearance;
  double swing_kp[3];
  double swing_max_clearance;
};

// host-side error plumbing (rg_api.cu)
void rg_set_error(const char* fmt, ...);
int rg_check_cuda(cudaError_t e, const char* what);
void rg_count_launch();
extern "C" uint64_t rg_launch_count(void);

// launchers implemented in the .cu files
struct rg_controller_state;
// chained = 1: the caller launched a kernel that signals griddepcontrol.launch_dependents right before (the step
// prologue) and launches one with the programmatic attribute right after (the epilogue): the first MPC kernel is then
// launched programmatically too.  Every MPC kernel starts with griddepcontrol.wait (a no-op after a plain launch).
// model: a per-env model with at least one non-NULL array, or NULL (the model-free kernels).
// plan: a [N,h,4] contact schedule (rg_mpc_build_solve_schedule) or NULL; non-NULL launches the schedule kernels, with
// `model` or, when it is NULL, the workspace's body and ground.
// feet: a [N,h,12] foothold plan (rg_mpc_build_solve_footholds) or NULL; non-NULL (with a plan) launches the foothold
// kernels.
int rg_launch_mpc(const RgMpcDev* ws, int horizon, int n_env, const rg_mpc_io& io, int two_kernel, cudaStream_t stream, int chained = 0,
                  const rg_mpc_env_model* model = nullptr, const uint8_t* plan = nullptr, const float* feet = nullptr);
// NULL, or a model whose three pointers are all NULL -> NULL; RG_ERR_BAD_ARG for an array that is not 8-byte aligned
int rg_check_env_model(const rg_mpc_env_model* model, const char* what, const rg_mpc_env_model** out);

// Kernel launch with or without the programmatic-stream-serialization attribute (programmatic dependent launch: the
// grid may become resident while its predecessor drains; it must execute griddepcontrol.wait before touching the
// predecessor's results, and the predecessor signals with griddepcontrol.launch_dependents).
template <class... KArgs, class... Args>
inline cudaError_t rg_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool programmatic, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = programmatic ? 1 : 0;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
  return e != cudaSuccess ? e : cudaGetLastError();
}
#define RG_GRID_WAIT() asm volatile("griddepcontrol.wait;" ::: "memory")
#define RG_GRID_LAUNCH_DEPENDENTS() asm volatile("griddepcontrol.launch_dependents;")
// host-side record of a workspace prepared by rg_mpc_setup (no device access on the launch path)
// dt: the planning step, which the control step's prologue needs to evaluate the gait across the horizon
struct RgMpcHostInfo { int horizon; int queue_capacity; int two_kernel; double dt; };
int rg_mpc_workspace_info(const void* workspace, RgMpcHostInfo* info);
