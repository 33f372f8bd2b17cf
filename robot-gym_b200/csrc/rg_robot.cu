// Gait generator, COM velocity estimator, Raibert swing controller, leg kinematics (FK / closed
// form IK / foot Jacobian), hybrid-action packing and the fused control step (sm_100a).
//
// These are the light, HBM-bound parts of the control step (~550 B per env-step): one thread per
// env or per (env, leg), float64 arithmetic on float32 state, coalesced row-major loads.
// The third-party routines they replace are cited per kernel; see include/rg_cuda.h.
#include "rg_common.cuh"

#include <math.h>
#include <string.h>

namespace {

// ------------------------------------------------------------------------------------ small math
struct V3 { double x, y, z; };
__host__ __device__ inline V3 v3(double x, double y, double z) { return V3{x, y, z}; }
__host__ __device__ inline V3 add(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
__host__ __device__ inline V3 sub(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
__host__ __device__ inline V3 mul(double s, V3 a) { return v3(s * a.x, s * a.y, s * a.z); }
__host__ __device__ inline double dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__host__ __device__ inline V3 cross(V3 a, V3 b) { return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
__host__ __device__ inline V3 ld3(const double* p) { return v3(p[0], p[1], p[2]); }
__host__ __device__ inline V3 mat_mul(const double* m, V3 v) {   // row-major 3x3
  return v3(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[3] * v.x + m[4] * v.y + m[5] * v.z, m[6] * v.x + m[7] * v.y + m[8] * v.z);
}
__host__ __device__ inline V3 mat_tmul(const double* m, V3 v) {  // M^T v
  return v3(m[0] * v.x + m[3] * v.y + m[6] * v.z, m[1] * v.x + m[4] * v.y + m[7] * v.z, m[2] * v.x + m[5] * v.y + m[8] * v.z);
}
// Rodrigues rotation of v about the unit axis a by angle q
// Rodrigues rotation of v about the unit axis a by the angle whose sine / cosine are (s, c)
__host__ __device__ inline V3 rot_sc(V3 a, double s, double c, V3 v) {
  return add(add(mul(c, v), mul(s, cross(a, v))), mul((1.0 - c) * dot(a, v), a));
}
__host__ __device__ inline double wrap_pi(double a) {
  const double two_pi = 6.283185307179586476925286766559;
  a = fmod(a + 3.14159265358979323846, two_pi);
  if (a < 0) a += two_pi;
  return a - 3.14159265358979323846;
}

// ------------------------------------------------------------------------------------ kinematics
// foot = p0 + R0 Rot(a0,q0) ( p1 + R1 Rot(a1,q1) ( p2 + R2 Rot(a2,q2) toe ) ), base frame.
// Also returns the translational Jacobian columns (axis_world x (foot - origin_world)).
// FAST_TRIG: single-precision sincosf of the (float32) joint angles -- 1e-7 absolute on a 0.5 m chain, below
// the float32 output resolution; used by the state provider, whose cost is otherwise all FP64 trigonometry.
template <bool FAST_TRIG = false>
__host__ __device__ inline V3 leg_fk(const RgLegDev& L, const double* q, V3* jac /* 3 columns or nullptr */) {
  const V3 a0 = ld3(L.axis[0]), a1 = ld3(L.axis[1]), a2 = ld3(L.axis[2]);
  double sn[3], cs[3];   // one sine / cosine per joint, shared by every rotation below
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    if (FAST_TRIG) {
      float sf, cf;
      sincosf((float)q[j], &sf, &cf);
      sn[j] = sf; cs[j] = cf;
    } else {
      sincos(q[j], &sn[j], &cs[j]);
    }
  }
  // innermost first
  V3 v2 = rot_sc(a2, sn[2], cs[2], ld3(L.toe));             // in joint-2 frame
  V3 w2 = add(ld3(L.p[2]), mat_mul(L.r[2], v2));            // in link-1 frame (joint-1 frame after rotation)
  V3 v1 = rot_sc(a1, sn[1], cs[1], w2);
  V3 w1 = add(ld3(L.p[1]), mat_mul(L.r[1], v1));            // in link-0 frame
  V3 v0 = rot_sc(a0, sn[0], cs[0], w1);
  V3 foot = add(ld3(L.p[0]), mat_mul(L.r[0], v0));
  if (jac) {
    // world (base) frame axes and origins
    const V3 ax0 = mat_mul(L.r[0], a0);
    const V3 o0 = ld3(L.p[0]);
    // F0 x = R0 Rot0 x
    const V3 o1 = add(o0, mat_mul(L.r[0], rot_sc(a0, sn[0], cs[0], ld3(L.p[1]))));
    const V3 ax1 = mat_mul(L.r[0], rot_sc(a0, sn[0], cs[0], mat_mul(L.r[1], a1)));
    const V3 p2_l0 = mat_mul(L.r[1], rot_sc(a1, sn[1], cs[1], ld3(L.p[2])));           // in link-0 frame
    const V3 o2 = add(o1, mat_mul(L.r[0], rot_sc(a0, sn[0], cs[0], p2_l0)));
    const V3 ax2_l0 = mat_mul(L.r[1], rot_sc(a1, sn[1], cs[1], mat_mul(L.r[2], a2)));
    const V3 ax2 = mat_mul(L.r[0], rot_sc(a0, sn[0], cs[0], ax2_l0));
    jac[0] = cross(ax0, sub(foot, o0));
    jac[1] = cross(ax1, sub(foot, o1));
    jac[2] = cross(ax2, sub(foot, o2));
  }
  return foot;
}

// Damped least squares on the exact chain, min |foot - FK(q)|, from q: the fallback of leg_ik where the Newton clean-up
// cannot run (target out of reach or inside the abduction cylinder, or a singular straight-knee pose).  The clamped
// closed form is the nearest reachable point only for the idealised geometry: the upper joint sits off the hip axis, so
// turning the hip can bring a straight leg closer.  Steps (J^T J + 1e-6 I) d = J^T err, capped at 0.5 rad, as the
// damped IK of the reference's kinematics; a step is kept only while it reduces the distance.
__host__ __device__ __noinline__ void leg_ik_dls(const RgLegDev& L, V3 foot, double* q) {
  double best[3] = {q[0], q[1], q[2]};
  double best_e = 1e300;
  for (int it = 0; it < 32; ++it) {
    V3 jac[3];
    const V3 err = sub(foot, leg_fk(L, q, jac));
    const double e = dot(err, err);
    if (!(e < best_e)) break;                          // no progress (or not finite): the best iterate stands
    best[0] = q[0]; best[1] = q[1]; best[2] = q[2];
    best_e = e;
    const double lam = 1e-6;
    const double a00 = dot(jac[0], jac[0]) + lam, a01 = dot(jac[0], jac[1]), a02 = dot(jac[0], jac[2]);
    const double a11 = dot(jac[1], jac[1]) + lam, a12 = dot(jac[1], jac[2]), a22 = dot(jac[2], jac[2]) + lam;
    const double g0 = dot(jac[0], err), g1 = dot(jac[1], err), g2 = dot(jac[2], err);
    const double c00 = a11 * a22 - a12 * a12, c01 = a02 * a12 - a01 * a22, c02 = a01 * a12 - a02 * a11;
    const double c11 = a00 * a22 - a02 * a02, c12 = a01 * a02 - a00 * a12, c22 = a00 * a11 - a01 * a01;
    const double id = 1.0 / (a00 * c00 + a01 * c01 + a02 * c02);
    double d0 = (c00 * g0 + c01 * g1 + c02 * g2) * id;
    double d1 = (c01 * g0 + c11 * g1 + c12 * g2) * id;
    double d2 = (c02 * g0 + c12 * g1 + c22 * g2) * id;
    const double nrm = sqrt(d0 * d0 + d1 * d1 + d2 * d2);
    if (nrm < 1e-13) break;
    if (nrm > 0.5) { const double s = 0.5 / nrm; d0 *= s; d1 *= s; d2 *= s; }
    q[0] = wrap_pi(q[0] + d0); q[1] = wrap_pi(q[1] + d1); q[2] = wrap_pi(q[2] + d2);
  }
  q[0] = best[0]; q[1] = best[1]; q[2] = best[2];
}

// Closed-form IK (derivation in DESIGN.md 4.3): hip abduction from the projection onto the plane
// normal to the hip axis, then a planar two-link problem in the plane normal to the upper axis.
__host__ __device__ inline void leg_ik(const RgLegDev& L, V3 foot, double* q) {
  const V3 ph = mat_tmul(L.r[0], sub(foot, ld3(L.p[0])));   // hip-joint frame
  const double P0 = dot(ph, ld3(L.e0)), P1 = dot(ph, ld3(L.e1)), P2 = dot(ph, ld3(L.e2));
  const double D = L.dconst;
  double rad = P1 * P1 + P2 * P2 - D * D;
  if (rad < 0.0) rad = 0.0;
  const double w2 = L.sign_hip * sqrt(rad);
  q[0] = wrap_pi(atan2(P2, P1) - atan2(w2, D));
  const double alpha = P0 - L.t1e0, beta = w2 - L.t1e2;    // planar target: X = beta (e2), Y = alpha (e0)
  const double r2 = alpha * alpha + beta * beta;
  double ct = (r2 - L.l1 * L.l1 - L.l2 * L.l2) / (2.0 * L.l1 * L.l2);
  ct = ct > 1.0 ? 1.0 : (ct < -1.0 ? -1.0 : ct);
  const double theta = L.sign_knee * acos(ct);
  q[2] = wrap_pi(L.s2 * (theta - L.phi2));
  const double delta = atan2(L.l2 * sin(theta), L.l1 + L.l2 * cos(theta));
  q[1] = wrap_pi(atan2(alpha, beta) - L.psi - delta);
  // Newton clean-up on the exact chain: the URDFs give their right angles to five digits
  // (rpy = 1.57079), so the perpendicular/parallel-axis assumptions hold only to ~1e-5 rad.
  for (int it = 0; it < 2; ++it) {
    V3 jac[3];
    const V3 err = sub(foot, leg_fk(L, q, jac));
    const V3 c12 = cross(jac[1], jac[2]);
    const double det = dot(jac[0], c12);
    if (fabs(det) < 1e-12) { leg_ik_dls(L, foot, q); return; }                      // singular pose (straight leg)
    const double d0 = dot(err, c12) / det;
    const double d1 = dot(jac[0], cross(err, jac[2])) / det;
    const double d2 = dot(jac[0], cross(jac[1], err)) / det;
    if (fabs(d0) + fabs(d1) + fabs(d2) > 0.1) { leg_ik_dls(L, foot, q); return; }   // target out of reach
    q[0] = wrap_pi(q[0] + d0); q[1] = wrap_pi(q[1] + d1); q[2] = wrap_pi(q[2] + d2);
  }
}

// ------------------------------------------------------------------------------------ gait
// One leg's OpenloopGaitGenerator arguments and what its __init__ derives from them (ratio = the share of the cycle
// spent in the initial state, next = the state after it), from one of two sources with the same accessors:
//  * WorkspaceGait reads the robot workspace (ratio and next precomputed by rg_robot_setup) at the point of use, so the
//    gait-free kernels load exactly what and when they always have;
//  * EnvGait holds one leg of a per-env gait (rg_gait_env_params), loaded once, ratio and next derived on the device
//    as OpenloopGaitGenerator.__init__ / rg_robot_setup derive them (1 - duty is one IEEE subtraction in all three).
struct WorkspaceGait {
  static constexpr bool kPerEnv = false;
  const RgRobotDev& R;
  int leg;
  __device__ __forceinline__ static WorkspaceGait load(const RgRobotDev& R, const rg_gait_env_params&, size_t, int leg) {
    return WorkspaceGait{R, leg};
  }
  __device__ __forceinline__ bool valid() const { return true; }
  __device__ __forceinline__ double stance() const { return R.stance_duration[leg]; }
  __device__ __forceinline__ double duty() const { return R.duty_factor[leg]; }
  __device__ __forceinline__ double phase0() const { return R.initial_leg_phase[leg]; }
  __device__ __forceinline__ double ratio() const { return R.initial_state_ratio[leg]; }
  __device__ __forceinline__ int init() const { return R.initial_leg_state[leg]; }
  __device__ __forceinline__ int next() const { return R.next_leg_state[leg]; }
};

struct EnvGait {
  static constexpr bool kPerEnv = true;
  double st, du, ph, ra;
  int in, nx;
  // leg idx (= 4 env + leg) of a per-env gait; a NULL array stands for the workspace's value
  __device__ __forceinline__ static EnvGait load(const RgRobotDev& R, const rg_gait_env_params& g, size_t idx, int leg) {
    EnvGait o;
    o.st = g.stance_duration ? g.stance_duration[idx] : R.stance_duration[leg];
    o.du = g.duty_factor ? g.duty_factor[idx] : R.duty_factor[leg];
    o.ph = g.initial_leg_phase ? g.initial_leg_phase[idx] : R.initial_leg_phase[leg];
    o.in = g.initial_leg_state ? g.initial_leg_state[idx] : R.initial_leg_state[leg];
    const bool swing_first = o.in == RG_LEG_SWING;
    o.ra = swing_first ? __dsub_rn(1.0, o.du) : o.du;
    o.nx = swing_first ? RG_LEG_STANCE : RG_LEG_SWING;
    return o;
  }
  // the row rule of rg_gait_env_params (rg_cuda.h); NaN fails every comparison
  __device__ __forceinline__ bool valid() const {
    return st > 0.0 && st <= 1.7976931348623157e308 && du > 0.0 && du <= 1.0 && ph >= 0.0 && ph < 1.0 &&
           (in == RG_LEG_SWING || in == RG_LEG_STANCE);
  }
  __device__ __forceinline__ double stance() const { return st; }
  __device__ __forceinline__ double duty() const { return du; }
  __device__ __forceinline__ double phase0() const { return ph; }
  __device__ __forceinline__ double ratio() const { return ra; }
  __device__ __forceinline__ int init() const { return in; }
  __device__ __forceinline__ int next() const { return nx; }
};

// OpenloopGaitGenerator.update(t) for one leg; every operation is a separately rounded IEEE double
// operation in CPython's order, so phases and states are bit-identical to the reference's floats.
template <class Gait>
__device__ __forceinline__ void gait_leg(const RgRobotDev& R, const Gait& g, double t, bool contact,
                                         int& desired, int& state, double& nphase) {
  const double period = __ddiv_rn(g.stance(), g.duty());
  const double aug = __dadd_rn(t, __dmul_rn(g.phase0(), period));
  const double ph = __ddiv_rn(fmod(aug, period), period);
  const double ratio = g.ratio();
  if (ph < ratio) {
    desired = g.init();
    nphase = __ddiv_rn(ph, ratio);
  } else {
    desired = g.next();
    nphase = __ddiv_rn(__dsub_rn(ph, ratio), __dsub_rn(1.0, ratio));
  }
  state = desired;
  if (nphase < R.contact_detection_phase_threshold) return;
  if (state == RG_LEG_SWING && contact) state = RG_LEG_EARLY_CONTACT;
  if (state == RG_LEG_STANCE && !contact) state = RG_LEG_LOSE_CONTACT;
}

// The desired state alone at time t (OpenloopGaitGenerator.update without the contact detection), in the same
// separately rounded arithmetic as gait_leg: the contact schedule of rg_control_step_plan.
template <class Gait>
__device__ __forceinline__ int gait_desired(const Gait& g, double t) {
  const double period = __ddiv_rn(g.stance(), g.duty());
  const double aug = __dadd_rn(t, __dmul_rn(g.phase0(), period));
  const double ph = __ddiv_rn(fmod(aug, period), period);
  return ph < g.ratio() ? g.init() : g.next();
}

// Rows 1 .. h-1 of one leg's contact schedule: desired stance at t_k = t + k dt (row 0 is the step's own contact flag).
// A gait row that is not valid holds the env in stance over the whole horizon.
template <class Gait>
__device__ __forceinline__ void plan_leg(const Gait& g, bool row_ok, double t, int h, double dt, uint8_t* __restrict__ col) {
  for (int k = 1; k < h; ++k)
    col[4 * k] = row_ok ? (gait_desired(g, __dadd_rn(t, __dmul_rn((double)k, dt))) == RG_LEG_STANCE) : 1;
}

__global__ void gait_kernel(const RgRobotDev* __restrict__ R, int n_env, const double* __restrict__ t,
                            const uint8_t* __restrict__ contacts, int32_t* __restrict__ desired,
                            int32_t* __restrict__ state, double* __restrict__ nphase) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * n_env) return;
  const int env = idx >> 2, leg = idx & 3;
  int d, s;
  double np;
  gait_leg(*R, WorkspaceGait{*R, leg}, t[env], contacts[idx] != 0, d, s, np);
  desired[idx] = d;
  state[idx] = s;
  nphase[idx] = np;
}

// ------------------------------------------------------------------------------------ estimator
// MovingWindowFilter.calculate_average with Neumaier compensated sums (one axis).
__device__ __forceinline__ void neumaier(double& sum, double& corr, double value) {
  const double new_sum = __dadd_rn(sum, value);
  if (fabs(sum) >= fabs(value)) corr = __dadd_rn(corr, __dadd_rn(__dsub_rn(sum, new_sum), value));
  else corr = __dadd_rn(corr, __dadd_rn(__dsub_rn(value, new_sum), sum));
  sum = new_sum;
}

// One axis of the moving-window average: ring-buffer update + Neumaier sums; returns the world-frame average.
__device__ __forceinline__ double com_velocity_axis(int W, int env, int a, int count, int head, const float* __restrict__ vel_world,
                                                    double* window, double* wsum, double* wcorr) {
  double* win = window + ((size_t)env * 3 + a) * W;
  double sum = wsum[3 * (size_t)env + a], corr = wcorr[3 * (size_t)env + a];
  const double nv = (double)vel_world[3 * (size_t)env + a];
  if (count >= W) neumaier(sum, corr, -win[head]);   // deque is full: drop the oldest sample
  neumaier(sum, corr, nv);
  win[head] = nv;
  wsum[3 * (size_t)env + a] = sum;
  wcorr[3 * (size_t)env + a] = corr;
  return __ddiv_rn(__dadd_rn(sum, corr), (double)W);
}

// body frame: R(q)^T v  (pybullet invertTransform + multiplyTransforms)
__device__ __forceinline__ void world_to_body(const float* __restrict__ quat, int env, const double* v_world, double* v_body) {
  const double qx = quat[4 * (size_t)env + 0], qy = quat[4 * (size_t)env + 1], qz = quat[4 * (size_t)env + 2], qw = quat[4 * (size_t)env + 3];
  const double d = qx * qx + qy * qy + qz * qz + qw * qw;
  const double s = 2.0 / d;
  const double xs = qx * s, ys = qy * s, zs = qz * s;
  const double wx = qw * xs, wy = qw * ys, wz = qw * zs, xx = qx * xs, xy = qx * ys, xz = qx * zs, yy = qy * ys, yz = qy * zs, zz = qz * zs;
  const double m[9] = {1.0 - (yy + zz), xy - wz, xz + wy, xy + wz, 1.0 - (xx + zz), yz - wx, xz - wy, yz + wx, 1.0 - (xx + yy)};
  const V3 vb = mat_tmul(m, v3(v_world[0], v_world[1], v_world[2]));
  v_body[0] = vb.x; v_body[1] = vb.y; v_body[2] = vb.z;
}

__device__ __forceinline__ void com_velocity_env(const RgRobotDev& R, int env, const float* __restrict__ vel_world,
                                                 const float* __restrict__ quat, double* window, double* wsum,
                                                 double* wcorr, int32_t* wcount, int32_t* whead,
                                                 double* v_body, double* v_world) {
  const int W = R.velocity_window;
  const int count = wcount[env], head = whead[env];
  for (int a = 0; a < 3; ++a) v_world[a] = com_velocity_axis(W, env, a, count, head, vel_world, window, wsum, wcorr);
  whead[env] = (head + 1) % W;
  if (count < W) wcount[env] = count + 1;
  world_to_body(quat, env, v_world, v_body);
}

__global__ void com_velocity_kernel(const RgRobotDev* __restrict__ R, int n_env, const float* __restrict__ vel_world,
                                    const float* __restrict__ quat, double* window, double* wsum, double* wcorr,
                                    int32_t* wcount, int32_t* whead, float* __restrict__ out_body,
                                    float* __restrict__ out_world) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n_env) return;
  double vb[3], vw[3];
  com_velocity_env(*R, env, vel_world, quat, window, wsum, wcorr, wcount, whead, vb, vw);
  for (int a = 0; a < 3; ++a) {
    out_body[3 * (size_t)env + a] = (float)vb[a];
    if (out_world) out_world[3 * (size_t)env + a] = (float)vw[a];
  }
}

// ------------------------------------------------------------------------------------ swing
__device__ __forceinline__ double gen_parabola(double phase, double start, double mid, double end) {
  const double mid_phase = 0.5;
  const double delta_1 = mid - start, delta_2 = end - start, delta_3 = mid_phase * mid_phase - mid_phase;
  const double coef_a = (delta_1 - delta_2 * mid_phase) / delta_3;
  const double coef_b = (delta_2 * mid_phase * mid_phase - delta_1) / delta_3;
  return coef_a * phase * phase + coef_b * phase + start;
}

// The Raibert foothold of one leg (RaibertSwingLegController.get_action's end point): the swing trajectory's target and
// the touchdown point of the foothold plan (rg_control_step_footholds).
template <class Gait>
__device__ __forceinline__ void raibert_end(const RgRobotDev& R, int leg, const Gait& gait, const double* v_body,
                                            double yaw_dot, const float* cmd, double* end) {
  const double hx = R.hip_positions[leg][0], hy = R.hip_positions[leg][1];
  const double tw[3] = {-hy, hx, 0.0};
  const double cv[3] = {v_body[0], v_body[1], 0.0};
  const double ds[3] = {(double)cmd[0], (double)cmd[1], 0.0};
  const double dtw = (double)cmd[2];
  const double hgt[3] = {0.0, 0.0, R.desired_height - R.foot_clearance};
  const double hip[3] = {hx, hy, 0.0};
  for (int a = 0; a < 3; ++a) {
    const double hv = cv[a] + yaw_dot * tw[a];
    const double thv = ds[a] + dtw * tw[a];
    end[a] = (hv * gait.stance() / 2.0 - R.swing_kp[a] * (thv - hv)) - hgt[a] + hip[a];
  }
}

// Rows 1 .. h-1 of one leg's contact schedule (as plan_leg) and rows 0 .. h-1 of its footholds, in one pass over the
// horizon (rg_control_step_footholds).  col[0] (the step's own contact flag) is written by the caller.  A planted foot
// stays where it is while the body walks over it at the commanded velocity; a touchdown inside the horizon (swing at
// k - 1, stance at k) plants it at the Raibert foothold.  Each product and difference is rounded separately; the yaw
// rate is not integrated (the QP's model holds the yaw).  A gait row that is not valid holds the current foot.
template <class Gait>
__device__ __forceinline__ void plan_leg_feet(const RgRobotDev& R, int leg, const Gait& g, bool row_ok, double t, int h,
                                              double dt, const float* foot, const double* v_body, double yaw_dot,
                                              const float* cmd, uint8_t* __restrict__ col, float* __restrict__ fcol) {
  const double v[2] = {(double)cmd[0], (double)cmd[1]};
  double end[3];
  raibert_end(R, leg, g, v_body, yaw_dot, cmd, end);
  double anchor[3] = {(double)foot[0], (double)foot[1], (double)foot[2]};
  int k_a = 0;
  bool prev = col[0] != 0;
  for (int k = 0; k < h; ++k) {
    bool cur = prev;
    if (k >= 1) {
      cur = row_ok ? (gait_desired(g, __dadd_rn(t, __dmul_rn((double)k, dt))) == RG_LEG_STANCE) : true;
      col[4 * k] = cur ? 1 : 0;
      if (cur && !prev) {   // touchdown (never for an invalid row: all of its rows are stance)
        anchor[0] = end[0]; anchor[1] = end[1]; anchor[2] = end[2];
        k_a = k;
      }
    }
    if (row_ok) {
      const double back = __dmul_rn((double)(k - k_a), dt);
      fcol[12 * k + 0] = (float)__dsub_rn(anchor[0], __dmul_rn(back, v[0]));
      fcol[12 * k + 1] = (float)__dsub_rn(anchor[1], __dmul_rn(back, v[1]));
      fcol[12 * k + 2] = (float)anchor[2];   // v_z = 0
    } else {
      fcol[12 * k + 0] = foot[0]; fcol[12 * k + 1] = foot[1]; fcol[12 * k + 2] = foot[2];
    }
    prev = cur;
  }
}

// RaibertSwingLegController.update (latch) + get_action up to the IK call, for one leg.
// Returns true if a swing target was produced (leg_state not in {STANCE, EARLY_CONTACT}).
template <class Gait>
__device__ __forceinline__ bool swing_leg(const RgRobotDev& R, int leg, const Gait& gait, int desired, int state, double nphase,
                                          const float* foot_pos /* this leg, 3 */, const double* v_body,
                                          double yaw_dot, const float* cmd, int32_t& last_state,
                                          float* latch /* this leg, 3 */, double* target_out) {
  if (desired == RG_LEG_SWING && last_state != desired && last_state >= 0) {
    latch[0] = foot_pos[0]; latch[1] = foot_pos[1]; latch[2] = foot_pos[2];
  }
  last_state = desired;
  if (state == RG_LEG_STANCE || state == RG_LEG_EARLY_CONTACT) return false;
  double end[3];
  raibert_end(R, leg, gait, v_body, yaw_dot, cmd, end);
  // _gen_swing_foot_trajectory
  double phase;
  if (nphase <= 0.5) phase = 0.8 * sin(nphase * 3.14159265358979323846);
  else phase = 0.8 + (nphase - 0.5) * 0.4;
  const double sx = latch[0], sy = latch[1], sz = latch[2];
  target_out[0] = (1.0 - phase) * sx + phase * end[0];
  target_out[1] = (1.0 - phase) * sy + phase * end[1];
  const double mid = fmax(end[2], sz) + R.swing_max_clearance;
  target_out[2] = gen_parabola(phase, sz, mid, end[2]);
  return true;
}

__global__ void swing_kernel(const RgRobotDev* __restrict__ R, int n_env, const int32_t* __restrict__ desired,
                             const int32_t* __restrict__ state, const double* __restrict__ nphase,
                             const float* __restrict__ feet, const float* __restrict__ v_body,
                             const float* __restrict__ rpy_rate, const float* __restrict__ cmd,
                             int32_t* last_state, float* latch, float* __restrict__ target) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * n_env) return;
  const int env = idx >> 2, leg = idx & 3;
  const double vb[3] = {v_body[3 * (size_t)env], v_body[3 * (size_t)env + 1], v_body[3 * (size_t)env + 2]};
  int32_t ls = last_state[idx];
  double tg[3];
  const bool has = swing_leg(*R, leg, WorkspaceGait{*R, leg}, desired[idx], state[idx], nphase[idx], feet + 3 * (size_t)idx, vb,
                             (double)rpy_rate[3 * (size_t)env + 2], cmd + 3 * (size_t)env, ls, latch + 3 * (size_t)idx, tg);
  last_state[idx] = ls;
  if (has) for (int a = 0; a < 3; ++a) target[3 * (size_t)idx + a] = (float)tg[a];
}

// ------------------------------------------------------------------------------------ IK / FK / J^T
__global__ void ik_kernel(const RgRobotDev* __restrict__ R, int n_env, const float* __restrict__ foot,
                          const uint8_t* __restrict__ mask, float* __restrict__ angles) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * n_env) return;
  if (mask && !mask[idx]) return;
  const int leg = idx & 3;
  double q[3];
  leg_ik(R->legs[leg], v3(foot[3 * (size_t)idx], foot[3 * (size_t)idx + 1], foot[3 * (size_t)idx + 2]), q);
  for (int j = 0; j < 3; ++j) {
    const int m = 3 * leg + j;
    angles[3 * (size_t)idx + j] = (float)((q[j] - R->motor_offset[m]) * R->motor_direction[m]);
  }
}

__global__ void fk_kernel(const RgRobotDev* __restrict__ R, int n_env, const float* __restrict__ angles,
                          float* __restrict__ foot) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * n_env) return;
  const int leg = idx & 3;
  double q[3];
  for (int j = 0; j < 3; ++j) {
    const int m = 3 * leg + j;
    q[j] = (double)angles[3 * (size_t)idx + j] * R->motor_direction[m] + R->motor_offset[m];
  }
  const V3 f = leg_fk(R->legs[leg], q, nullptr);
  foot[3 * (size_t)idx] = (float)f.x; foot[3 * (size_t)idx + 1] = (float)f.y; foot[3 * (size_t)idx + 2] = (float)f.z;
}

// ---- state provider: raw rigid-body state -> the controller's inputs ---------------------------------
// One thread per (env, leg): the leg's FK and motor angles; leg 0 also does the base quantities.
__global__ void state_from_sim_kernel(const RgRobotDev* __restrict__ R, int n_env, const float* __restrict__ quat,
                                      const float* __restrict__ ang_vel_world, const float* __restrict__ joint_angles,
                                      float* __restrict__ rpy, float* __restrict__ rpy_rate, float* __restrict__ motor_angles,
                                      float* __restrict__ foot) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * n_env) return;
  const int env = idx >> 2, leg = idx & 3;
  double q[3];
  for (int j = 0; j < 3; ++j) {
    const int m = 3 * leg + j;
    q[j] = joint_angles[12 * (size_t)env + m];
    // Robot.GetMotorAngles (robot.py:231-236): (joint - MOTOR_OFFSET) * MOTOR_DIRECTION
    if (motor_angles) motor_angles[12 * (size_t)env + m] = (float)((q[j] - R->motor_offset[m]) * R->motor_direction[m]);
  }
  if (foot) {
    const V3 f = leg_fk<true>(R->legs[leg], q, nullptr);
    foot[3 * (size_t)idx] = (float)f.x; foot[3 * (size_t)idx + 1] = (float)f.y; foot[3 * (size_t)idx + 2] = (float)f.z;
  }
  if (leg != 0) return;
  const double qx = quat[4 * (size_t)env + 0], qy = quat[4 * (size_t)env + 1], qz = quat[4 * (size_t)env + 2], qw = quat[4 * (size_t)env + 3];
  if (rpy) {
    // Bullet's getEulerFromQuaternion (ZYX convention, with its two gimbal-lock branches)
    const double sqx = qx * qx, sqy = qy * qy, sqz = qz * qz, sqw = qw * qw;
    const double sarg = -2.0 * (qx * qz - qw * qy);
    double roll, pitch, yaw;
    // single-precision inverse trigonometry on double-precision arguments: the outputs are float32
    if (sarg <= -0.99999) { pitch = -0.5 * 3.14159265358979323846; roll = 0.0; yaw = 2.0 * atan2f((float)qx, (float)-qy); }
    else if (sarg >= 0.99999) { pitch = 0.5 * 3.14159265358979323846; roll = 0.0; yaw = 2.0 * atan2f((float)-qx, (float)qy); }
    else {
      roll = atan2f((float)(2.0 * (qy * qz + qw * qx)), (float)(sqw - sqx - sqy + sqz));
      pitch = asinf((float)sarg);
      yaw = atan2f((float)(2.0 * (qx * qy + qw * qz)), (float)(sqw + sqx - sqy - sqz));
    }
    rpy[3 * (size_t)env] = (float)roll; rpy[3 * (size_t)env + 1] = (float)pitch; rpy[3 * (size_t)env + 2] = (float)yaw;
  }
  if (rpy_rate) {
    // Robot.TransformAngularVelocityToLocalFrame (robot.py:185-203): w_body = R(q)^T w_world
    const double wx = ang_vel_world[3 * (size_t)env], wy = ang_vel_world[3 * (size_t)env + 1], wz = ang_vel_world[3 * (size_t)env + 2];
    const double r00 = 1 - 2 * (qy * qy + qz * qz), r01 = 2 * (qx * qy - qz * qw), r02 = 2 * (qx * qz + qy * qw);
    const double r10 = 2 * (qx * qy + qz * qw), r11 = 1 - 2 * (qx * qx + qz * qz), r12 = 2 * (qy * qz - qx * qw);
    const double r20 = 2 * (qx * qz - qy * qw), r21 = 2 * (qy * qz + qx * qw), r22 = 1 - 2 * (qx * qx + qy * qy);
    rpy_rate[3 * (size_t)env] = (float)(r00 * wx + r10 * wy + r20 * wz);
    rpy_rate[3 * (size_t)env + 1] = (float)(r01 * wx + r11 * wy + r21 * wz);
    rpy_rate[3 * (size_t)env + 2] = (float)(r02 * wx + r12 * wy + r22 * wz);
  }
}

__device__ __forceinline__ void leg_torque(const RgRobotDev& R, int leg, const float* force, const float* angles, double* tau) {
  double q[3];
  for (int j = 0; j < 3; ++j) {
    const int m = 3 * leg + j;
    q[j] = (double)angles[j] * R.motor_direction[m] + R.motor_offset[m];
  }
  V3 jac[3];
  leg_fk(R.legs[leg], q, jac);
  const V3 f = v3(force[0], force[1], force[2]);
  for (int j = 0; j < 3; ++j) tau[j] = dot(f, jac[j]) * R.motor_direction[3 * leg + j];
}

__global__ void torque_kernel(const RgRobotDev* __restrict__ R, int n_env, const float* __restrict__ forces,
                              const float* __restrict__ angles, float* __restrict__ torques) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * n_env) return;
  double tau[3];
  leg_torque(*R, idx & 3, forces + 3 * (size_t)idx, angles + 3 * (size_t)idx, tau);
  for (int j = 0; j < 3; ++j) torques[3 * (size_t)idx + j] = (float)tau[j];
}

// ------------------------------------------------------------------------------------ action pack
__device__ __forceinline__ void pack_leg(const RgRobotDev& R, int leg, int desired, bool valid,
                                         const float* swing_angles, const float* tau, float* out15) {
  const bool swing = desired == RG_LEG_SWING && valid;
  for (int j = 0; j < 3; ++j) {
    const int m = 3 * leg + j;
    float* o = out15 + 5 * j;
    if (swing) { o[0] = swing_angles[j]; o[1] = (float)R.motor_kp[m]; o[2] = 0.f; o[3] = (float)R.motor_kd[m]; o[4] = 0.f; }
    else { o[0] = 0.f; o[1] = 0.f; o[2] = 0.f; o[3] = 0.f; o[4] = tau[j]; }
  }
}

__global__ void pack_kernel(const RgRobotDev* __restrict__ R, int n_env, const int32_t* __restrict__ desired,
                            const float* __restrict__ swing_angles, const uint8_t* __restrict__ valid,
                            const float* __restrict__ torques, float* __restrict__ action) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * n_env) return;
  pack_leg(*R, idx & 3, desired[idx], valid[idx] != 0, swing_angles + 3 * (size_t)idx, torques + 3 * (size_t)idx,
           action + 15 * (size_t)idx);
}

// ------------------------------------------------------------------------------------ fused step
// Prologue: gait + estimator + swing latch/target + IK, one thread per (env, leg): the four legs of an env are four
// adjacent lanes; the estimator's three axes are updated by the lanes of legs 0-2 and handed round with shuffles (a
// single thread per env did the four legs and three axes one after the other: 4x the dependent chain at N = 1 and a
// quarter of the threads at large N).  Epilogue: J^T force -> torque + pack, one thread per leg.
// Gait = EnvGait: the gait of each env comes from `gp` (rg_gait_env_params) instead of the workspace.  The gait-free
// kernels instantiate the bodies with WorkspaceGait and keep their own parameter list (an extra kernel parameter, even an
// unused one, moves ptxas's register assignment: DESIGN.md §3.12), so they compile to the code they had before the
// per-env gait existed (DESIGN.md §3.14).
// PLAN = true (Gait = EnvGait): the prologue also writes the env's contact schedule `plan` ([N,h,4], rg_control_step_plan).
// FEET = true (with PLAN): ... and its foothold plan `feet` ([N,h,12], rg_control_step_footholds).
template <class Gait, bool PLAN = false, bool FEET = false>
__device__ __forceinline__ void step_prologue_leg(const RgRobotDev* __restrict__ R, int n_env, const rg_controller_state& s,
                                                  const rg_gait_env_params& gp, uint8_t* __restrict__ plan = nullptr,
                                                  int h = 0, double dt = 0.0, float* __restrict__ feet = nullptr) {
  RG_GRID_LAUNCH_DEPENDENTS();   // the solve kernel is launched programmatically behind this grid (rg_control_step)
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int env = (int)(idx >> 2), leg = (int)(idx & 3);
  const bool ok = env < n_env;
  // estimator: every lane reads the ring-buffer cursor before the lane of leg 3 advances it
  const int W = R->velocity_window;
  int count = 0, head = 0;
  if (ok) { count = s.vel_window_count[env]; head = s.vel_window_head[env]; }
  __syncwarp();
  double vw_axis = 0.0;
  if (ok && leg < 3) vw_axis = com_velocity_axis(W, env, leg, count, head, s.base_velocity_world, s.vel_window, s.vel_window_sum, s.vel_window_corr);
  if (ok && leg == 3) {
    s.vel_window_head[env] = (head + 1) % W;
    if (count < W) s.vel_window_count[env] = count + 1;
  }
  const int lane0 = (int)(threadIdx.x & 31u) & ~3;
  double vw[3];
  for (int a = 0; a < 3; ++a) vw[a] = __shfl_sync(0xffffffffu, vw_axis, lane0 + a);
  if (!ok) return;
  double vb[3];
  world_to_body(s.base_orientation_xyzw, env, vw, vb);
  const float vbf[3] = {(float)vb[0], (float)vb[1], (float)vb[2]};
  if (leg < 3) s.com_velocity_body[3 * (size_t)env + leg] = leg == 0 ? vbf[0] : (leg == 1 ? vbf[1] : vbf[2]);
  // the swing controller and the MPC read the estimator output as the reference does: float64 in the
  // reference, float32 state arrays here -> use the float32-rounded value everywhere for consistency
  const double vbr[3] = {(double)vbf[0], (double)vbf[1], (double)vbf[2]};
  const double t = s.time_since_reset[env];
  const double yaw_dot = (double)s.base_rpy_rate[3 * (size_t)env + 2];
  int d, st;
  double np;
  const Gait g = Gait::load(*R, gp, idx, leg);
  // a row is valid when its four legs are: the four lanes of the env vote (all four are past the `ok` return)
  const bool row_ok = !Gait::kPerEnv || __all_sync(0xfu << lane0, g.valid());
  if (row_ok) {
    gait_leg(*R, g, t, s.foot_contacts[idx] != 0, d, st, np);
  } else {
    d = st = RG_LEG_STANCE;
    np = -1.0;
  }
  s.desired_leg_state[idx] = d;
  s.leg_state[idx] = st;
  s.normalized_phase[idx] = np;
  s.mpc_contact_state[idx] = (d == RG_LEG_STANCE || d == RG_LEG_EARLY_CONTACT) ? 1 : 0;
  if constexpr (PLAN) {
    uint8_t* col = plan + 4 * (size_t)h * env + leg;
    col[0] = (d == RG_LEG_STANCE || d == RG_LEG_EARLY_CONTACT) ? 1 : 0;
    if constexpr (FEET)
      plan_leg_feet(*R, leg, g, row_ok, t, h, dt, s.foot_positions_base + 3 * idx, vbr, yaw_dot, s.command + 3 * (size_t)env,
                    col, feet + 12 * (size_t)h * env + 3 * leg);
    else
      plan_leg(g, row_ok, t, h, dt, col);
  }
  int32_t ls = s.last_leg_state[idx];
  double tg[3];
  const bool has = swing_leg(*R, leg, g, d, st, np, s.foot_positions_base + 3 * idx, vbr, yaw_dot,
                             s.command + 3 * (size_t)env, ls, s.phase_switch_foot_local_position + 3 * idx, tg);
  s.last_leg_state[idx] = ls;
  if (has) {
    const float tf[3] = {(float)tg[0], (float)tg[1], (float)tg[2]};
    double q[3];
    leg_ik(R->legs[leg], v3(tf[0], tf[1], tf[2]), q);
    for (int j = 0; j < 3; ++j) {
      const int m = 3 * leg + j;
      s.swing_foot_target[3 * idx + j] = tf[j];
      s.swing_joint_angles[3 * idx + j] = (float)((q[j] - R->motor_offset[m]) * R->motor_direction[m]);
    }
    s.swing_joint_valid[idx] = 1;
  }
}

// The same prologue with one thread per env (the four legs unrolled): fewer, fatter threads -- the faster mapping for
// large batches, where the kernel is bound by its FP64 instruction count and per-leg lanes diverge (swing legs run the IK,
// stance legs idle).  Bit-identical results: both call the same per-leg / per-axis routines.
template <class Gait, bool PLAN = false, bool FEET = false>
__device__ __forceinline__ void step_prologue_env(const RgRobotDev* __restrict__ R, int n_env, const rg_controller_state& s,
                                                  const rg_gait_env_params& gp, uint8_t* __restrict__ plan = nullptr,
                                                  int h = 0, double dt = 0.0, float* __restrict__ feet = nullptr) {
  RG_GRID_LAUNCH_DEPENDENTS();   // the solve kernel is launched programmatically behind this grid (rg_control_step)
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n_env) return;
  double vb[3], vw[3];
  com_velocity_env(*R, env, s.base_velocity_world, s.base_orientation_xyzw, s.vel_window, s.vel_window_sum,
                   s.vel_window_corr, s.vel_window_count, s.vel_window_head, vb, vw);
  const float vbf[3] = {(float)vb[0], (float)vb[1], (float)vb[2]};
  for (int a = 0; a < 3; ++a) s.com_velocity_body[3 * (size_t)env + a] = vbf[a];
  // the swing controller and the MPC read the estimator output as the reference does: float64 in the
  // reference, float32 state arrays here -> use the float32-rounded value everywhere for consistency
  const double vbr[3] = {(double)vbf[0], (double)vbf[1], (double)vbf[2]};
  const double t = s.time_since_reset[env];
  const double yaw_dot = (double)s.base_rpy_rate[3 * (size_t)env + 2];
  // the row's validity first (a pass over its four legs: holding the four legs' values live costs registers)
  bool valid = true;
  if (Gait::kPerEnv)
    for (int leg = 0; leg < 4; ++leg) valid = valid && Gait::load(*R, gp, 4 * (size_t)env + leg, leg).valid();
  unsigned row0 = 0u;   // PLAN: the env's planned-stance word of horizon step 0
  for (int leg = 0; leg < 4; ++leg) {
    const size_t idx = 4 * (size_t)env + leg;
    int d, st;
    double np;
    const Gait g = Gait::load(*R, gp, idx, leg);
    if (valid) {
      gait_leg(*R, g, t, s.foot_contacts[idx] != 0, d, st, np);
    } else {
      d = st = RG_LEG_STANCE;
      np = -1.0;
    }
    s.desired_leg_state[idx] = d;
    s.leg_state[idx] = st;
    s.normalized_phase[idx] = np;
    s.mpc_contact_state[idx] = (d == RG_LEG_STANCE || d == RG_LEG_EARLY_CONTACT) ? 1 : 0;
    if constexpr (PLAN) row0 |= (d == RG_LEG_STANCE || d == RG_LEG_EARLY_CONTACT) ? 1u << (8 * leg) : 0u;
    if constexpr (FEET) {   // the leg's schedule column and footholds in one pass (byte stores instead of row words)
      uint8_t* col = plan + 4 * (size_t)h * env + leg;
      col[0] = (d == RG_LEG_STANCE || d == RG_LEG_EARLY_CONTACT) ? 1 : 0;
      plan_leg_feet(*R, leg, g, valid, t, h, dt, s.foot_positions_base + 3 * idx, vbr, yaw_dot, s.command + 3 * (size_t)env,
                    col, feet + 12 * (size_t)h * env + 3 * leg);
    }
    int32_t ls = s.last_leg_state[idx];
    double tg[3];
    const bool has = swing_leg(*R, leg, g, d, st, np, s.foot_positions_base + 3 * idx, vbr, yaw_dot,
                               s.command + 3 * (size_t)env, ls, s.phase_switch_foot_local_position + 3 * idx, tg);
    s.last_leg_state[idx] = ls;
    if (has) {
      const float tf[3] = {(float)tg[0], (float)tg[1], (float)tg[2]};
      double q[3];
      leg_ik(R->legs[leg], v3(tf[0], tf[1], tf[2]), q);
      for (int j = 0; j < 3; ++j) {
        const int m = 3 * leg + j;
        s.swing_foot_target[3 * idx + j] = tf[j];
        s.swing_joint_angles[3 * idx + j] = (float)((q[j] - R->motor_offset[m]) * R->motor_direction[m]);
      }
      s.swing_joint_valid[idx] = 1;
    }
  }
  if constexpr (PLAN && !FEET) {   // one 4-byte store per row: the row's four leg bytes assembled in a register
    unsigned* rows = reinterpret_cast<unsigned*>(plan + 4 * (size_t)h * env);
    rows[0] = row0;
    for (int k = 1; k < h; ++k) {
      const double tk = __dadd_rn(t, __dmul_rn((double)k, dt));
      unsigned w = 0x01010101u;
      if (valid) {
        w = 0u;
        for (int leg = 0; leg < 4; ++leg)
          if (gait_desired(Gait::load(*R, gp, 4 * (size_t)env + leg, leg), tk) == RG_LEG_STANCE) w |= 1u << (8 * leg);
      }
      rows[k] = w;
    }
  }
}

__global__ void step_prologue_kernel(const RgRobotDev* __restrict__ R, int n_env, rg_controller_state s) {
  step_prologue_leg<WorkspaceGait>(R, n_env, s, rg_gait_env_params{});
}

__global__ void step_prologue_env_kernel(const RgRobotDev* __restrict__ R, int n_env, rg_controller_state s) {
  step_prologue_env<WorkspaceGait>(R, n_env, s, rg_gait_env_params{});
}

// Per-env gait (rg_control_step_env): each (env, leg) loads its own 28 B of gait arguments, coalesced in the per-leg
// mapping.  An invalid row holds its env in stance (rg_cuda.h).
__global__ void step_prologue_gait_kernel(const RgRobotDev* __restrict__ R, int n_env, rg_controller_state s,
                                          rg_gait_env_params gp) {
  step_prologue_leg<EnvGait>(R, n_env, s, gp);
}

__global__ void step_prologue_env_gait_kernel(const RgRobotDev* __restrict__ R, int n_env, rg_controller_state s,
                                              rg_gait_env_params gp) {
  step_prologue_env<EnvGait>(R, n_env, s, gp);
}

// Contact-schedule twins (rg_control_step_plan): always with EnvGait, whose NULL arrays stand for the workspace's gait.
__global__ void step_prologue_plan_kernel(const RgRobotDev* __restrict__ R, int n_env, rg_controller_state s,
                                          rg_gait_env_params gp, uint8_t* __restrict__ plan, int h, double dt) {
  step_prologue_leg<EnvGait, true>(R, n_env, s, gp, plan, h, dt);
}

__global__ void step_prologue_env_plan_kernel(const RgRobotDev* __restrict__ R, int n_env, rg_controller_state s,
                                              rg_gait_env_params gp, uint8_t* __restrict__ plan, int h, double dt) {
  step_prologue_env<EnvGait, true>(R, n_env, s, gp, plan, h, dt);
}

// Foothold-plan twins (rg_control_step_footholds): the schedule twins that also write the foothold plan.
__global__ void step_prologue_feet_kernel(const RgRobotDev* __restrict__ R, int n_env, rg_controller_state s,
                                          rg_gait_env_params gp, uint8_t* __restrict__ plan, float* __restrict__ feet,
                                          int h, double dt) {
  step_prologue_leg<EnvGait, true, true>(R, n_env, s, gp, plan, h, dt, feet);
}

__global__ void step_prologue_env_feet_kernel(const RgRobotDev* __restrict__ R, int n_env, rg_controller_state s,
                                              rg_gait_env_params gp, uint8_t* __restrict__ plan, float* __restrict__ feet,
                                              int h, double dt) {
  step_prologue_env<EnvGait, true, true>(R, n_env, s, gp, plan, h, dt, feet);
}

__global__ void step_epilogue_kernel(const RgRobotDev* __restrict__ R, int n_env, rg_controller_state s) {
  RG_GRID_WAIT();                // launched programmatically behind the last solve kernel: its forces must be complete
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * n_env) return;
  const int leg = idx & 3;
  double tau[3];
  leg_torque(*R, leg, s.contact_forces + 3 * (size_t)idx, s.motor_angles + 3 * (size_t)idx, tau);
  float tf[3];
  for (int j = 0; j < 3; ++j) { tf[j] = (float)tau[j]; s.motor_torques[3 * (size_t)idx + j] = tf[j]; }
  float cmd[15];
  pack_leg(*R, leg, s.desired_leg_state[idx], s.swing_joint_valid[idx] != 0, s.swing_joint_angles + 3 * (size_t)idx, tf, cmd);
  for (int i = 0; i < 15; ++i) s.action[15 * (size_t)idx + i] = cmd[i];
  if (s.applied_motor_torques) {
    // torque consumer attached: HYBRID motor model on the command just packed (first physics tick of the step)
    for (int j = 0; j < 3; ++j) {
      const size_t m = 3 * (size_t)idx + j;
      const float* a = cmd + 5 * j;
      float tau = -1.f * (a[1] * (s.motor_angles[m] - a[0])) - a[3] * (s.motor_velocities[m] - a[2]) + a[4];
      if (s.motor_strength_ratios) tau *= s.motor_strength_ratios[m];
      s.applied_motor_torques[m] = tau * (float)R->motor_direction[3 * leg + j];
    }
  }
}

__global__ void hybrid_motor_kernel(int n, const float* __restrict__ action, const float* __restrict__ q,
                                    const float* __restrict__ qd, float* __restrict__ tau) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // over N*12 motors
  if (idx >= n) return;
  const float* a = action + 5 * (size_t)idx;
  // -1 * (kp * (q - q_des)) - kd * (qd - qd_des) + tau_ff   (simple_motor.py:138-139)
  tau[idx] = -1.f * (a[1] * (q[idx] - a[0])) - a[3] * (qd[idx] - a[2]) + a[4];
}

__global__ void hybrid_motor_ex_kernel(const RgRobotDev* __restrict__ R, int n, const float* __restrict__ action,
                                       const float* __restrict__ q, const float* __restrict__ qd,
                                       const float* __restrict__ strength, float* __restrict__ observed,
                                       float* __restrict__ applied) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // over N*12 motors
  if (idx >= n) return;
  const float* a = action + 5 * (size_t)idx;
  float tau = -1.f * (a[1] * (q[idx] - a[0])) - a[3] * (qd[idx] - a[2]) + a[4];
  if (strength) tau *= strength[idx];                      // simple_motor.py:140
  if (observed) observed[idx] = tau;
  if (applied) applied[idx] = tau * (float)R->motor_direction[idx % RG_NUM_MOTORS];   // robot.py:291-292
}

// ------------------------------------------------------------------------------------ host: setup
bool near_zero(double v) { return fabs(v) < 1e-3; }   // URDF right angles are given to 5 digits

int derive_ik_constants(const rg_leg_chain& c, RgLegDev& L, int leg) {
  memcpy(L.p, c.p, sizeof(L.p));
  memcpy(L.r, c.r, sizeof(L.r));
  memcpy(L.toe, c.toe, sizeof(L.toe));
  for (int j = 0; j < 3; ++j) {
    const double n = sqrt(c.axis[j][0] * c.axis[j][0] + c.axis[j][1] * c.axis[j][1] + c.axis[j][2] * c.axis[j][2]);
    if (n < 1e-12) { rg_set_error("leg %d joint %d: zero axis", leg, j); return RG_ERR_BAD_ARG; }
    for (int a = 0; a < 3; ++a) L.axis[j][a] = c.axis[j][a] / n;
  }
  const V3 a0 = ld3(L.axis[0]), a1 = ld3(L.axis[1]), a2 = ld3(L.axis[2]);
  const V3 e0 = a0;
  const V3 e1 = mat_mul(L.r[1], a1);
  if (!near_zero(dot(e0, e1))) {
    rg_set_error("leg %d: upper joint axis is not perpendicular to the hip axis (closed-form IK unsupported)", leg);
    return RG_ERR_UNSUPPORTED;
  }
  const V3 e2 = cross(e0, e1);
  const V3 a2_in1 = mat_mul(L.r[2], a2);          // lower axis seen from the upper-joint frame
  const double par = dot(a2_in1, a1);
  if (fabs(fabs(par) - 1.0) > 1e-6) {
    rg_set_error("leg %d: lower joint axis is not parallel to the upper axis (closed-form IK unsupported)", leg);
    return RG_ERR_UNSUPPORTED;
  }
  L.s2 = par > 0 ? 1.0 : -1.0;
  L.e0[0] = e0.x; L.e0[1] = e0.y; L.e0[2] = e0.z;
  L.e1[0] = e1.x; L.e1[1] = e1.y; L.e1[2] = e1.z;
  L.e2[0] = e2.x; L.e2[1] = e2.y; L.e2[2] = e2.z;
  const V3 p1 = ld3(L.p[1]), p2 = ld3(L.p[2]);
  const V3 toe1 = mat_mul(L.r[2], ld3(L.toe));    // toe offset in the upper-joint frame at q2 = 0
  L.t1e0 = dot(p1, e0);
  L.t1e2 = dot(p1, e2);
  L.dconst = dot(p1, e1) + dot(a1, p2) + dot(a1, toe1);
  const V3 l1v = sub(p2, mul(dot(a1, p2), a1));
  const V3 l2v = sub(toe1, mul(dot(a1, toe1), a1));
  L.l1 = sqrt(dot(l1v, l1v));
  L.l2 = sqrt(dot(l2v, l2v));
  if (L.l1 < 1e-9 || L.l2 < 1e-9) { rg_set_error("leg %d: degenerate link length", leg); return RG_ERR_UNSUPPORTED; }
  const V3 bx = mul(1.0 / L.l1, l1v);
  const V3 by = cross(a1, bx);
  L.phi2 = atan2(dot(l2v, by), dot(l2v, bx));
  const V3 bxh = mat_mul(L.r[1], bx);             // plane basis vector in the hip-link frame
  L.psi = atan2(dot(bxh, e0), dot(bxh, e2));
  L.sign_hip = c.ik_sign_hip >= 0 ? 1.0 : -1.0;
  L.sign_knee = c.ik_sign_knee >= 0 ? 1.0 : -1.0;
  return RG_OK;
}

inline int grid_for(int n, int block) { return (n + block - 1) / block; }

}  // namespace

// Chooses the two IK branch signs of every leg so that IK(FK(q_ref)) == q_ref (host only).
extern "C" int rg_robot_calibrate_ik(rg_robot_params* p, const double* ref_motor_angles) {
  if (!p || !ref_motor_angles) { rg_set_error("rg_robot_calibrate_ik: NULL argument"); return RG_ERR_BAD_ARG; }
  for (int l = 0; l < RG_NUM_LEGS; ++l) {
    double q_ref[3];
    for (int j = 0; j < 3; ++j) {
      const int m = 3 * l + j;
      q_ref[j] = ref_motor_angles[m] * p->motor_direction[m] + p->motor_offset[m];
    }
    double best = 1e30;
    double best_h = 1.0, best_k = 1.0;
    for (int sh = -1; sh <= 1; sh += 2)
      for (int sk = -1; sk <= 1; sk += 2) {
        rg_leg_chain c = p->legs[l];
        c.ik_sign_hip = sh;
        c.ik_sign_knee = sk;
        RgLegDev L;
        int rc = derive_ik_constants(c, L, l);
        if (rc != RG_OK) return rc;
        const V3 foot = leg_fk(L, q_ref, nullptr);
        double q[3];
        leg_ik(L, foot, q);
        double err = 0.0;
        for (int j = 0; j < 3; ++j) err += fabs(wrap_pi(q[j] - q_ref[j]));
        if (err < best) { best = err; best_h = sh; best_k = sk; }
      }
    if (best > 1e-6) {
      rg_set_error("leg %d: no IK branch reproduces the reference pose (residual %.3g rad)", l, best);
      return RG_ERR_UNSUPPORTED;
    }
    p->legs[l].ik_sign_hip = best_h;
    p->legs[l].ik_sign_knee = best_k;
  }
  return RG_OK;
}

extern "C" int rg_robot_workspace_bytes(size_t* bytes) {
  if (!bytes) { rg_set_error("rg_robot_workspace_bytes: NULL"); return RG_ERR_BAD_ARG; }
  *bytes = (sizeof(RgRobotDev) + 255) & ~size_t(255);
  return RG_OK;
}

extern "C" int rg_robot_setup(const rg_robot_params* p, void* ws, size_t bytes, void* stream) {
  if (!p || !ws) { rg_set_error("rg_robot_setup: NULL argument"); return RG_ERR_BAD_ARG; }
  if (bytes < sizeof(RgRobotDev)) { rg_set_error("robot workspace too small: %zu < %zu", bytes, sizeof(RgRobotDev)); return RG_ERR_WORKSPACE; }
  if (p->velocity_window < 1 || p->velocity_window > RG_VEL_WINDOW_MAX) {
    rg_set_error("velocity_window %d outside [1, %d]", p->velocity_window, RG_VEL_WINDOW_MAX);
    return RG_ERR_UNSUPPORTED;
  }
  static RgRobotDev h;   // large: keep off the stack
  memset(&h, 0, sizeof(h));
  h.magic = RG_WS_MAGIC_ROBOT;
  h.velocity_window = p->velocity_window;
  for (int l = 0; l < RG_NUM_LEGS; ++l) {
    int rc = derive_ik_constants(p->legs[l], h.legs[l], l);
    if (rc != RG_OK) return rc;
    memcpy(h.hip_positions[l], p->hip_positions[l], 3 * sizeof(double));
    if (!(p->stance_duration[l] > 0) || !(p->duty_factor[l] > 0) || p->duty_factor[l] > 1.0) {
      rg_set_error("leg %d: need stance_duration>0 and 0<duty_factor<=1", l);
      return RG_ERR_BAD_ARG;
    }
    h.stance_duration[l] = p->stance_duration[l];
    h.duty_factor[l] = p->duty_factor[l];
    h.initial_leg_phase[l] = p->initial_leg_phase[l];
    h.initial_leg_state[l] = p->initial_leg_state[l];
    // OpenloopGaitGenerator.__init__: ratio = 1 - duty (SWING first) or duty (otherwise)
    if (p->initial_leg_state[l] == RG_LEG_SWING) {
      h.initial_state_ratio[l] = 1.0 - p->duty_factor[l];
      h.next_leg_state[l] = RG_LEG_STANCE;
    } else {
      h.initial_state_ratio[l] = p->duty_factor[l];
      h.next_leg_state[l] = RG_LEG_SWING;
    }
  }
  for (int m = 0; m < RG_NUM_MOTORS; ++m) {
    if (fabs(fabs(p->motor_direction[m]) - 1.0) > 1e-12) { rg_set_error("motor_direction[%d] must be +-1", m); return RG_ERR_BAD_ARG; }
    h.motor_offset[m] = p->motor_offset[m];
    h.motor_direction[m] = p->motor_direction[m];
    h.motor_kp[m] = p->motor_kp[m];
    h.motor_kd[m] = p->motor_kd[m];
  }
  h.contact_detection_phase_threshold = p->contact_detection_phase_threshold;
  h.desired_height = p->desired_height;
  h.foot_clearance = p->foot_clearance;
  for (int a = 0; a < 3; ++a) h.swing_kp[a] = p->swing_kp[a];
  h.swing_max_clearance = p->swing_max_clearance;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = rg_check_cuda(cudaMemcpyAsync(ws, &h, sizeof(h), cudaMemcpyHostToDevice, st), "rg_robot_setup upload");
  if (rc != RG_OK) return rc;
  return rg_check_cuda(cudaStreamSynchronize(st), "rg_robot_setup sync");
}

#define RG_REQUIRE(cond, name)                                             \
  do {                                                                     \
    if (!(cond)) { rg_set_error("%s: NULL or invalid argument", name); return RG_ERR_BAD_ARG; } \
  } while (0)

extern "C" int rg_gait_step(const void* ws, int n_env, const double* t, const uint8_t* contacts,
                            int32_t* desired, int32_t* state, double* nphase, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  RG_REQUIRE(ws && t && contacts && desired && state && nphase && n_env >= 0, "rg_gait_step");
  gait_kernel<<<grid_for(4 * n_env, 256), 256, 0, (cudaStream_t)stream>>>((const RgRobotDev*)ws, n_env, t, contacts, desired, state, nphase);
  rg_count_launch();
  return rg_check_cuda(cudaGetLastError(), "gait_kernel launch");
}

extern "C" int rg_com_velocity_update(const void* ws, int n_env, const float* vel_world, const float* quat,
                                      double* window, double* wsum, double* wcorr, int32_t* wcount, int32_t* whead,
                                      float* v_body, float* v_world, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  RG_REQUIRE(ws && vel_world && quat && window && wsum && wcorr && wcount && whead && v_body && n_env >= 0, "rg_com_velocity_update");
  com_velocity_kernel<<<grid_for(n_env, 128), 128, 0, (cudaStream_t)stream>>>((const RgRobotDev*)ws, n_env, vel_world, quat, window,
                                                                             wsum, wcorr, wcount, whead, v_body, v_world);
  rg_count_launch();
  return rg_check_cuda(cudaGetLastError(), "com_velocity_kernel launch");
}

extern "C" int rg_swing_targets(const void* ws, int n_env, const int32_t* desired, const int32_t* state,
                                const double* nphase, const float* feet, const float* v_body, const float* rpy_rate,
                                const float* cmd, int32_t* last_state, float* latch, float* target, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  RG_REQUIRE(ws && desired && state && nphase && feet && v_body && rpy_rate && cmd && last_state && latch && target && n_env >= 0,
             "rg_swing_targets");
  swing_kernel<<<grid_for(4 * n_env, 256), 256, 0, (cudaStream_t)stream>>>((const RgRobotDev*)ws, n_env, desired, state, nphase, feet,
                                                                          v_body, rpy_rate, cmd, last_state, latch, target);
  rg_count_launch();
  return rg_check_cuda(cudaGetLastError(), "swing_kernel launch");
}

extern "C" int rg_leg_ik(const void* ws, int n_env, const float* foot, const uint8_t* mask, float* angles, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  RG_REQUIRE(ws && foot && angles && n_env >= 0, "rg_leg_ik");
  ik_kernel<<<grid_for(4 * n_env, 256), 256, 0, (cudaStream_t)stream>>>((const RgRobotDev*)ws, n_env, foot, mask, angles);
  rg_count_launch();
  return rg_check_cuda(cudaGetLastError(), "ik_kernel launch");
}

extern "C" int rg_leg_fk(const void* ws, int n_env, const float* angles, float* foot, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  RG_REQUIRE(ws && foot && angles && n_env >= 0, "rg_leg_fk");
  fk_kernel<<<grid_for(4 * n_env, 256), 256, 0, (cudaStream_t)stream>>>((const RgRobotDev*)ws, n_env, angles, foot);
  rg_count_launch();
  return rg_check_cuda(cudaGetLastError(), "fk_kernel launch");
}

extern "C" int rg_state_from_sim(const void* ws, int n_env, const float* base_quat, const float* base_ang_vel_world,
                                 const float* joint_angles, float* base_rpy, float* base_rpy_rate, float* motor_angles,
                                 float* foot_positions_base, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  RG_REQUIRE(ws && base_quat && joint_angles && n_env >= 0 && (!base_rpy_rate || base_ang_vel_world) &&
             (base_rpy || base_rpy_rate || motor_angles || foot_positions_base), "rg_state_from_sim");
  state_from_sim_kernel<<<grid_for(4 * n_env, 256), 256, 0, (cudaStream_t)stream>>>(
      (const RgRobotDev*)ws, n_env, base_quat, base_ang_vel_world, joint_angles, base_rpy, base_rpy_rate, motor_angles, foot_positions_base);
  rg_count_launch();
  return rg_check_cuda(cudaGetLastError(), "state_from_sim_kernel launch");
}

extern "C" int rg_force_to_torque(const void* ws, int n_env, const float* forces, const float* angles, float* torques, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  RG_REQUIRE(ws && forces && angles && torques && n_env >= 0, "rg_force_to_torque");
  torque_kernel<<<grid_for(4 * n_env, 256), 256, 0, (cudaStream_t)stream>>>((const RgRobotDev*)ws, n_env, forces, angles, torques);
  rg_count_launch();
  return rg_check_cuda(cudaGetLastError(), "torque_kernel launch");
}

extern "C" int rg_pack_hybrid_action(const void* ws, int n_env, const int32_t* desired, const float* swing_angles,
                                     const uint8_t* valid, const float* torques, float* action, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  RG_REQUIRE(ws && desired && swing_angles && valid && torques && action && n_env >= 0, "rg_pack_hybrid_action");
  pack_kernel<<<grid_for(4 * n_env, 256), 256, 0, (cudaStream_t)stream>>>((const RgRobotDev*)ws, n_env, desired, swing_angles, valid, torques, action);
  rg_count_launch();
  return rg_check_cuda(cudaGetLastError(), "pack_kernel launch");
}

extern "C" int rg_hybrid_motor_torque(int n_env, const float* action, const float* q, const float* qd, float* tau, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  RG_REQUIRE(action && q && qd && tau && n_env >= 0, "rg_hybrid_motor_torque");
  hybrid_motor_kernel<<<grid_for(12 * n_env, 256), 256, 0, (cudaStream_t)stream>>>(12 * n_env, action, q, qd, tau);
  rg_count_launch();
  return rg_check_cuda(cudaGetLastError(), "hybrid_motor_kernel launch");
}

extern "C" int rg_hybrid_motor_torque_ex(const void* ws, int n_env, const float* action, const float* q, const float* qd,
                                         const float* strength, float* observed, float* applied, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  RG_REQUIRE(ws && action && q && qd && (observed || applied) && n_env >= 0, "rg_hybrid_motor_torque_ex");
  hybrid_motor_ex_kernel<<<grid_for(12 * n_env, 256), 256, 0, (cudaStream_t)stream>>>((const RgRobotDev*)ws, 12 * n_env, action, q, qd,
                                                                                       strength, observed, applied);
  rg_count_launch();
  return rg_check_cuda(cudaGetLastError(), "hybrid_motor_ex_kernel launch");
}

// Batches up to this many envs run the per-(env, leg) prologue (a quarter of the dependent chain per thread), larger ones
// the per-env one.  Measured on the B200 (tools/gpu/lat_step.py, warm-started control step): per leg -8 us at 1 ... 1024
// envs (88 -> 80 us with the Python call), -9 us at 4096, -6 us at 16384, +13 us at 65536.
constexpr int kPrologueLegMaxEnvs = 32768;

extern "C" int rg_control_step(const void* mpc_ws, const void* robot_ws, int n_env, const rg_controller_state* s, void* stream) {
  return rg_control_step_model(mpc_ws, robot_ws, n_env, s, nullptr, stream);
}

extern "C" int rg_control_step_model(const void* mpc_ws, const void* robot_ws, int n_env, const rg_controller_state* s,
                                     const rg_mpc_env_model* model, void* stream) {
  return rg_control_step_env(mpc_ws, robot_ws, n_env, s, model, nullptr, stream);
}

// NULL, or a gait whose four pointers are all NULL -> NULL (the gait-free prologues); RG_ERR_BAD_ARG for a misaligned array
static int rg_check_env_gait(const rg_gait_env_params* gait, const char* what, const rg_gait_env_params** out) {
  *out = nullptr;
  if (!gait || (!gait->stance_duration && !gait->duty_factor && !gait->initial_leg_phase && !gait->initial_leg_state)) return RG_OK;
  if (((uintptr_t)gait->stance_duration | (uintptr_t)gait->duty_factor | (uintptr_t)gait->initial_leg_phase) & 7u) {
    rg_set_error("%s: gait arrays stance_duration, duty_factor and initial_leg_phase must be 8-byte aligned float64", what);
    return RG_ERR_BAD_ARG;
  }
  if ((uintptr_t)gait->initial_leg_state & 3u) {
    rg_set_error("%s: gait array initial_leg_state must be 4-byte aligned int32", what);
    return RG_ERR_BAD_ARG;
  }
  *out = gait;
  return RG_OK;
}

extern "C" int rg_control_step_env(const void* mpc_ws, const void* robot_ws, int n_env, const rg_controller_state* s,
                                   const rg_mpc_env_model* model, const rg_gait_env_params* gait, void* stream) {
  return rg_control_step_plan(mpc_ws, robot_ws, n_env, s, model, gait, nullptr, stream);
}

extern "C" int rg_control_step_plan(const void* mpc_ws, const void* robot_ws, int n_env, const rg_controller_state* s,
                                    const rg_mpc_env_model* model, const rg_gait_env_params* gait, uint8_t* plan,
                                    void* stream) {
  return rg_control_step_footholds(mpc_ws, robot_ws, n_env, s, model, gait, plan, nullptr, stream);
}

extern "C" int rg_control_step_footholds(const void* mpc_ws, const void* robot_ws, int n_env, const rg_controller_state* s,
                                         const rg_mpc_env_model* model, const rg_gait_env_params* gait, uint8_t* plan,
                                         float* feet, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  RG_REQUIRE(mpc_ws && robot_ws && s && n_env >= 0, "rg_control_step");
  RG_REQUIRE(s->time_since_reset && s->foot_contacts && s->base_velocity_world && s->base_orientation_xyzw && s->base_rpy &&
             s->base_rpy_rate && s->foot_positions_base && s->motor_angles && s->command, "rg_control_step inputs");
  RG_REQUIRE(s->vel_window && s->vel_window_sum && s->vel_window_corr && s->vel_window_count && s->vel_window_head &&
             s->last_leg_state && s->phase_switch_foot_local_position && s->swing_joint_angles && s->swing_joint_valid,
             "rg_control_step state");
  RG_REQUIRE(s->desired_leg_state && s->leg_state && s->normalized_phase && s->mpc_contact_state && s->swing_foot_target &&
             s->com_velocity_body && s->contact_forces && s->motor_torques && s->action, "rg_control_step outputs");
  RG_REQUIRE(!s->applied_motor_torques || s->motor_velocities, "rg_control_step torque consumer (motor_velocities)");
  RG_REQUIRE(((uintptr_t)s->foot_positions_base & 15u) == 0, "rg_control_step foot_positions_base (16-byte alignment)");
  const rg_mpc_env_model* m = nullptr;
  int rc = rg_check_env_model(model, "rg_control_step_env", &m);
  if (rc != RG_OK) return rc;
  const rg_gait_env_params* g = nullptr;
  rc = rg_check_env_gait(gait, "rg_control_step_env", &g);
  if (rc != RG_OK) return rc;
  if ((uintptr_t)plan & 3u) {
    rg_set_error("rg_control_step_plan: contact_schedule_out must be 4-byte aligned");
    return RG_ERR_BAD_ARG;
  }
  if (feet && !plan) {
    rg_set_error("rg_control_step_footholds: a foothold plan needs contact_schedule_out");
    return RG_ERR_BAD_ARG;
  }
  if ((uintptr_t)feet & 15u) {
    rg_set_error("rg_control_step_footholds: foothold_plan_out must be 16-byte aligned");
    return RG_ERR_BAD_ARG;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const RgRobotDev* R = (const RgRobotDev*)robot_ws;
  RgMpcHostInfo info;
  if (plan) {   // the prologue needs the horizon and dt: look the workspace up before the first launch
    rc = rg_mpc_workspace_info(mpc_ws, &info);
    if (rc != RG_OK) return rc;
    const rg_gait_env_params gp = g ? *g : rg_gait_env_params{nullptr, nullptr, nullptr, nullptr};
    if (feet && n_env <= kPrologueLegMaxEnvs)
      step_prologue_feet_kernel<<<grid_for(4 * n_env, 128), 128, 0, st>>>(R, n_env, *s, gp, plan, feet, info.horizon, info.dt);
    else if (feet)
      step_prologue_env_feet_kernel<<<grid_for(n_env, 128), 128, 0, st>>>(R, n_env, *s, gp, plan, feet, info.horizon, info.dt);
    else if (n_env <= kPrologueLegMaxEnvs)
      step_prologue_plan_kernel<<<grid_for(4 * n_env, 128), 128, 0, st>>>(R, n_env, *s, gp, plan, info.horizon, info.dt);
    else
      step_prologue_env_plan_kernel<<<grid_for(n_env, 128), 128, 0, st>>>(R, n_env, *s, gp, plan, info.horizon, info.dt);
  } else if (n_env <= kPrologueLegMaxEnvs) {
    if (g) step_prologue_gait_kernel<<<grid_for(4 * n_env, 128), 128, 0, st>>>(R, n_env, *s, *g);
    else step_prologue_kernel<<<grid_for(4 * n_env, 128), 128, 0, st>>>(R, n_env, *s);
  } else {
    if (g) step_prologue_env_gait_kernel<<<grid_for(n_env, 128), 128, 0, st>>>(R, n_env, *s, *g);
    else step_prologue_env_kernel<<<grid_for(n_env, 128), 128, 0, st>>>(R, n_env, *s);
  }
  rg_count_launch();
  rc = rg_check_cuda(cudaGetLastError(), "step_prologue_kernel launch");
  if (rc != RG_OK) return rc;
  if (!plan) {
    rc = rg_mpc_workspace_info(mpc_ws, &info);
    if (rc != RG_OK) return rc;
  }
  // TorqueStanceLegController.get_action zeroes the yaw before the solve ("yaw aligned world frame")
  rg_mpc_io io;
  memset(&io, 0, sizeof(io));
  io.com_velocity_body = s->com_velocity_body;
  io.base_rpy = s->base_rpy;
  io.base_rpy_rate = s->base_rpy_rate;
  io.foot_contact_state = s->mpc_contact_state;
  io.foot_positions_base = s->foot_positions_base;
  io.command = s->command;
  io.contact_forces = s->contact_forces;
  io.solve_info = s->solve_info;
  io.active_set_io = s->mpc_active_set;
  io.zero_yaw = 1;
  // prologue -> solve kernel(s) -> epilogue are chained by programmatic dependent launches: each grid becomes resident
  // while its predecessor drains and waits (griddepcontrol.wait) for it to complete, so the launch latencies overlap
  rc = rg_launch_mpc((const RgMpcDev*)mpc_ws, info.horizon, n_env, io, info.two_kernel && info.queue_capacity >= n_env, st, 1, m, plan, feet);
  if (rc != RG_OK) return rc;
  rc = rg_check_cuda(rg_launch(step_epilogue_kernel, dim3((unsigned)grid_for(4 * n_env, 256)), dim3(256), 0, st, true,
                               (const RgRobotDev*)robot_ws, n_env, *s), "step_epilogue_kernel launch");
  rg_count_launch();
  return rc;
}

// ---- the control step as ONE graph launch ---------------------------------------------------------------------------
// For small batches the step is launch-bound: prologue, solve (one kernel when the batch fits a wave) and epilogue are
// three dependent launches of a few microseconds each.  Captured once into a CUDA graph they are replayed with a single
// cudaGraphLaunch.  The graph bakes in the pointers of `s`: the caller re-creates it when a buffer moves.
struct RgStepGraph {
  cudaGraph_t graph;
  cudaGraphExec_t exec;
  int kernels;
};

extern "C" int rg_control_step_graph_create(const void* mpc_ws, const void* robot_ws, int n_env, const rg_controller_state* s,
                                            void* stream, void** graph_out) {
  return rg_control_step_graph_create_model(mpc_ws, robot_ws, n_env, s, nullptr, stream, graph_out);
}

extern "C" int rg_control_step_graph_create_model(const void* mpc_ws, const void* robot_ws, int n_env, const rg_controller_state* s,
                                                  const rg_mpc_env_model* model, void* stream, void** graph_out) {
  return rg_control_step_graph_create_env(mpc_ws, robot_ws, n_env, s, model, nullptr, stream, graph_out);
}

extern "C" int rg_control_step_graph_create_env(const void* mpc_ws, const void* robot_ws, int n_env, const rg_controller_state* s,
                                                const rg_mpc_env_model* model, const rg_gait_env_params* gait, void* stream,
                                                void** graph_out) {
  return rg_control_step_graph_create_plan(mpc_ws, robot_ws, n_env, s, model, gait, nullptr, stream, graph_out);
}

extern "C" int rg_control_step_graph_create_plan(const void* mpc_ws, const void* robot_ws, int n_env, const rg_controller_state* s,
                                                 const rg_mpc_env_model* model, const rg_gait_env_params* gait, uint8_t* plan,
                                                 void* stream, void** graph_out) {
  return rg_control_step_graph_create_footholds(mpc_ws, robot_ws, n_env, s, model, gait, plan, nullptr, stream, graph_out);
}

extern "C" int rg_control_step_graph_create_footholds(const void* mpc_ws, const void* robot_ws, int n_env,
                                                      const rg_controller_state* s, const rg_mpc_env_model* model,
                                                      const rg_gait_env_params* gait, uint8_t* plan, float* feet,
                                                      void* stream, void** graph_out) {
  RG_REQUIRE(mpc_ws && robot_ws && s && graph_out && n_env > 0, "rg_control_step_graph_create");
  *graph_out = nullptr;
  // one eager step on the caller's stream first: kernel attributes get configured outside the capture, and argument
  // errors surface here with their own message.  The controller state advances by this step -- the caller accounts for it
  // by creating the graph INSTEAD of a step, not before one (see rg_cuda.h).
  int rc = rg_control_step_footholds(mpc_ws, robot_ws, n_env, s, model, gait, plan, feet, stream);
  if (rc == RG_OK) rc = rg_check_cuda(cudaStreamSynchronize((cudaStream_t)stream), "graph warm-up step");
  if (rc != RG_OK) return rc;
  cudaStream_t cap = nullptr;
  rc = rg_check_cuda(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking), "graph capture stream");
  if (rc != RG_OK) return rc;
  const uint64_t before = rg_launch_count();
  RgStepGraph* g = new RgStepGraph{nullptr, nullptr, 0};
  cudaError_t e = cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal);
  if (e == cudaSuccess) {
    rc = rg_control_step_footholds(mpc_ws, robot_ws, n_env, s, model, gait, plan, feet, cap);
    e = cudaStreamEndCapture(cap, &g->graph);
    if (rc != RG_OK) e = cudaErrorUnknown;
  }
  if (e == cudaSuccess) e = cudaGraphInstantiate(&g->exec, g->graph, 0);
  cudaStreamDestroy(cap);
  if (e != cudaSuccess) {
    if (g->graph) cudaGraphDestroy(g->graph);
    delete g;
    cudaGetLastError();
    if (rc == RG_OK) rc = rg_check_cuda(e, "control-step graph capture");
    return rc;
  }
  g->kernels = (int)(rg_launch_count() - before);
  *graph_out = g;
  return RG_OK;
}

extern "C" int rg_control_step_graph_launch(void* graph, void* stream) {
  RG_REQUIRE(graph, "rg_control_step_graph_launch");
  RgStepGraph* g = (RgStepGraph*)graph;
  const int rc = rg_check_cuda(cudaGraphLaunch(g->exec, (cudaStream_t)stream), "cudaGraphLaunch(control step)");
  for (int i = 0; i < g->kernels; ++i) rg_count_launch();
  return rc;
}

extern "C" int rg_control_step_graph_destroy(void* graph) {
  if (!graph) return RG_OK;
  RgStepGraph* g = (RgStepGraph*)graph;
  if (g->exec) cudaGraphExecDestroy(g->exec);
  if (g->graph) cudaGraphDestroy(g->graph);
  delete g;
  return RG_OK;
}
