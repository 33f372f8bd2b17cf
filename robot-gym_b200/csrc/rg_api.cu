// C-ABI entry points (include/rg_cuda.h): argument validation, one-time table setup, launches.
#include "rg_common.cuh"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <unordered_map>
#include <vector>

namespace {
thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};
std::mutex g_ws_mutex;
std::unordered_map<const void*, RgMpcHostInfo> g_ws_info;   // workspaces prepared by rg_mpc_setup in this process
}  // namespace

// Host-side record of a prepared workspace.  The launch path never touches the device for it (no synchronising
// header read: that would break stream ordering and CUDA-graph capture); a workspace this process did not prepare
// is rejected, and the kernels re-check magic and horizon on the device, so a stale record (memory freed and
// reused without rg_mpc_release) yields RG_STATUS_BAD_WORKSPACE instead of an out-of-bounds access.
int rg_mpc_workspace_info(const void* workspace, RgMpcHostInfo* info) {
  std::lock_guard<std::mutex> lock(g_ws_mutex);
  auto it = g_ws_info.find(workspace);
  if (it == g_ws_info.end()) {
    rg_set_error("workspace was not prepared by rg_mpc_setup (in this process)");
    return RG_ERR_WORKSPACE;
  }
  *info = it->second;
  return RG_OK;
}

void rg_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int rg_check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return RG_OK;
  rg_set_error("%s: %s", what, cudaGetErrorString(e));
  return RG_ERR_CUDA;
}

void rg_count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

extern "C" uint64_t rg_launch_count(void) { return g_launches.load(); }
extern "C" const char* rg_last_error(void) { return g_err; }
extern "C" const char* rg_version(void) { return "rg_cuda 0.1 (sm_100a)"; }

// ------------------------------------------------------------------------------------------------
// Host-side horizon tables: generalised symmetric eigenproblem c2 U = c1 U diag(gamma), U^T c1 U = I
// via Cholesky of c1 + cyclic Jacobi on the reduced matrix (h <= 20, done once per setup).
namespace {

void horizon_tables(int h, std::vector<double>& c1, std::vector<double>& c2) {
  c1.assign(h * h, 0.0);
  c2.assign(h * h, 0.0);
  for (int j = 0; j < h; ++j)
    for (int k = 0; k < h; ++k) {
      const int m = j > k ? j : k;
      c1[j * h + k] = h - m;
      double s = 0.0;
      for (int i = m + 1; i <= h; ++i) s += (i - j - 0.5) * (i - k - 0.5);
      c2[j * h + k] = s;
    }
}

bool generalized_eigen(int h, const std::vector<double>& c1, const std::vector<double>& c2,
                       double* u_out /* [j][t] row-major h*h */, double* gamma_out) {
  // c1 = L L^T
  std::vector<double> l(h * h, 0.0);
  for (int i = 0; i < h; ++i)
    for (int j = 0; j <= i; ++j) {
      double v = c1[i * h + j];
      for (int k = 0; k < j; ++k) v -= l[i * h + k] * l[j * h + k];
      if (i == j) {
        if (!(v > 0.0)) return false;
        l[i * h + i] = sqrt(v);
      } else {
        l[i * h + j] = v / l[j * h + j];
      }
    }
  // S = L^-1 c2 L^-T
  std::vector<double> tmp(h * h), s(h * h);
  for (int c = 0; c < h; ++c)          // solve L X = c2 (column by column)
    for (int i = 0; i < h; ++i) {
      double v = c2[i * h + c];
      for (int k = 0; k < i; ++k) v -= l[i * h + k] * tmp[k * h + c];
      tmp[i * h + c] = v / l[i * h + i];
    }
  for (int r = 0; r < h; ++r)          // solve S L^T = X  <=>  L S^T = X^T
    for (int i = 0; i < h; ++i) {
      double v = tmp[r * h + i];
      for (int k = 0; k < i; ++k) v -= l[i * h + k] * s[r * h + k];
      s[r * h + i] = v / l[i * h + i];
    }
  for (int i = 0; i < h; ++i)
    for (int j = 0; j < i; ++j) { const double m = 0.5 * (s[i * h + j] + s[j * h + i]); s[i * h + j] = s[j * h + i] = m; }
  // cyclic Jacobi: S = Q diag(gamma) Q^T
  std::vector<double> qm(h * h, 0.0);
  for (int i = 0; i < h; ++i) qm[i * h + i] = 1.0;
  for (int sweep = 0; sweep < 100; ++sweep) {
    double off = 0.0, diag = 0.0;
    for (int i = 0; i < h; ++i)
      for (int j = 0; j < h; ++j) (i == j ? diag : off) += s[i * h + j] * s[i * h + j];
    if (off <= 1e-30 * diag) break;
    for (int p = 0; p < h - 1; ++p)
      for (int q = p + 1; q < h; ++q) {
        const double apq = s[p * h + q];
        if (fabs(apq) < 1e-300) continue;
        const double theta = (s[q * h + q] - s[p * h + p]) / (2.0 * apq);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
        for (int k = 0; k < h; ++k) {
          const double skp = s[k * h + p], skq = s[k * h + q];
          s[k * h + p] = c * skp - sn * skq;
          s[k * h + q] = sn * skp + c * skq;
        }
        for (int k = 0; k < h; ++k) {
          const double spk = s[p * h + k], sqk = s[q * h + k];
          s[p * h + k] = c * spk - sn * sqk;
          s[q * h + k] = sn * spk + c * sqk;
        }
        for (int k = 0; k < h; ++k) {
          const double qkp = qm[k * h + p], qkq = qm[k * h + q];
          qm[k * h + p] = c * qkp - sn * qkq;
          qm[k * h + q] = sn * qkp + c * qkq;
        }
      }
  }
  // U = L^-T Q
  for (int t = 0; t < h; ++t) {
    gamma_out[t] = s[t * h + t];
    for (int i = h - 1; i >= 0; --i) {
      double v = qm[i * h + t];
      for (int k = i + 1; k < h; ++k) v -= l[k * h + i] * u_out[k * h + t];
      u_out[i * h + t] = v / l[i * h + i];
    }
  }
  return true;
}

bool inv3(const double* m, double* o) {
  const double c00 = m[4] * m[8] - m[5] * m[7], c01 = m[5] * m[6] - m[3] * m[8], c02 = m[3] * m[7] - m[4] * m[6];
  const double det = m[0] * c00 + m[1] * c01 + m[2] * c02;
  if (fabs(det) < 1e-300) return false;
  const double id = 1.0 / det;
  o[0] = c00 * id; o[1] = (m[2] * m[7] - m[1] * m[8]) * id; o[2] = (m[1] * m[5] - m[2] * m[4]) * id;
  o[3] = c01 * id; o[4] = (m[0] * m[8] - m[2] * m[6]) * id; o[5] = (m[2] * m[3] - m[0] * m[5]) * id;
  o[6] = c02 * id; o[7] = (m[1] * m[6] - m[0] * m[7]) * id; o[8] = (m[0] * m[4] - m[1] * m[3]) * id;
  return true;
}

}  // namespace

extern "C" int rg_mpc_default_params(rg_mpc_params* p, double mass, const double* inertia9,
                                     double desired_body_height, int horizon) {
  if (!p || !inertia9) { rg_set_error("rg_mpc_default_params: NULL argument"); return RG_ERR_BAD_ARG; }
  memset(p, 0, sizeof(*p));
  p->mass = mass;
  memcpy(p->inertia, inertia9, 9 * sizeof(double));
  p->num_legs = 4;
  p->horizon = horizon;
  p->dt = 0.025;
  const double w[13] = {5, 5, 0.2, 0, 0, 10, 0.5, 0.5, 0.2, 0.2, 0.2, 0.1, 0};
  memcpy(p->weights, w, sizeof(w));
  p->alpha = 1e-5;
  for (int i = 0; i < 4; ++i) p->friction_coeffs[i] = 0.45;
  p->gravity = 9.8;
  p->fz_max = mass * 9.8 * 10.0;
  p->fz_min = mass * 9.8 * 0.1;
  p->desired_body_height = desired_body_height;
  p->ipm_tol = 1e-6;
  p->max_ipm_iters = 40;
  p->max_polish_rounds = 3;
  p->cold_start_rounds = 12;
  p->cold_start_max_violations = 0;   // 0 = no limit
  p->two_kernel_solve = 1;
  return RG_OK;
}

extern "C" int rg_workspace_bytes(int n_env, int horizon, int num_legs, size_t* bytes) {
  if (!bytes || n_env < 0) { rg_set_error("rg_workspace_bytes: bad argument"); return RG_ERR_BAD_ARG; }
  if (num_legs != 4) { rg_set_error("num_legs=%d unsupported (4 only)", num_legs); return RG_ERR_UNSUPPORTED; }
  if (horizon != 5 && horizon != 10 && horizon != 20) {
    rg_set_error("unsupported horizon %d (kernels are built for 5, 10, 20)", horizon);
    return RG_ERR_UNSUPPORTED;
  }
  // parameter block + horizon tables, then the fallback queue of the two-kernel solve for n_env envs
  *bytes = RG_MPC_SCRATCH_OFFSET + ((offsetof(RgMpcScratch, queue) + sizeof(int32_t) * (size_t)(n_env > 0 ? n_env : 1) + 255) & ~size_t(255));
  return RG_OK;
}

extern "C" int rg_mpc_setup(const rg_mpc_params* p, void* workspace, size_t workspace_bytes, void* stream) {
  if (!p || !workspace) { rg_set_error("rg_mpc_setup: NULL argument"); return RG_ERR_BAD_ARG; }
  size_t need = 0;
  int rc = rg_workspace_bytes(0, p->horizon, p->num_legs, &need);
  if (rc != RG_OK) return rc;
  if (workspace_bytes < need) { rg_set_error("workspace too small: %zu < %zu", workspace_bytes, need); return RG_ERR_WORKSPACE; }
  if (!(p->mass > 0) || !(p->dt > 0) || !(p->alpha > 0) || !(p->fz_max > p->fz_min) || !(p->fz_min >= 0)) {
    rg_set_error("rg_mpc_setup: need mass>0, dt>0, alpha>0, 0<=fz_min<fz_max");
    return RG_ERR_BAD_ARG;
  }
  for (int i = 0; i < 4; ++i)
    if (!(p->friction_coeffs[i] > 0)) { rg_set_error("friction coefficient %d must be > 0", i); return RG_ERR_BAD_ARG; }
  for (int i = 0; i < 13; ++i)
    if (!(p->weights[i] >= 0)) { rg_set_error("weight %d must be >= 0", i); return RG_ERR_BAD_ARG; }
  // K = c1 (x) K1 + c2 (x) K2 must be positive definite: every acceleration channel needs a
  // velocity weight or (for the angular channels: all three) a position weight.
  const bool ang_pos = p->weights[0] > 0 && p->weights[1] > 0 && p->weights[2] > 0;
  for (int c = 0; c < 3; ++c) {
    if (!(p->weights[6 + c] > 0) && !ang_pos) {
      rg_set_error("weights leave angular channel %d unpenalised (need w[%d]>0 or w[0..2]>0)", c, 6 + c);
      return RG_ERR_SINGULAR;
    }
    if (!(p->weights[9 + c] > 0) && !(p->weights[3 + c] > 0)) {
      rg_set_error("weights leave linear channel %d unpenalised (need w[%d]>0 or w[%d]>0)", c, 9 + c, 3 + c);
      return RG_ERR_SINGULAR;
    }
  }
  RgMpcDev h;
  memset(&h, 0, sizeof(h));
  h.magic = RG_WS_MAGIC_MPC;
  h.horizon = p->horizon;
  h.max_ipm_iters = p->max_ipm_iters > 0 ? p->max_ipm_iters : 40;
  h.max_polish_rounds = p->max_polish_rounds;
  // the cold start is the polish without an interior-point guess: it needs the polish enabled
  h.cold_start_rounds = (p->max_polish_rounds > 0 && p->cold_start_rounds > 0) ? p->cold_start_rounds : 0;
  h.cold_start_max_violations = p->cold_start_max_violations > 0 ? p->cold_start_max_violations : (1 << 30);
  h.inv_mass = 1.0 / p->mass;
  h.mass = p->mass;
  if (!inv3(p->inertia, h.inv_inertia)) { rg_set_error("inertia matrix is singular"); return RG_ERR_SINGULAR; }
  h.dt = p->dt;
  for (int i = 0; i < 6; ++i) { h.w_rho[i] = p->weights[i]; h.w_nu[i] = p->weights[6 + i]; }
  h.alpha = p->alpha;
  for (int i = 0; i < 4; ++i) h.mu[i] = p->friction_coeffs[i];
  h.gravity = p->gravity;
  h.fz_max = p->fz_max;
  h.fz_min = p->fz_min;
  h.height = p->desired_body_height;
  h.ipm_tol = p->ipm_tol > 0 ? p->ipm_tol : 1e-6;
  std::vector<double> c1, c2;
  horizon_tables(p->horizon, c1, c2);
  if (!generalized_eigen(p->horizon, c1, c2, h.eig_u, h.eig_gamma)) {
    rg_set_error("horizon table factorisation failed");
    return RG_ERR_SINGULAR;
  }
  for (int jj = 0; jj < p->horizon; ++jj)
    for (int kk = 0; kk <= jj; ++kk)
      for (int t = 0; t < p->horizon; ++t)
        h.eig_uu[(jj * (jj + 1) / 2 + kk) * p->horizon + t] = h.eig_u[jj * p->horizon + t] * h.eig_u[kk * p->horizon + t];

  {
    // env-independent tables: c2 and the inverse of the three linear channels of K,
    // K_lin,c = 2 dt^2 w_v,c c1 + 2 dt^4 w_p,c c2  =>  K_lin,c^-1 = U diag(1 / (k1 + gamma_t k2)) U^T
    const int hz = p->horizon;
    const double dt2 = p->dt * p->dt, dt4 = dt2 * dt2;
    for (int i = 0; i < hz * hz; ++i) h.c2tab[i] = c2[i];
    for (int c = 0; c < 3; ++c) {
      const double k1 = 2.0 * dt2 * p->weights[9 + c], k2 = 2.0 * dt4 * p->weights[3 + c];
      for (int j = 0; j < hz; ++j)
        for (int k = 0; k <= j; ++k) {
          double v = 0.0;
          for (int t = 0; t < hz; ++t) v += h.eig_u[j * hz + t] * h.eig_u[k * hz + t] / (k1 + h.eig_gamma[t] * k2);
          h.kinv_lin[c][j * (j + 1) / 2 + k] = v;
        }
    }
  }
  if (((uintptr_t)workspace & 255u) != 0) { rg_set_error("workspace must be 256-byte aligned"); return RG_ERR_BAD_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  rc = rg_check_cuda(cudaMemcpyAsync(workspace, &h, sizeof(h), cudaMemcpyHostToDevice, st), "rg_mpc_setup upload");
  if (rc != RG_OK) return rc;
  // fallback queue: whatever follows the parameter block holds the list (capacity = envs it was sized for)
  RgMpcScratch sc;
  memset(&sc, 0, sizeof(sc));
  const size_t avail = workspace_bytes - RG_MPC_SCRATCH_OFFSET;
  const size_t cap = avail > offsetof(RgMpcScratch, queue) ? (avail - offsetof(RgMpcScratch, queue)) / sizeof(int32_t) : 0;
  sc.capacity = (int32_t)(cap > 0x7fffffff ? 0x7fffffff : cap);
  rc = rg_check_cuda(cudaMemcpyAsync((char*)workspace + RG_MPC_SCRATCH_OFFSET, &sc, offsetof(RgMpcScratch, queue), cudaMemcpyHostToDevice, st),
                     "rg_mpc_setup scratch upload");
  if (rc != RG_OK) return rc;
  rc = rg_check_cuda(cudaStreamSynchronize(st), "rg_mpc_setup sync");
  if (rc != RG_OK) return rc;
  RgMpcHostInfo info;
  info.horizon = p->horizon;
  info.queue_capacity = sc.capacity;
  info.two_kernel = (p->two_kernel_solve != 0 && h.cold_start_rounds > 0) ? 1 : 0;
  info.dt = p->dt;
  std::lock_guard<std::mutex> lock(g_ws_mutex);
  g_ws_info[workspace] = info;
  return RG_OK;
}

extern "C" int rg_mpc_release(const void* workspace) {
  std::lock_guard<std::mutex> lock(g_ws_mutex);
  g_ws_info.erase(workspace);
  return RG_OK;
}

int rg_check_env_model(const rg_mpc_env_model* model, const char* what, const rg_mpc_env_model** out) {
  *out = nullptr;
  if (!model || (!model->mass && !model->inertia && !model->friction_coeffs)) return RG_OK;
  if (((uintptr_t)model->mass | (uintptr_t)model->inertia | (uintptr_t)model->friction_coeffs) & 7u) {
    rg_set_error("%s: env model arrays must be 8-byte aligned float64", what);
    return RG_ERR_BAD_ARG;
  }
  *out = model;
  return RG_OK;
}

extern "C" int rg_mpc_build_solve_io(const void* workspace, int n_env, const rg_mpc_io* io, void* stream) {
  return rg_mpc_build_solve_model(workspace, n_env, io, nullptr, stream);
}

extern "C" int rg_mpc_build_solve_model(const void* workspace, int n_env, const rg_mpc_io* io,
                                        const rg_mpc_env_model* model, void* stream) {
  return rg_mpc_build_solve_schedule(workspace, n_env, io, model, nullptr, stream);
}

extern "C" int rg_mpc_build_solve_schedule(const void* workspace, int n_env, const rg_mpc_io* io,
                                           const rg_mpc_env_model* model, const uint8_t* contact_schedule, void* stream) {
  return rg_mpc_build_solve_footholds(workspace, n_env, io, model, contact_schedule, nullptr, stream);
}

extern "C" int rg_mpc_build_solve_footholds(const void* workspace, int n_env, const rg_mpc_io* io,
                                            const rg_mpc_env_model* model, const uint8_t* contact_schedule,
                                            const float* foothold_plan, void* stream) {
  if (n_env == 0) return RG_OK;   // empty batch: nothing to validate, nothing to launch
  if (foothold_plan && !contact_schedule) {
    rg_set_error("rg_mpc_build_solve_footholds: a foothold plan needs a contact schedule");
    return RG_ERR_BAD_ARG;
  }
  // with a schedule the contact row is not read (it may be NULL), with a foothold plan the current feet are not
  if (!workspace || !io || !io->com_velocity_body || !io->base_rpy || !io->base_rpy_rate ||
      (!io->foot_contact_state && !contact_schedule) || (!io->foot_positions_base && !foothold_plan) || !io->command ||
      !io->contact_forces) {
    rg_set_error("rg_mpc_build_solve: NULL argument");
    return RG_ERR_BAD_ARG;
  }
  if (n_env < 0) { rg_set_error("rg_mpc_build_solve: n_env < 0"); return RG_ERR_BAD_ARG; }
  if (!contact_schedule && ((uintptr_t)io->foot_contact_state & 3u) != 0) {   // the kernel reads the four contact flags of an env as one 32-bit word
    rg_set_error("rg_mpc_build_solve: foot_contact_state must be 4-byte aligned");
    return RG_ERR_BAD_ARG;
  }
  if (((uintptr_t)contact_schedule & 3u) != 0) {   // ... and each row of a schedule likewise
    rg_set_error("rg_mpc_build_solve_schedule: contact_schedule must be 4-byte aligned");
    return RG_ERR_BAD_ARG;
  }
  if (!foothold_plan && ((uintptr_t)io->foot_positions_base & 15u) != 0) {  // ... and the twelve foot coordinates with three 128-bit loads
    rg_set_error("rg_mpc_build_solve: foot_positions_base must be 16-byte aligned");
    return RG_ERR_BAD_ARG;
  }
  if (((uintptr_t)foothold_plan & 15u) != 0) {   // ... and each row of a foothold plan likewise
    rg_set_error("rg_mpc_build_solve_footholds: foothold_plan must be 16-byte aligned");
    return RG_ERR_BAD_ARG;
  }
  const rg_mpc_env_model* m = nullptr;
  int rc = rg_check_env_model(model, "rg_mpc_build_solve_model", &m);
  if (rc != RG_OK) return rc;
  RgMpcHostInfo info;
  rc = rg_mpc_workspace_info(workspace, &info);
  if (rc != RG_OK) return rc;
  return rg_launch_mpc((const RgMpcDev*)workspace, info.horizon, n_env, *io, info.two_kernel && info.queue_capacity >= n_env,
                       (cudaStream_t)stream, 0, m, contact_schedule, foothold_plan);
}

extern "C" int rg_mpc_build_solve(const void* workspace, int n_env, const float* com_velocity_body,
                                  const float* base_rpy, const float* base_rpy_rate,
                                  const uint8_t* foot_contact_state, const float* foot_positions_base,
                                  const float* command, const float* com_height, float* contact_forces,
                                  float* horizon_forces, int32_t* solve_info, void* stream) {
  return rg_mpc_build_solve_warm(workspace, n_env, com_velocity_body, base_rpy, base_rpy_rate, foot_contact_state,
                                 foot_positions_base, command, com_height, contact_forces, horizon_forces, solve_info,
                                 nullptr, stream);
}

extern "C" int rg_mpc_build_solve_warm(const void* workspace, int n_env, const float* com_velocity_body,
                                       const float* base_rpy, const float* base_rpy_rate,
                                       const uint8_t* foot_contact_state, const float* foot_positions_base,
                                       const float* command, const float* com_height, float* contact_forces,
                                       float* horizon_forces, int32_t* solve_info, uint16_t* active_set_io, void* stream) {
  rg_mpc_io io;
  memset(&io, 0, sizeof(io));
  io.com_velocity_body = com_velocity_body;
  io.base_rpy = base_rpy;
  io.base_rpy_rate = base_rpy_rate;
  io.foot_contact_state = foot_contact_state;
  io.foot_positions_base = foot_positions_base;
  io.command = command;
  io.com_height = com_height;
  io.contact_forces = contact_forces;
  io.horizon_forces = horizon_forces;
  io.solve_info = solve_info;
  io.active_set_io = active_set_io;
  return rg_mpc_build_solve_io(workspace, n_env, &io, stream);
}

// ------------------------------------------------------------------------------------------------
// Diagnostic: measured CUDA-core FMA peak (the roofline denominator this path is actually bound by;
// MEASURED_PEAKS.json only has HBM and bf16 tensor numbers).  8 independent FMA chains per thread.
namespace {
template <typename T>
__global__ void fma_peak_kernel(T* out, int iters, T a, T b) {
  T x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
    x0 = x0 * a + b; x1 = x1 * a + b; x2 = x2 * a + b; x3 = x3 * a + b;
    x4 = x4 * a + b; x5 = x5 * a + b; x6 = x6 * a + b; x7 = x7 * a + b;
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

template <typename T>
int measure_fma(int iters, double* tflops) {
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int blocks = sms * 8, threads = 256;
  T* buf = nullptr;
  int rc = rg_check_cuda(cudaMalloc(&buf, sizeof(T) * blocks * threads), "fma peak cudaMalloc");
  if (rc != RG_OK) return rc;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    fma_peak_kernel<T><<<blocks, threads>>>(buf, iters, (T)0.999, (T)0.001);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
    if (rep > 0 && ms > 0.f) best = fmax(best, flops / (ms * 1e-3) * 1e-12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(buf);
  *tflops = best;
  return rg_check_cuda(cudaGetLastError(), "fma peak kernel");
}
}  // namespace

extern "C" int rg_measure_fma_peak(int use_fp64, int iters, double* tflops_host) {
  if (!tflops_host || iters <= 0) { rg_set_error("rg_measure_fma_peak: bad argument"); return RG_ERR_BAD_ARG; }
  return use_fp64 ? measure_fma<double>(iters, tflops_host) : measure_fma<float>(iters, tflops_host);
}
