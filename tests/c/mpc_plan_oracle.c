/*
 * mpc_plan_oracle.c -- the C oracle's stance QP over a contact schedule.  TEST INFRASTRUCTURE ONLY.
 *
 * rgo_compute_contact_forces_schedule is oracle/c/mpc_oracle.c's rgo_compute_contact_forces with a [h, k] contact
 * schedule in place of the one contact row the reference's wrapper tiles over the horizon: the swing variables are
 * eliminated per (step, leg) from the schedule, and the com height is taken over the stance feet of row 0, or of the
 * first row with a stance foot (include/rg_cuda.h, rg_mpc_build_solve_schedule).  The oracle source is included
 * unchanged for its helpers and its own entry points; the body below is its function with those three edits.
 */
#include "../../oracle/c/mpc_oracle.c"

/* Solves one QP over a schedule; out = -(solution) (3*k*h doubles).  Returns the interior-point iteration count. */
int rgo_compute_contact_forces_schedule(const rgo_params* p, const double* com_vel, const double* rpy, const double* ang_vel,
                                        const int* schedule /* [h * k] */, const double* feet_base, const double* des_pos,
                               const double* des_vel, const double* des_rpy, const double* des_w,
                               const double* com_pos /* 3 or NULL */, double* out, double* scratch) {
  const int h = p->horizon, k = p->num_legs, m3 = 3 * k, n_all = m3 * h, ns = S13 * h;
  const double dt = p->dt, g = p->gravity;
  memset(out, 0, sizeof(double) * n_all);
  /* the com height is taken over the stance feet of row 0, or of the first row with one; no stance at all: zero forces */
  const int* contacts = schedule;
  for (int t = 0; t < h; ++t) {
    int any = 0;
    for (int i = 0; i < k; ++i) any |= schedule[t * k + i] != 0;
    if (any) { contacts = schedule + t * k; break; }
  }
  int n_stance = 0;
  for (int i = 0; i < k; ++i) n_stance += contacts[i] != 0;
  if (n_stance == 0) return 0;

  /* foot positions in the world frame: R = Rx Ry Rz (sic) */
  double rx[9], ry[9], rz[9], t33[9], rfeet[9], rbody[9];
  rot_x(rpy[0], rx); rot_y(rpy[1], ry); rot_z(rpy[2], rz);
  matmul(rx, ry, t33, 3, 3, 3); matmul(t33, rz, rfeet, 3, 3, 3);
  matmul(rz, ry, t33, 3, 3, 3); matmul(t33, rx, rbody, 3, 3, 3);
  double feet_w[MAXK][3];
  double zsum = 0.0;
  for (int i = 0; i < k; ++i) {
    for (int r = 0; r < 3; ++r)
      feet_w[i][r] = rfeet[3 * r] * feet_base[3 * i] + rfeet[3 * r + 1] * feet_base[3 * i + 1] + rfeet[3 * r + 2] * feet_base[3 * i + 2];
    if (contacts[i]) zsum += feet_w[i][2];
  }
  const double com_z = com_pos ? com_pos[2] : fabs(zsum / n_stance);

  double x0[S13] = {rpy[0], rpy[1], rpy[2], 0.0, 0.0, com_z, ang_vel[0], ang_vel[1], ang_vel[2],
                    com_vel[0], com_vel[1], com_vel[2], -g};

  /* continuous A, B and the exponential of [[A,B],[0,0]] dt */
  const int nab = S13 + m3;
  double ab[(S13 + 3 * MAXK) * (S13 + 3 * MAXK)], abexp[(S13 + 3 * MAXK) * (S13 + 3 * MAXK)];
  memset(ab, 0, sizeof(ab));
  {
    const double cy = cos(rpy[2]), sy = sin(rpy[2]), cp = cos(rpy[1]), tp = tan(rpy[1]);
    const double tm[9] = {cy / cp, sy / cp, 0, -sy, cy, 0, cy * tp, sy * tp, 1};
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) ab[r * nab + 6 + c] = tm[3 * r + c] * dt;
    ab[3 * nab + 9] = ab[4 * nab + 10] = ab[5 * nab + 11] = dt;
    ab[11 * nab + 12] = dt;
    double inv_i[9] = {0}, iw[9];
    inv3(p->inertia, inv_i);
    matmul(rbody, inv_i, t33, 3, 3, 3);
    for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) {
      double v = 0.0; for (int c = 0; c < 3; ++c) v += t33[3 * a + c] * rbody[3 * b + c];
      iw[3 * a + b] = v;
    }
    for (int i = 0; i < k; ++i) {
      const double* r = feet_w[i];
      const double sk[9] = {0, -r[2], r[1], r[2], 0, -r[0], -r[1], r[0], 0};
      double blk[9];
      matmul(iw, sk, blk, 3, 3, 3);
      for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) ab[(6 + a) * nab + S13 + 3 * i + b] = blk[3 * a + b] * dt;
      for (int a = 0; a < 3; ++a) ab[(9 + a) * nab + S13 + 3 * i + a] = dt / p->mass;
    }
  }
  expm_pade(ab, abexp, nab);
  double a_exp[S13 * S13], b_exp[S13 * 3 * MAXK];
  for (int r = 0; r < S13; ++r) {
    for (int c = 0; c < S13; ++c) a_exp[r * S13 + c] = abexp[r * nab + c];
    for (int c = 0; c < m3; ++c) b_exp[r * m3 + c] = abexp[r * nab + S13 + c];
  }

  /* carve the scratch buffer */
  double* w = scratch;
  double* b_qp = w; w += (size_t)ns * n_all;
  double* p_full = w; w += (size_t)n_all * n_all;
  double* q_full = w; w += n_all;
  /* A_qp x0 (free response) and A^i B blocks */
  double anb[MAXH][S13 * 3 * MAXK];
  double free_resp[MAXH * S13];
  {
    double apow[S13 * S13], nxt[S13 * S13], xs[S13], xn[S13];
    memcpy(anb[0], b_exp, sizeof(double) * S13 * m3);
    memcpy(apow, a_exp, sizeof(apow));
    memcpy(xs, x0, sizeof(xs));
    for (int i = 0; i < h; ++i) {
      matmul(a_exp, xs, xn, S13, S13, 1);
      memcpy(xs, xn, sizeof(xs));
      memcpy(free_resp + i * S13, xs, sizeof(xs));
      if (i + 1 < h) { matmul(a_exp, anb[i], anb[i + 1], S13, S13, m3); }
    }
    (void)apow; (void)nxt;
  }
  memset(b_qp, 0, sizeof(double) * (size_t)ns * n_all);
  for (int i = 0; i < h; ++i)
    for (int j = 0; j <= i; ++j)
      for (int r = 0; r < S13; ++r)
        memcpy(b_qp + (size_t)(i * S13 + r) * n_all + j * m3, anb[i - j] + r * m3, sizeof(double) * m3);
  /* state error and q = 2 B^T L (A x0 - x_ref);  P = 2 (B^T L B + alpha I) */
  double sd[MAXH * S13];
  for (int i = 0; i < h; ++i) {
    double ref[S13] = {des_rpy[0], des_rpy[1], rpy[2] + dt * (i + 1) * des_w[2], dt * (i + 1) * des_vel[0],
                       dt * (i + 1) * des_vel[1], des_pos[2], 0.0, 0.0, des_w[2], des_vel[0], des_vel[1], 0.0, -g};
    for (int r = 0; r < S13; ++r) sd[i * S13 + r] = p->weights[r] * (free_resp[i * S13 + r] - ref[r]);
  }
  for (int c = 0; c < n_all; ++c) {
    double v = 0.0;
    for (int r = 0; r < ns; ++r) v += b_qp[(size_t)r * n_all + c] * sd[r];
    q_full[c] = 2.0 * v;
  }
  for (int a = 0; a < n_all; ++a)
    for (int b = 0; b <= a; ++b) {
      double v = 0.0;
      const int first = (a / m3) * S13;       /* B_qp is block lower triangular */
      for (int r = first; r < ns; ++r) v += p->weights[r % S13] * b_qp[(size_t)r * n_all + a] * b_qp[(size_t)r * n_all + b];
      v = 2.0 * (v + (a == b ? p->alpha : 0.0));
      p_full[(size_t)a * n_all + b] = p_full[(size_t)b * n_all + a] = v;
    }

  /* eliminate swing feet */
  int idx[3 * MAXK * MAXH];
  int n = 0;
  for (int t = 0; t < h; ++t)
    for (int l = 0; l < k; ++l)
      if (schedule[t * k + l]) for (int d = 0; d < 3; ++d) idx[n++] = (t * k + l) * 3 + d;
  const int nblk = n / 3, m = 10 * nblk;
  double* pm = w; w += (size_t)n * n;
  double* phi = w; w += (size_t)n * n;
  double* qv = w; w += n;
  double* x = w; w += n; double* xbest = w; w += n;
  double* rd = w; w += n; double* rhs = w; w += n; double* dxa = w; w += n; double* dx = w; w += n; double* pux = w; w += n;
  double* s = w; w += m; double* lam = w; w += m; double* dsa = w; w += m; double* dla = w; w += m;
  double* ds = w; w += m; double* dl = w; w += m; double* wv = w; w += m;
  for (int a = 0; a < n; ++a) {
    qv[a] = q_full[idx[a]];
    for (int b = 0; b < n; ++b) pm[(size_t)a * n + b] = p_full[(size_t)idx[a] * n_all + idx[b]];
  }
  const double* mu = p->mu;
  const double grow[5][3] = {{-1, 0, mu[0]}, {1, 0, mu[1]}, {0, -1, mu[2]}, {0, 1, mu[3]}, {0, 0, 1}};
  const double big_u = (mu[0] + 1.0) * p->fz_max;
  const double hup[5] = {big_u, big_u, big_u, big_u, p->fz_max};
  const double lo[5] = {0, 0, 0, 0, p->fz_min};

  double qscale = 1.0;
  for (int a = 0; a < n; ++a) if (fabs(qv[a]) > qscale) qscale = fabs(qv[a]);
  const double fz0 = sqrt(fmax(p->fz_min, 1e-3 * p->fz_max) * p->fz_max);
  for (int b = 0; b < nblk; ++b) {
    x[3 * b] = x[3 * b + 1] = 0.0; x[3 * b + 2] = fz0;
    for (int r = 0; r < 5; ++r) {
      const double c = grow[r][0] * x[3 * b] + grow[r][1] * x[3 * b + 1] + grow[r][2] * x[3 * b + 2];
      s[10 * b + r] = hup[r] - c;
      s[10 * b + 5 + r] = c - lo[r];
    }
    for (int r = 0; r < 10; ++r) lam[10 * b + r] = 0.1 * qscale / s[10 * b + r];
  }
  memcpy(xbest, x, sizeof(double) * n);
  double best = 1e300, prev = 1e300;
  int stall = 0, it = 0;
  const double tol = 1e-12;
  for (;;) {
    matmul(pm, x, pux, n, n, 1);
    double rdmax = 0.0, sl = 0.0;
    for (int b = 0; b < nblk; ++b) {
      double e[5];
      for (int r = 0; r < 5; ++r) e[r] = lam[10 * b + r] - lam[10 * b + 5 + r];
      const double gl[3] = {e[1] - e[0], e[3] - e[2], mu[0] * e[0] + mu[1] * e[1] + mu[2] * e[2] + mu[3] * e[3] + e[4]};
      for (int d = 0; d < 3; ++d) { rd[3 * b + d] = pux[3 * b + d] + qv[3 * b + d] + gl[d]; if (fabs(rd[3 * b + d]) > rdmax) rdmax = fabs(rd[3 * b + d]); }
      for (int r = 0; r < 10; ++r) sl += s[10 * b + r] * lam[10 * b + r];
    }
    const double mu_c = sl / m;
    const double res = fmax(rdmax, mu_c) / qscale;
    if (res < best) { best = res; memcpy(xbest, x, sizeof(double) * n); }
    if (res < tol) break;
    stall = (res > 0.9 * prev && res < 1e-7) ? stall + 1 : 0;
    prev = res;
    if (it >= 60 || stall >= 4) break;
    ++it;
    /* Phi = P + G^T D G */
    memcpy(phi, pm, sizeof(double) * (size_t)n * n);
    for (int b = 0; b < nblk; ++b) {
      double dd[5];
      for (int r = 0; r < 5; ++r) dd[r] = lam[10 * b + r] / s[10 * b + r] + lam[10 * b + 5 + r] / s[10 * b + 5 + r];
      for (int a = 0; a < 3; ++a) for (int c = 0; c < 3; ++c) {
        double v = 0.0; for (int r = 0; r < 5; ++r) v += dd[r] * grow[r][a] * grow[r][c];
        phi[(size_t)(3 * b + a) * n + 3 * b + c] += v;
      }
    }
    if (cholesky(phi, n) != 0) break;
    for (int a = 0; a < n; ++a) dxa[a] = -(pux[a] + qv[a]);
    chol_solve(phi, dxa, n);
    double amax = 1.0;
    for (int b = 0; b < nblk; ++b) {
      double c5[5];
      for (int r = 0; r < 5; ++r) c5[r] = grow[r][0] * dxa[3 * b] + grow[r][1] * dxa[3 * b + 1] + grow[r][2] * dxa[3 * b + 2];
      for (int r = 0; r < 10; ++r) {
        const int j = 10 * b + r;
        dsa[j] = r < 5 ? -c5[r] : c5[r - 5];
        dla[j] = -lam[j] - lam[j] * dsa[j] / s[j];
        if (dsa[j] < 0 && -s[j] / dsa[j] < amax) amax = -s[j] / dsa[j];
        if (dla[j] < 0 && -lam[j] / dla[j] < amax) amax = -lam[j] / dla[j];
      }
    }
    double mu_aff = 0.0;
    for (int j = 0; j < m; ++j) mu_aff += (s[j] + amax * dsa[j]) * (lam[j] + amax * dla[j]);
    mu_aff /= m;
    const double sig = pow(mu_aff / mu_c, 3.0), sigmu = sig * mu_c;
    for (int j = 0; j < m; ++j) wv[j] = (s[j] * lam[j] + dsa[j] * dla[j] - sigmu) / s[j];
    for (int b = 0; b < nblk; ++b) {
      double e[5];
      for (int r = 0; r < 5; ++r) e[r] = wv[10 * b + r] - wv[10 * b + 5 + r];
      const double gw[3] = {e[1] - e[0], e[3] - e[2], mu[0] * e[0] + mu[1] * e[1] + mu[2] * e[2] + mu[3] * e[3] + e[4]};
      for (int d = 0; d < 3; ++d) dx[3 * b + d] = -rd[3 * b + d] + gw[d];
    }
    chol_solve(phi, dx, n);
    double step = 1e30;
    for (int b = 0; b < nblk; ++b) {
      double c5[5];
      for (int r = 0; r < 5; ++r) c5[r] = grow[r][0] * dx[3 * b] + grow[r][1] * dx[3 * b + 1] + grow[r][2] * dx[3 * b + 2];
      for (int r = 0; r < 10; ++r) {
        const int j = 10 * b + r;
        ds[j] = r < 5 ? -c5[r] : c5[r - 5];
        dl[j] = (-(s[j] * lam[j] + dsa[j] * dla[j] - sigmu) - lam[j] * ds[j]) / s[j];
        if (ds[j] < 0 && -s[j] / ds[j] < step) step = -s[j] / ds[j];
        if (dl[j] < 0 && -lam[j] / dl[j] < step) step = -lam[j] / dl[j];
      }
    }
    step = fmin(1.0, 0.99 * step);
    for (int a = 0; a < n; ++a) x[a] += step * dx[a];
    for (int j = 0; j < m; ++j) { s[j] += step * ds[j]; lam[j] += step * dl[j]; }
  }
  /* Active-set polish (the counterpart of OSQP's polish and of oracle/convex_mpc.py's refinement): solve the
   * equality-constrained QP on the rows the interior point marks active exactly,
   *     x = x_unc - Y y,   Y = P^-1 C_a^T,   (C_a Y) y = C_a x_unc - b_a,
   * add violated rows, drop rows whose multiplier has the wrong sign, repeat.  Accepted only when a round
   * changes nothing (a KKT point of a strictly convex QP = the optimum); otherwise the interior-point
   * iterate stands.  phi / dxa / dx / rhs / wv are free here and reused as scratch. */
  {
    int* side = (int*)malloc(sizeof(int) * (size_t)(5 * nblk));          /* +1 upper, -1 lower, 0 free */
    int* rows = (int*)malloc(sizeof(int) * (size_t)(5 * nblk));
    double* lfac = phi;                                                    /* Cholesky factor of P */
    double* xunc = dxa;
    double* xp = dx;
    memcpy(lfac, pm, sizeof(double) * (size_t)n * n);
    int ok = cholesky(lfac, n) == 0;
    if (ok) {
      for (int a = 0; a < n; ++a) xunc[a] = -qv[a];
      chol_solve(lfac, xunc, n);
      for (int b = 0; b < nblk; ++b)
        for (int r = 0; r < 5; ++r) {
          const double c = grow[r][0] * xbest[3 * b] + grow[r][1] * xbest[3 * b + 1] + grow[r][2] * xbest[3 * b + 2];
          const double span_hi = fmax(1.0, fabs(hup[r])), span_lo = fmax(1.0, fabs(lo[r]));
          side[5 * b + r] = 0;
          if (lam[10 * b + r] > s[10 * b + r] && hup[r] - c < 1e-5 * span_hi) side[5 * b + r] = 1;
          if (lam[10 * b + 5 + r] > s[10 * b + 5 + r] && c - lo[r] < 1e-5 * fmax(span_hi, span_lo)) side[5 * b + r] = -1;
        }
    }
    const double feas_tol = 1e-11 * fmax(1.0, big_u);
    for (int round = 0; ok && round < 20; ++round) {
      int ma = 0;
      for (int j = 0; j < 5 * nblk; ++j) if (side[j]) rows[ma++] = j;
      double* ymat = (double*)malloc(sizeof(double) * (size_t)(ma > 0 ? ma : 1) * n);      /* rows of Y^T */
      double* smat = (double*)malloc(sizeof(double) * (size_t)(ma > 0 ? ma : 1) * (ma > 0 ? ma : 1));
      double* yv = (double*)malloc(sizeof(double) * (size_t)(ma > 0 ? ma : 1));
      for (int i = 0; i < ma; ++i) {
        const int b = rows[i] / 5, r = rows[i] % 5;
        double* col = ymat + (size_t)i * n;
        memset(col, 0, sizeof(double) * n);
        for (int d = 0; d < 3; ++d) col[3 * b + d] = grow[r][d];
        chol_solve(lfac, col, n);
      }
      for (int i = 0; i < ma; ++i) {
        const int b = rows[i] / 5, r = rows[i] % 5;
        for (int j = 0; j < ma; ++j) {
          const double* col = ymat + (size_t)j * n;
          smat[(size_t)i * ma + j] = grow[r][0] * col[3 * b] + grow[r][1] * col[3 * b + 1] + grow[r][2] * col[3 * b + 2];
        }
        const double target = side[rows[i]] > 0 ? hup[r] : lo[r];
        yv[i] = grow[r][0] * xunc[3 * b] + grow[r][1] * xunc[3 * b + 1] + grow[r][2] * xunc[3 * b + 2] - target;
      }
      if (ma > 0) {
        if (cholesky(smat, ma) != 0) { ok = 0; free(ymat); free(smat); free(yv); break; }   /* dependent rows: keep the IPM point */
        chol_solve(smat, yv, ma);
      }
      memcpy(xp, xunc, sizeof(double) * n);
      for (int i = 0; i < ma; ++i) {
        const double* col = ymat + (size_t)i * n;
        for (int a = 0; a < n; ++a) xp[a] -= yv[i] * col[a];
      }
      int changed = 0;
      double ymax = 1.0;
      for (int i = 0; i < ma; ++i) if (fabs(yv[i]) > ymax) ymax = fabs(yv[i]);
      for (int b = 0; b < nblk; ++b)
        for (int r = 0; r < 5; ++r) {
          if (side[5 * b + r]) continue;
          const double c = grow[r][0] * xp[3 * b] + grow[r][1] * xp[3 * b + 1] + grow[r][2] * xp[3 * b + 2];
          if (c - hup[r] > feas_tol) { side[5 * b + r] = 1; changed = 1; }
          else if (lo[r] - c > feas_tol) { side[5 * b + r] = -1; changed = 1; }
        }
      for (int i = 0; i < ma; ++i)
        if (side[rows[i]] * yv[i] < -1e-12 * ymax) { side[rows[i]] = 0; changed = 1; }
      free(ymat); free(smat); free(yv);
      if (!changed) { memcpy(xbest, xp, sizeof(double) * n); break; }
      if (round == 19) ok = 0;
    }
    free(side); free(rows);
  }
  for (int a = 0; a < n; ++a) out[idx[a]] = -xbest[a];
  (void)rhs;
  return it;
}
