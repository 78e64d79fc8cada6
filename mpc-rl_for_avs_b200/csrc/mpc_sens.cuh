// mpc_sens.cuh -- per-problem FP64 sensitivity of the first control to the problem-level parameters the RL policy sets.
//
// For controls U at a local optimum of the objective the solver minimises (the problem of mpc_kkt.cuh: the same
// Problem / Config / load_problem, path table and objective variants), the implicit-function theorem applied to the
// KKT system with the active set held fixed gives
//     [ H  A^T ] [ dU  ]   [ -G ]        H = Hessian of the Lagrangian J - sum_q nu_q c_q over U
//     [ A   0  ] [ -dnu] = [  0 ]        A = active constraint rows, G = d(grad_U J) / dp
// with p = (vr_b, w_speed, w_control, w_diff).  Returned: J_sens = dU_0 / dp (2 x 4).
//
// Method: an O(N) sweep per problem, FP64, state in registers / local memory.
//   * active set of mpc_kkt: control bounds and theta / v bounds of nodes 1..N within act_tol.  A pinned control removes
//     its coordinate; the node rows are functionals on (theta, v), which do not depend on (x, y).
//   * multipliers: the least-squares fit min |g_free - A_free^T nu| (g = grad_U J) is a chain in the 2-vector psi_k of
//     the node multipliers propagated to (theta_k, v_k); one forward dynamic-programming pass and one backward pass give
//     the node multipliers, the stationarity residual over the free coordinates and the control-bound multipliers.
//   * LICQ: stage k resolves the rows its u_k can satisfy (Householder reflections with column pivoting on the rows'
//     u-parts) and carries the rest back to stage k-1 as rows on (theta_k, v_k) (the constraint-to-go).  A carried row
//     with no part left, more than two, or one that reaches stage 0 means linearly dependent rows.
//   * one backward Riccati sweep on z = (x, y, theta, v, a_prev, delta_prev) with the exact Hessian of the Lagrangian
//     (cost Hessians incl. the distance term's radial and tangential curvature, and the second-order terms of the
//     dynamics weighted by the costates, node multipliers included), no flooring, no Levenberg term: the rows a stage
//     resolves fix u_k as a function of z_k, the free directions of u_k minimise the stage's Q-function (its reduced
//     Q_uu must be positive definite: the SOSC test), and the four parameter columns ride along as feed-forward terms.
//     dU_0/dp is stage 0's feed-forward term.
#pragma once
#include "mpc_kkt.cuh"

namespace mpcb {
namespace sens {

using kkt::Config;
using kkt::Problem;

// flag bits (include/mpc_b200.h MPC_SENS_*)
constexpr int kNotStationary = 1, kWeaklyActive = 2, kDegenerate = 4, kNotSosc = 8, kNonfinite = 16;
constexpr double kLicqTol = 1e-9;      // remaining norm of an active row against its norm: below = linearly dependent
constexpr double kSoscTol = 1e-10;     // Cholesky pivot of Z^T H Z against max(1, max |H_ff|): below = not positive definite
constexpr double kWeakTol = 1e-6;      // |multiplier| <= kWeakTol (1 + |J|): weakly active; below -kWeakTol (1 + |J|): wrong sign

KKT_HD inline double val(double a) { return a; }
KKT_HD inline double s_sin(double a) { return sin(a); }
KKT_HD inline double s_cos(double a) { return cos(a); }
KKT_HD inline double s_tan(double a) { return tan(a); }
KKT_HD inline double s_atan(double a) { return atan(a); }
KKT_HD inline double s_hypot(double a, double b) { return hypot(a, b); }
KKT_HD inline double s_floor(double a, double lo) { return a > lo ? a : lo; }

// Objective J(U; p) and g = grad_U [J + sum_{k=1..N} (wth[k] theta_k + wv[k] v_k)] by one rollout (into X) and one
// adjoint sweep.  prm = (vr_b, w_speed, w_control, w_diff).  The same terms as kkt::certify's gradient.  lam (may be
// null): [N][4] the adjoint of X[k + 1] as stage k sees it.  Written for a scalar type T so that a test can run it on dual
// numbers.
template <typename T>
KKT_HD T lagrangian_grad(const Config& cfg, const Problem& p, const T* U, const T* prm, const double* wth, const double* wv,
                         T (*X)[4], T* g, T (*lam_out)[4] = nullptr) {
  const int N = cfg.N;
  const double dt = cfg.dt;
  const bool track = !cfg.literal_no_collision;
  for (int c = 0; c < 4; ++c) X[0][c] = T{} + p.s0[c];
  for (int k = 0; k < N; ++k) {
    const T beta = s_atan(0.5 * s_tan(U[2 * k + 1]));
    const T* x = X[k];
    X[k + 1][0] = x[0] + dt * x[3] * s_cos(x[2] + beta);
    X[k + 1][1] = x[1] + dt * x[3] * s_sin(x[2] + beta);
    X[k + 1][2] = x[2] + dt * (x[3] / kkt::kL) * s_sin(beta);
    X[k + 1][3] = x[3] + dt * U[2 * k];
  }
  T J = T{};
  T lam[4] = {T{}, T{}, T{} + wth[N], T{} + wv[N]};   // adjoint of X[N]: no cost, the node-bound terms only
  for (int k = N - 1; k >= 0; --k) {
    const T* x = X[k];
    const T t = s_tan(U[2 * k + 1]);
    const T beta = s_atan(0.5 * t);
    const T db = 0.5 * (1.0 + t * t) / (1.0 + 0.25 * t * t);
    const T c = s_cos(x[2] + beta), sn = s_sin(x[2] + beta), v = x[3];
    if (lam_out) for (int e = 0; e < 4; ++e) lam_out[k][e] = lam[e];
    g[2 * k] = dt * lam[3];
    g[2 * k + 1] = (-dt * v * sn * db) * lam[0] + (dt * v * c * db) * lam[1] + (dt / kkt::kL) * v * s_cos(beta) * db * lam[2];
    T lx[4] = {T{}, T{}, T{}, T{}};
    if (track) {
      int j = p.ego_index + k;
      j = j < kkt::kNRefRows - 1 ? j : kkt::kNRefRows - 1;
      const double rx = cfg.ref[4 * j], ry = cfg.ref[4 * j + 1], rh = cfg.ref[4 * j + 3];
      const double sh = sin(rh), ch = cos(rh);
      const T dx = x[0] - rx, dy = x[1] - ry;
      const T perp = dx * sh - dy * ch, para = dx * ch + dy * sh;
      const T rv = k < p.vr_n ? T{} + (p.vr_a + double(k) * p.vr_slope) : prm[0];
      const T ev = x[3] - rv, eh = x[2] - rh;
      J = J + 10.0 * (4.0 * perp * perp + 2.0 * para * para + prm[1] * ev * ev + 0.5 * eh * eh);
      lx[0] = 10.0 * (8.0 * perp * sh + 4.0 * para * ch);
      lx[1] = 10.0 * (-8.0 * perp * ch + 4.0 * para * sh);
      lx[2] = 10.0 * eh;
      lx[3] = 20.0 * prm[1] * ev;
      if (cfg.w_distance != 0.0)
        for (int mo = 0; mo < p.n_obs; ++mo) {
          const float* o = p.obstacles + (long long)mo * 4 * p.obs_stride;
          const double ox = (double)o[0], oy = (double)o[p.obs_stride];
          const double ix = (double)o[2 * p.obs_stride], iy = (double)o[3 * p.obs_stride];
          const T ex = x[0] - (ox + double(k) * ix), ey = x[1] - (oy + double(k) * iy);
          const T dd = s_hypot(ex, ey);
          const double cc = val(dd) < 1.0 ? 1000.0 : 100.0;
          const T e1 = dd + 1e-6;
          J = J + cfg.w_distance * cc / (e1 * e1);
          const T coef = cfg.w_distance * (-2.0 * cc) / (e1 * e1 * e1 * s_floor(dd, 1e-300));
          lx[0] = lx[0] + coef * ex;
          lx[1] = lx[1] + coef * ey;
        }
      if (cfg.w_collision != 0.0 && p.is_collide) {
        J = J + cfg.w_collision * 3000.0 * x[3] * x[3];
        lx[3] = lx[3] + cfg.w_collision * 6000.0 * x[3];
      }
    }
    if (k == 0) break;
    lx[2] = lx[2] + wth[k];
    lx[3] = lx[3] + wv[k];
    const T A02 = -dt * v * sn, A03 = dt * c, A12 = dt * v * c, A13 = dt * sn, A23 = (dt / kkt::kL) * s_sin(beta);
    const T l2 = lam[2] + A02 * lam[0] + A12 * lam[1];
    const T l3 = lam[3] + A03 * lam[0] + A13 * lam[1] + A23 * lam[2];
    lam[0] = lx[0] + lam[0];
    lam[1] = lx[1] + lam[1];
    lam[2] = lx[2] + l2;
    lam[3] = lx[3] + l3;
  }
  for (int k = 0; k < N; ++k)
    for (int c = 0; c < 2; ++c) {
      const T u = U[2 * k + c];
      T gu = prm[2] * 0.02 * u;
      J = J + prm[2] * 0.01 * u * u;
      if (k > 0) {
        const T du = u - U[2 * (k - 1) + c];
        gu = gu + prm[3] * 0.02 * du;
        J = J + prm[3] * 0.01 * du * du;
      }
      if (k < N - 1) gu = gu - prm[3] * 0.02 * (U[2 * (k + 1) + c] - u);
      g[2 * k + c] = g[2 * k + c] + gu;
    }
  return J;
}

// ---------------------------------------------------------------------------------------------------------------------
// The sweep.  Stage k owns u_k and the constraint rows it can satisfy: its pinned control bounds, the theta / v bounds
// of node k+1, and the rows carried back from stage k+1.  Every node or carried row is a functional f on
// w_{k+1} = (theta_{k+1}, v_{k+1}), which depend on (theta_k, v_k, u_k) only:
//     w_{k+1} = T_k w_k + Bt_k u_k,   T_k = [[1, dt sin(beta_k) / L], [0, 1]],   Bt_k = [[0, wd_k], [dt, 0]]
// so a row's gradient is T_k^T f on w_k and Bt_k^T f on u_k.  Householder reflections with column pivoting on the rows'
// u-parts (m x 2) leave r <= 2 rows that fix u_k and m - r rows with no u-part, which are carried to stage k-1 as
// T_k^T f (the constraint-to-go).  A carried row with no w-part, more than two carried rows, or a carried row at
// stage 0 means the active rows are linearly dependent (DEGENERATE).  No carried row ever leaves the (theta, v) plane.

constexpr int kMaxRows = 6;             // 2 control bounds + 2 node bounds + 2 carried rows

struct StageRows {
  int m, r, piv, nc;                    // rows, rows that fix u_k, first pivot column, carried rows in
  int8_t tag[kMaxRows];                 // 0 bound of a_k, 1 of delta_k, 2 theta_{k+1}, 3 v_{k+1}, 4 + j carried row j
  double f[kMaxRows][2], du[kMaxRows][2];   // after the reflections
  double v0[kMaxRows], v1[kMaxRows], b0, b1;  // reflectors (b = 0: none)
};

template <int NMAX> struct Sweep {
  double X[NMAX + 1][4];
  double U[2 * NMAX], g[2 * NMAX];
  double lam[NMAX][4];                  // x-costate of X[k+1] of the Lagrangian (node multipliers included)
  double wth[NMAX + 1], wv[NMAX + 1];
  double sb[NMAX], wd[NMAX];            // sin(beta_k), d theta_{k+1} / d delta_k
  int8_t cs[2 * NMAX];                  // control: 0 free, +1 lower bound active, -1 upper
  int8_t nth[NMAX + 1], nv[NMAX + 1];   // node bound: 0 inactive, +1 lower, -1 upper
  double Mw[NMAX + 1][3], bw[NMAX + 1][2];   // W_k of the multiplier least squares (M symmetric 00 01 11, b)
  double mu[NMAX][4];                   // multipliers of the original rows by tag 0..3 (>= 0 at a KKT point)
  int8_t ncar[NMAX + 1];                // rows carried into stage k from stage k+1
  double car[NMAX + 1][2][2];           // those rows as functionals on w_{k+1}
};

KKT_HD inline void reflect(double (*f)[2], double (*du)[2], int lo, int m, double* v, double b) {
  for (int c = 0; c < 4; ++c) {
    double s = 0.0;
    for (int i = lo; i < m; ++i) s += v[i] * (c < 2 ? f[i][c] : du[i][c - 2]);
    s *= b;
    for (int i = lo; i < m; ++i) (c < 2 ? f[i][c] : du[i][c - 2]) -= s * v[i];
  }
}

// Householder vector for x[lo..m) of column `col` of du; returns false when its norm is <= tol
KKT_HD inline bool householder(double (*du)[2], int col, int lo, int m, double tol, double* v, double* b) {
  double nrm = 0.0;
  for (int i = lo; i < m; ++i) nrm += du[i][col] * du[i][col];
  nrm = sqrt(nrm);
  if (!(nrm > tol)) { *b = 0.0; return false; }
  const double x0 = du[lo][col], alpha = x0 > 0.0 ? -nrm : nrm;
  for (int i = 0; i < kMaxRows; ++i) v[i] = 0.0;
  for (int i = lo; i < m; ++i) v[i] = du[i][col];
  v[lo] -= alpha;
  double vv = 0.0;
  for (int i = lo; i < m; ++i) vv += v[i] * v[i];
  *b = 2.0 / vv;
  return true;
}

// Rows of stage k, reflected; writes the carried rows of stage k-1 into w.car[k] / w.ncar[k].  Returns false when the
// active rows are linearly dependent.
template <int NMAX> KKT_HD bool stage_rows(Sweep<NMAX>& w, int k, double dt, StageRows& s) {
  const double t01 = dt * w.sb[k] / kkt::kL;
  int m = 0;
  for (int c = 0; c < 2; ++c)
    if (w.cs[2 * k + c]) {
      s.tag[m] = (int8_t)c;
      s.f[m][0] = s.f[m][1] = 0.0;
      s.du[m][c] = w.cs[2 * k + c];
      s.du[m][1 - c] = 0.0;
      ++m;
    }
  double fr[4][2];
  int8_t tg[4];
  int nf = 0;
  if (w.nth[k + 1]) { fr[nf][0] = w.nth[k + 1]; fr[nf][1] = 0.0; tg[nf++] = 2; }
  if (w.nv[k + 1]) { fr[nf][0] = 0.0; fr[nf][1] = w.nv[k + 1]; tg[nf++] = 3; }
  s.nc = w.ncar[k + 1];
  for (int j = 0; j < s.nc; ++j) { fr[nf][0] = w.car[k + 1][j][0]; fr[nf][1] = w.car[k + 1][j][1]; tg[nf++] = (int8_t)(4 + j); }
  double scale = 1.0;
  for (int j = 0; j < nf; ++j) {
    s.tag[m] = tg[j];
    s.f[m][0] = fr[j][0]; s.f[m][1] = fr[j][1];
    s.du[m][0] = dt * fr[j][1];
    s.du[m][1] = w.wd[k] * fr[j][0];
    const double z0 = fr[j][0], z1 = t01 * fr[j][0] + fr[j][1];
    scale = fmax(scale, sqrt(z0 * z0 + z1 * z1 + s.du[m][0] * s.du[m][0] + s.du[m][1] * s.du[m][1]));
    ++m;
  }
  s.m = m;
  const double tol = kLicqTol * scale;
  double n0 = 0.0, n1 = 0.0;
  for (int i = 0; i < m; ++i) { n0 += s.du[i][0] * s.du[i][0]; n1 += s.du[i][1] * s.du[i][1]; }
  s.piv = n1 > n0 ? 1 : 0;
  s.r = 0;
  s.b1 = 0.0;
  if (householder(s.du, s.piv, 0, m, tol, s.v0, &s.b0)) {
    reflect(s.f, s.du, 0, m, s.v0, s.b0);
    s.r = 1;
    if (householder(s.du, 1 - s.piv, 1, m, tol, s.v1, &s.b1)) {
      reflect(s.f, s.du, 1, m, s.v1, s.b1);
      s.r = 2;
    }
  }
  const int nc = m - s.r;
  w.ncar[k] = (int8_t)nc;
  if (nc > 2 || (nc > 0 && k == 0)) return false;
  for (int j = 0; j < nc; ++j) {
    const double* f = s.f[s.r + j];
    const double z0 = f[0], z1 = t01 * f[0] + f[1];
    if (!(sqrt(z0 * z0 + z1 * z1) > tol)) return false;
    w.car[k][j][0] = z0;
    w.car[k][j][1] = z1;
  }
  return true;
}

// The sensitivity of one problem.  jac: [2][4] dU_0/dp (NaN unless the flags allow it).  mult (may be null): [N][4] in
// the layout of mpc_kkt's multipliers (> 0 at an upper bound, < 0 at a lower bound, 0 when inactive), written when the
// multipliers exist.  Returns the flag bits.
template <int NMAX>
KKT_HD int sensitivity(const Config& cfg, const Problem& p, const float* Uf, double act_tol, double stat_tol, Sweep<NMAX>& w,
                       double* jac, float* mult) {
  const int N = cfg.N, n = 2 * N;
  const double dt = cfg.dt;
  const double qnan = nan("");
  for (int c = 0; c < 8; ++c) jac[c] = qnan;
  if (mult) for (int i = 0; i < 4 * N; ++i) mult[i] = (float)qnan;
  const double prm[4] = {p.vr_b, p.w_speed, p.w_control, p.w_diff};
  for (int i = 0; i < n; ++i) w.U[i] = (double)Uf[i];
  for (int k = 0; k <= N; ++k) w.wth[k] = w.wv[k] = 0.0;
  const double J = lagrangian_grad<double>(cfg, p, w.U, prm, w.wth, w.wv, w.X, w.g);
  bool fin = kkt::finite_(J);
  for (int i = 0; i < n; ++i) fin = fin && kkt::finite_(w.U[i]) && kkt::finite_(w.g[i]);
  for (int k = 0; k <= N; ++k)
    for (int c = 0; c < 4; ++c) fin = fin && kkt::finite_(w.X[k][c]);
  if (!fin) return kNonfinite;
  // ---- active set
  bool dep = false;
  for (int i = 0; i < n; ++i) {
    const double u = w.U[i], lim = (i & 1) ? kkt::kDMax : kkt::kAMax;
    const bool lo = u + lim <= act_tol, hi = lim - u <= act_tol;
    dep = dep || (lo && hi);
    w.cs[i] = (int8_t)(lo ? 1 : hi ? -1 : 0);
  }
  w.nth[0] = w.nv[0] = 0;
  for (int k = 1; k <= N; ++k) {
    const double v = w.X[k][3], th = w.X[k][2];
    const bool vl = v - kkt::kVMin <= act_tol, vh = kkt::kVMax - v <= act_tol;
    const bool tl = th + kkt::kThMax <= act_tol, th_ = kkt::kThMax - th <= act_tol;
    dep = dep || (vl && vh) || (tl && th_);
    w.nv[k] = (int8_t)(vl ? 1 : vh ? -1 : 0);
    w.nth[k] = (int8_t)(tl ? 1 : th_ ? -1 : 0);
  }
  if (dep) return kDegenerate;
  for (int k = 0; k < N; ++k) {
    const double t = tan(w.U[2 * k + 1]);
    const double beta = atan(0.5 * t);
    const double db = 0.5 * (1.0 + t * t) / (1.0 + 0.25 * t * t);
    w.sb[k] = sin(beta);
    w.wd[k] = dt * (w.X[k][3] / kkt::kL) * cos(beta) * db;
  }
  // ---- the rows each stage resolves and carries (LICQ; the constraint-to-go of the Riccati pass below)
  StageRows s;
  w.ncar[N] = 0;
  for (int k = N - 1; k >= 0; --k)
    if (!stage_rows(w, k, dt, s)) return kDegenerate;
  // ---- multipliers: min over nu of sum_k |D_k (g_k - Bt_k^T psi_{k+1})|^2 with psi_k = E_k nu_k + T_k^T psi_{k+1},
  // psi_{N+1} = 0 (D_k keeps the free coordinates of u_k; the control-bound multipliers take the pinned ones exactly).
  // W_k(psi) = psi^T M psi - 2 b^T psi + const, the least cost of stages 0..k-1 given psi_k, forward in k; then back.
  double M[3] = {0.0, 0.0, 0.0}, bv[2] = {0.0, 0.0};   // M symmetric: 00, 01, 11
  auto stage_cost = [&](int k) {                       // + c_k(psi_{k+1}) = |D_k (g_k - Bt_k^T psi)|^2
    const double fa = w.cs[2 * k] ? 0.0 : 1.0, fd = w.cs[2 * k + 1] ? 0.0 : 1.0;
    M[0] += w.wd[k] * w.wd[k] * fd;
    M[2] += dt * dt * fa;
    bv[0] += w.wd[k] * fd * w.g[2 * k + 1];
    bv[1] += dt * fa * w.g[2 * k];
  };
  auto node_cols = [&](int k, double (*E)[2]) {        // active rows of node k as columns on w_k
    int q = 0;
    if (w.nth[k]) { E[q][0] = w.nth[k]; E[q][1] = 0.0; ++q; }
    if (w.nv[k]) { E[q][0] = 0.0; E[q][1] = w.nv[k]; ++q; }
    return q;
  };
  // nu = G^{-1} E^T (b - M a), G = E^T M E; false when G is singular (the rows of node k depend on the later ones)
  auto solve_nu = [&](const double* Mk, const double* bk, const double (*E)[2], int q, const double* a, double* nu) {
    double G[2][2], rhs[2];
    for (int i = 0; i < q; ++i) {
      const double me0 = Mk[0] * E[i][0] + Mk[1] * E[i][1], me1 = Mk[1] * E[i][0] + Mk[2] * E[i][1];
      for (int j = 0; j < q; ++j) G[j][i] = E[j][0] * me0 + E[j][1] * me1;
      const double ma0 = Mk[0] * a[0] + Mk[1] * a[1], ma1 = Mk[1] * a[0] + Mk[2] * a[1];
      rhs[i] = E[i][0] * (bk[0] - ma0) + E[i][1] * (bk[1] - ma1);
    }
    const double sc = kLicqTol * kLicqTol * fmax(fabs(Mk[0]) + fabs(Mk[2]), 1e-300);
    if (q == 1) {
      if (!(G[0][0] > sc)) return false;
      nu[0] = rhs[0] / G[0][0];
    } else if (q == 2) {
      const double d1 = G[1][1] - G[1][0] * G[0][1] / G[0][0];
      if (!(G[0][0] > sc) || !(d1 > sc)) return false;
      const double det = G[0][0] * G[1][1] - G[0][1] * G[1][0];
      nu[0] = (rhs[0] * G[1][1] - G[0][1] * rhs[1]) / det;
      nu[1] = (G[0][0] * rhs[1] - G[1][0] * rhs[0]) / det;
    }
    return true;
  };
  stage_cost(0);
  for (int k = 1; k < N; ++k) {                        // W_k -> W_{k+1}
    w.Mw[k][0] = M[0]; w.Mw[k][1] = M[1]; w.Mw[k][2] = M[2]; w.bw[k][0] = bv[0]; w.bw[k][1] = bv[1];
    double E[2][2];
    const int q = node_cols(k, E);
    if (q) {                                           // minimise over nu_k: Schur complement of E^T M E
      double MinvE[2][2];                              // columns: G^{-1}-weighted M E
      const double z[2] = {0.0, 0.0};
      double Mn[3] = {M[0], M[1], M[2]}, bn[2] = {bv[0], bv[1]};
      for (int e = 0; e < 2; ++e) {                    // M' = M - M E G^{-1} E^T M by probing with unit vectors
        double nu[2], ae[2] = {e == 0 ? 1.0 : 0.0, e == 1 ? 1.0 : 0.0};
        double b0[2] = {0.0, 0.0};
        if (!solve_nu(M, b0, E, q, ae, nu)) return kDegenerate;   // nu = -G^{-1} E^T M e
        for (int c = 0; c < 2; ++c) MinvE[e][c] = 0.0;
        double v0 = 0.0, v1 = 0.0;                     // E nu
        for (int i = 0; i < q; ++i) { v0 += E[i][0] * nu[i]; v1 += E[i][1] * nu[i]; }
        MinvE[e][0] = v0; MinvE[e][1] = v1;            // (I + E L) e with L = -G^{-1} E^T M
      }
      {
        double nu[2];
        if (!solve_nu(M, bv, E, q, z, nu)) return kDegenerate;   // nu = G^{-1} E^T b
        double v0 = 0.0, v1 = 0.0;
        for (int i = 0; i < q; ++i) { v0 += E[i][0] * nu[i]; v1 += E[i][1] * nu[i]; }
        bn[0] = bv[0] - (M[0] * v0 + M[1] * v1);       // b' = b - M E G^{-1} E^T b
        bn[1] = bv[1] - (M[1] * v0 + M[2] * v1);
      }
      // M' = M (I + E L) (symmetric): column e of M' = M (e + E L e)
      const double c00 = 1.0 + MinvE[0][0], c10 = MinvE[0][1], c01 = MinvE[1][0], c11 = 1.0 + MinvE[1][1];
      Mn[0] = M[0] * c00 + M[1] * c10;
      Mn[1] = 0.5 * ((M[0] * c01 + M[1] * c11) + (M[1] * c00 + M[2] * c10));
      Mn[2] = M[1] * c01 + M[2] * c11;
      M[0] = Mn[0]; M[1] = Mn[1]; M[2] = Mn[2]; bv[0] = bn[0]; bv[1] = bn[1];
    }
    // psi_k = T_k^T psi_{k+1} (+ E nu): W(T^T psi): M <- T M T^T, b <- T b, T = [[1, t], [0, 1]]
    const double t = dt * w.sb[k] / kkt::kL;
    const double m00 = M[0] + 2.0 * t * M[1] + t * t * M[2], m01 = M[1] + t * M[2];
    M[0] = m00; M[1] = m01;
    bv[0] += t * bv[1];
    stage_cost(k);
  }
  w.Mw[N][0] = M[0]; w.Mw[N][1] = M[1]; w.Mw[N][2] = M[2]; w.bw[N][0] = bv[0]; w.bw[N][1] = bv[1];
  // back: nu_N from psi_{N+1} = 0, then nu_k given psi_{k+1}; residual and control-bound multipliers per stage
  double psi[2] = {0.0, 0.0}, res2 = 0.0;              // psi_{k+1}
  for (int k = N; k >= 1; --k) {
    double E[2][2], nu[2] = {0.0, 0.0};
    const int q = node_cols(k, E);
    double a[2] = {psi[0], psi[1]};                    // T_k^T psi_{k+1} (k < N)
    if (k < N) a[1] += dt * w.sb[k] / kkt::kL * psi[0];
    if (k == N) a[0] = a[1] = 0.0;
    if (q && !solve_nu(w.Mw[k], w.bw[k], E, q, a, nu)) return kDegenerate;
    for (int c = 2; c < 4; ++c) w.mu[k - 1][c] = 0.0;
    for (int i = 0; i < q; ++i) {
      a[0] += E[i][0] * nu[i];
      a[1] += E[i][1] * nu[i];
      w.mu[k - 1][E[i][1] != 0.0 ? 3 : 2] = nu[i];
    }
    psi[0] = a[0]; psi[1] = a[1];                      // psi_k
    // stage k-1 sees psi_k
    const int j = k - 1;
    const double r[2] = {w.g[2 * j] - dt * psi[1], w.g[2 * j + 1] - w.wd[j] * psi[0]};
    for (int c = 0; c < 2; ++c) {
      if (w.cs[2 * j + c]) w.mu[j][c] = double(w.cs[2 * j + c]) * r[c];
      else { w.mu[j][c] = 0.0; res2 += r[c] * r[c]; }
    }
  }
  const double tau = stat_tol * (1.0 + fabs(J)), tw = kWeakTol * (1.0 + fabs(J));
  int flags = sqrt(res2) > tau ? kNotStationary : 0;
  double mmin = 1e300;
  if (mult) for (int i = 0; i < 4 * N; ++i) mult[i] = 0.f;
  for (int k = 0; k < N; ++k) {
    const int8_t sg[4] = {w.cs[2 * k], w.cs[2 * k + 1], w.nth[k + 1], w.nv[k + 1]};
    for (int c = 0; c < 4; ++c)
      if (sg[c]) {
        mmin = fmin(mmin, w.mu[k][c]);
        if (mult) mult[k * 4 + c] = (float)(-double(sg[c]) * w.mu[k][c]);
      }
    w.wth[k + 1] = w.nth[k + 1] ? -double(w.nth[k + 1]) * w.mu[k][2] : 0.0;   // L = J - sum nu c, c = s (x - bound)
    w.wv[k + 1] = w.nv[k + 1] ? -double(w.nv[k + 1]) * w.mu[k][3] : 0.0;
  }
  if (mmin < -tw) flags |= kNotStationary;
  else if (mmin <= tw) flags |= kWeaklyActive;
  // ---- costates of the Lagrangian
  lagrangian_grad<double>(cfg, p, w.U, prm, w.wth, w.wv, w.X, w.g, w.lam);
  // ---- backward pass 2: Riccati on z = (x, y, theta, v, a_prev, delta_prev) with the exact Lagrangian Hessian
  double P[6][6], pv[6][4];
  for (int i = 0; i < 6; ++i) {
    for (int j = 0; j < 6; ++j) P[i][j] = 0.0;
    for (int c = 0; c < 4; ++c) pv[i][c] = 0.0;
  }
  const bool track = !cfg.literal_no_collision;
  for (int k = N - 1; k >= 0; --k) {
    stage_rows(w, k, dt, s);
    const double* x = w.X[k];
    const double ud = w.U[2 * k + 1];
    const double t = tan(ud), beta = atan(0.5 * t);
    const double db = 0.5 * (1.0 + t * t) / (1.0 + 0.25 * t * t);
    const double d2b = 0.75 * t * (1.0 + t * t) / ((1.0 + 0.25 * t * t) * (1.0 + 0.25 * t * t));
    const double c = cos(x[2] + beta), sn = sin(x[2] + beta), v = x[3], cb = cos(beta), sbk = sin(beta);
    double A[4][4] = {{1, 0, -dt * v * sn, dt * c}, {0, 1, dt * v * c, dt * sn}, {0, 0, 1, dt * sbk / kkt::kL}, {0, 0, 0, 1}};
    double Bm[4][2] = {{0, -dt * v * sn * db}, {0, dt * v * c * db}, {0, dt * v * cb * db / kkt::kL}, {dt, 0}};
    // stage Hessians and parameter gradients
    double lzz[6][6] = {}, luz[2][6] = {}, luu[2][2] = {}, lzp[6][4] = {}, lup[2][4] = {};
    if (track && k > 0) {
      int j = p.ego_index + k;
      j = j < kkt::kNRefRows - 1 ? j : kkt::kNRefRows - 1;
      const double rh = cfg.ref[4 * j + 3], sh = sin(rh), ch = cos(rh);
      lzz[0][0] = 10.0 * (8.0 * sh * sh + 4.0 * ch * ch);
      lzz[1][1] = 10.0 * (8.0 * ch * ch + 4.0 * sh * sh);
      lzz[0][1] = lzz[1][0] = 10.0 * (-8.0 * sh * ch + 4.0 * ch * sh);
      lzz[2][2] = 10.0;
      lzz[3][3] = 20.0 * p.w_speed + (cfg.w_collision != 0.0 && p.is_collide ? cfg.w_collision * 6000.0 : 0.0);
      const double rv = k < p.vr_n ? p.vr_a + double(k) * p.vr_slope : p.vr_b;
      lzp[3][0] = k < p.vr_n ? 0.0 : -20.0 * p.w_speed;
      lzp[3][1] = 20.0 * (x[3] - rv);
      if (cfg.w_distance != 0.0)
        for (int mo = 0; mo < p.n_obs; ++mo) {             // radial phi'' rr^T and tangential phi'/d (I - rr^T) curvature
          const float* o = p.obstacles + (long long)mo * 4 * p.obs_stride;
          const double ex = x[0] - ((double)o[0] + double(k) * (double)o[2 * p.obs_stride]);
          const double ey = x[1] - ((double)o[p.obs_stride] + double(k) * (double)o[3 * p.obs_stride]);
          const double dd = hypot(ex, ey), cc = dd < 1.0 ? 1000.0 : 100.0, e1 = dd + 1e-6;
          const double d1 = -2.0 * cfg.w_distance * cc / (e1 * e1 * e1), d2 = 6.0 * cfg.w_distance * cc / (e1 * e1 * e1 * e1);
          const double dm = fmax(dd, 1e-300), rx = ex / dm, ry = ey / dm, tg = d1 / dm;
          lzz[0][0] += d2 * rx * rx + tg * (1.0 - rx * rx);
          lzz[1][1] += d2 * ry * ry + tg * (1.0 - ry * ry);
          lzz[0][1] += (d2 - tg) * rx * ry;
          lzz[1][0] += (d2 - tg) * rx * ry;
        }
    }
    const double wdk = k > 0 ? p.w_diff : 0.0;
    for (int a = 0; a < 2; ++a) {
      const double u = w.U[2 * k + a], up = k > 0 ? w.U[2 * k - 2 + a] : 0.0;
      luu[a][a] = 0.02 * (p.w_control + wdk);
      luz[a][4 + a] = -0.02 * wdk;
      lzz[4 + a][4 + a] = 0.02 * wdk;
      lup[a][2] = 0.02 * u;
      if (k > 0) { lup[a][3] = 0.02 * (u - up); lzp[4 + a][3] = -0.02 * (u - up); }
    }
    // multiplier-weighted second-order terms of the dynamics, variables (theta, v, delta)
    const double* l = w.lam[k];
    const double htt = l[0] * (-dt * v * c) + l[1] * (-dt * v * sn);
    const double htv = l[0] * (-dt * sn) + l[1] * (dt * c);
    const double htd = l[0] * (-dt * v * c * db) + l[1] * (-dt * v * sn * db);
    const double hvd = l[0] * (-dt * sn * db) + l[1] * (dt * c * db) + l[2] * (dt * cb * db / kkt::kL);
    const double hdd = l[0] * (-dt * v * (c * db * db + sn * d2b)) + l[1] * (dt * v * (-sn * db * db + c * d2b))
                     + l[2] * (dt * v * (-sbk * db * db + cb * d2b) / kkt::kL);
    lzz[2][2] += htt; lzz[2][3] += htv; lzz[3][2] += htv;
    luz[1][2] += htd; luz[1][3] += hvd; luu[1][1] += hdd;
    // Q = l + F^T V' F with F_z = [A 0; 0 0], F_u = [B; I]
    double PA[6][4], PB[6][2];                   // P F_z (columns 0..3), P F_u
    for (int i = 0; i < 6; ++i) {
      for (int j = 0; j < 4; ++j) { double a = 0.0; for (int q = 0; q < 4; ++q) a += P[i][q] * A[q][j]; PA[i][j] = a; }
      for (int j = 0; j < 2; ++j) {
        double a = P[i][4 + j];
        for (int q = 0; q < 4; ++q) a += P[i][q] * Bm[q][j];
        PB[i][j] = a;
      }
    }
    double Qzz[6][6], Quz[2][6], Quu[2][2], qz[6][4], qu[2][4];
    for (int i = 0; i < 6; ++i)
      for (int j = 0; j < 6; ++j) {
        double a = lzz[i][j];
        if (i < 4 && j < 4) for (int q = 0; q < 4; ++q) a += A[q][i] * PA[q][j];
        Qzz[i][j] = a;
      }
    for (int i = 0; i < 2; ++i) {
      for (int j = 0; j < 6; ++j) {
        double a = luz[i][j];
        if (j < 4) {
          a += PA[4 + i][j];
          for (int q = 0; q < 4; ++q) a += Bm[q][i] * PA[q][j];
        }
        Quz[i][j] = a;
      }
      for (int j = 0; j < 2; ++j) {
        double a = luu[i][j] + PB[4 + i][j];
        for (int q = 0; q < 4; ++q) a += Bm[q][i] * PB[q][j];
        Quu[i][j] = a;
      }
      for (int cc = 0; cc < 4; ++cc) {
        double a = lup[i][cc] + pv[4 + i][cc];
        for (int q = 0; q < 4; ++q) a += Bm[q][i] * pv[q][cc];
        qu[i][cc] = a;
      }
    }
    for (int i = 0; i < 6; ++i)
      for (int cc = 0; cc < 4; ++cc) {
        double a = lzp[i][cc];
        if (i < 4) for (int q = 0; q < 4; ++q) a += A[q][i] * pv[q][cc];
        qz[i][cc] = a;
      }
    // policy du = K dz + kff under the rows that fix u_k: du_j . du + (T_k^T f_j) . (dtheta_k, dv_k) = 0
    double K[2][6] = {}, kff[2][4] = {};
    const double t01 = dt * sbk / kkt::kL;
    const double sosc_tol = kSoscTol * fmax(1.0, fmax(fabs(Quu[0][0]), fabs(Quu[1][1])));
    if (s.r == 2) {
      const double a = s.du[0][0], b = s.du[0][1], c2 = s.du[1][0], d = s.du[1][1], det = a * d - b * c2;
      double Z[2][2];                             // rows: the w_k-parts
      for (int j = 0; j < 2; ++j) { Z[j][0] = s.f[j][0]; Z[j][1] = t01 * s.f[j][0] + s.f[j][1]; }
      for (int q = 0; q < 2; ++q) {               // du = -M^{-1} Z dw, M rows du_j
        K[0][2 + q] = -(d * Z[0][q] - b * Z[1][q]) / det;
        K[1][2 + q] = -(-c2 * Z[0][q] + a * Z[1][q]) / det;
      }
    } else if (s.r == 1) {
      const double r0 = s.du[0][0], r1 = s.du[0][1], nn = r0 * r0 + r1 * r1, ln = sqrt(nn);
      const double z0 = s.f[0][0], z1 = t01 * s.f[0][0] + s.f[0][1];
      const double nv0 = -r1 / ln, nv1 = r0 / ln;
      K[0][2] = -r0 * z0 / nn; K[0][3] = -r0 * z1 / nn;
      K[1][2] = -r1 * z0 / nn; K[1][3] = -r1 * z1 / nn;
      const double h = nv0 * (Quu[0][0] * nv0 + Quu[0][1] * nv1) + nv1 * (Quu[1][0] * nv0 + Quu[1][1] * nv1);
      if (!(h > sosc_tol)) { flags |= kNotSosc; break; }
      double row[6];
      for (int j = 0; j < 6; ++j)
        row[j] = nv0 * (Quu[0][0] * K[0][j] + Quu[0][1] * K[1][j] + Quz[0][j]) + nv1 * (Quu[1][0] * K[0][j] + Quu[1][1] * K[1][j] + Quz[1][j]);
      for (int j = 0; j < 6; ++j) { K[0][j] -= nv0 * row[j] / h; K[1][j] -= nv1 * row[j] / h; }
      for (int cc = 0; cc < 4; ++cc) {
        const double rq = (nv0 * qu[0][cc] + nv1 * qu[1][cc]) / h;
        kff[0][cc] = -nv0 * rq; kff[1][cc] = -nv1 * rq;
      }
    } else {
      const double d0 = Quu[0][0];
      const double l10 = Quu[1][0] / d0, d1 = Quu[1][1] - l10 * Quu[0][1];
      if (!(d0 > sosc_tol) || !(d1 > sosc_tol)) { flags |= kNotSosc; break; }
      const double det = Quu[0][0] * Quu[1][1] - Quu[0][1] * Quu[1][0];
      const double i00 = Quu[1][1] / det, i01 = -Quu[0][1] / det, i10 = -Quu[1][0] / det, i11 = Quu[0][0] / det;
      for (int j = 0; j < 6; ++j) { K[0][j] = -(i00 * Quz[0][j] + i01 * Quz[1][j]); K[1][j] = -(i10 * Quz[0][j] + i11 * Quz[1][j]); }
      for (int cc = 0; cc < 4; ++cc) { kff[0][cc] = -(i00 * qu[0][cc] + i01 * qu[1][cc]); kff[1][cc] = -(i10 * qu[0][cc] + i11 * qu[1][cc]); }
    }
    if (k == 0) {
      for (int cc = 0; cc < 4; ++cc) { jac[cc] = kff[0][cc]; jac[4 + cc] = kff[1][cc]; }
      break;
    }
    // V_k: P = Qzz + K^T (Quu K + Quz) + Quz^T K, p = qz + K^T qu + (Quz^T + K^T Quu) kff
    double QK[2][6];                              // Quu K + Quz
    for (int i = 0; i < 2; ++i)
      for (int j = 0; j < 6; ++j) QK[i][j] = Quu[i][0] * K[0][j] + Quu[i][1] * K[1][j] + Quz[i][j];
    for (int i = 0; i < 6; ++i)
      for (int j = 0; j <= i; ++j) {
        const double a = Qzz[i][j] + K[0][i] * QK[0][j] + K[1][i] * QK[1][j] + Quz[0][i] * K[0][j] + Quz[1][i] * K[1][j];
        const double b = Qzz[j][i] + K[0][j] * QK[0][i] + K[1][j] * QK[1][i] + Quz[0][j] * K[0][i] + Quz[1][j] * K[1][i];
        P[i][j] = P[j][i] = 0.5 * (a + b);
      }
    for (int i = 0; i < 6; ++i)
      for (int cc = 0; cc < 4; ++cc)
        pv[i][cc] = qz[i][cc] + K[0][i] * qu[0][cc] + K[1][i] * qu[1][cc]
                  + (Quz[0][i] + Quu[0][0] * K[0][i] + Quu[1][0] * K[1][i]) * kff[0][cc]
                  + (Quz[1][i] + Quu[0][1] * K[0][i] + Quu[1][1] * K[1][i]) * kff[1][cc];
  }
  if (flags & (kNotStationary | kNotSosc)) for (int c = 0; c < 8; ++c) jac[c] = qnan;
  return flags;
}
}  // namespace sens
}  // namespace mpcb
