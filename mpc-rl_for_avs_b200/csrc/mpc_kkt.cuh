// mpc_kkt.cuh -- per-problem FP64 optimality certificate (first-order KKT residual) of given controls.
//
// What is computed is exactly the oracle's `kkt_residual(U, prob, act_tol)`, in FP64 on the
// float32 controls as given:
//   rollout    explicit Euler, no clamping (pure_mpc.py:220-228, 252-254)
//   g          grad_U J of the objective the solver minimises (tracking, unwrapped heading, speed against the per-stage
//              reference-speed descriptor, control, input difference, the archive distance term with its d < 1 branch,
//              the collision term when is_collide; control + input difference only under literal_no_collision), by one
//              reverse (adjoint) sweep
//   active set a control bound, or a theta / v bound of nodes 1..N, within act_tol
//   residual   min_{mu >= 0} || g - J_act^T mu ||_2   (the projection of g onto the cone of the active constraint
//              gradients is unique, so the residual is well defined even where the multipliers are not)
//   violation  the largest bound violation
// The node bounds only involve (theta, v), which do not depend on (x, y): v_k = v_0 + dt sum_{j<k} a_j and
// theta_k = theta_0 + (dt / L) sum_{j<k} v_j sin beta_j.  A node row d x_k[theta|v] / dU therefore has O(1) closed-form
// entries (prefix sums of sin beta), so no row is ever stored.  The control-bound columns are +-unit vectors on distinct
// coordinates: for fixed node multipliers nu their best multiplier is max(0, +-r_i), which the Lawson-Hanson NNLS below
// exploits by treating a passive control column as "coordinate i removed from the least-squares problem".  The normal
// matrix of the passive node columns lives in caller-provided storage of `cap` x `cap` doubles.
//
// The functions compile for the device (k_kkt, csrc/mpc_kkt.cu) and for the host (the test-only host harness).
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define KKT_HD __host__ __device__
#else
#define KKT_HD
#endif

namespace mpcb {
namespace kkt {

constexpr double kL = 2.5;                                   // wheelbase, agents/utils.py:18
constexpr double kAMax = 5.0;                                // pure_mpc.py:279-280
constexpr double kDMax = 3.14159265358979323846 / 3.0;
constexpr double kVMin = 0.0, kVMax = 30.0;                  // pure_mpc.py:273-274
constexpr double kThMax = 3.14159265358979323846;
constexpr int kNRefRows = 85;

// one problem as the batch holds it (MpcProblemBatch, float32), widened to FP64
struct Problem {
  double s0[4];
  int ego_index, n_obs, is_collide;
  double w_speed, w_control, w_diff;
  double vr_a, vr_slope, vr_b;
  int vr_n;
  const float* obstacles;      // [M][4][stride] base + problem index: x, y, speed*dt*cos h, speed*dt*sin h
  long long obs_stride;
};
struct Config {
  int N;
  double dt;                   // the double 1 / policy_frequency
  double w_distance, w_collision;
  int literal_no_collision;
  const double* ref;           // [85][4] x, y, v, heading (RefTables::ref)
};
struct Result {
  double residual, grad_norm, violation;
  int n_active;
};

// problem i of a batch of B in the MpcProblemBatch layout (any struct with its field names)
template <typename BatchT> KKT_HD Problem load_problem(const BatchT& b, long long B, long long i, int M) {
  Problem p;
  for (int c = 0; c < 4; ++c) p.s0[c] = (double)b.s0[c * B + i];
  p.ego_index = b.ego_index[i];
  p.n_obs = (b.n_obs && b.obstacles) ? b.n_obs[i] : 0;
  p.n_obs = p.n_obs < M ? p.n_obs : M;
  p.is_collide = b.is_collide ? b.is_collide[i] : 0;
  p.w_speed = (double)b.w_speed[i]; p.w_control = (double)b.w_control[i]; p.w_diff = (double)b.w_diff[i];
  p.vr_a = (double)b.vr_a[i]; p.vr_slope = (double)b.vr_slope[i]; p.vr_b = (double)b.vr_b[i]; p.vr_n = b.vr_n[i];
  p.obstacles = b.obstacles ? b.obstacles + i : nullptr;
  p.obs_stride = B;
  return p;
}

// Per-problem work arrays for horizons up to NMAX.
template <int NMAX> struct Work {
  double X[NMAX + 1][4];
  double g[2 * NMAX];
  double wd[NMAX];             // d theta_{j+1} / d delta_j = dt v_j cos beta_j beta'(delta_j) / L
  double S[NMAX + 1];          // S[n] = sum_{m<n} sin beta_m
  double mu[2 * NMAX];         // control multipliers (>= 0), trial values in sc
  double sc[2 * NMAX];
  double nu[4 * NMAX];         // node multipliers (>= 0), trial values in sq
  double sq[4 * NMAX];
  double r[2 * NMAX];          // residual vector
  int8_t cs[2 * NMAX];        // control coordinate: 0 inactive, +1 lower bound active, -1 upper, 2 both
  uint8_t pc[2 * NMAX];        // control column passive
  uint8_t bc[2 * NMAX];        // control column excluded until the iterate moves
  uint16_t node[4 * NMAX];     // active node bound q: k << 2 | comp << 1 | upper   (comp 0 = theta, 1 = v)
  uint8_t pq[4 * NMAX];        // node column passive
  uint8_t ban[4 * NMAX];       // node column excluded until the iterate moves (dependent on the passive set)
  int16_t Q[4 * NMAX];         // passive node columns in order of entry
  int nq, m;
};

KKT_HD inline bool finite_(double x) { return x - x == 0.0; }

// entry i of d x_k[comp] / dU (no sign)
template <int NMAX> KKT_HD inline double node_row(const Work<NMAX>& w, double dt, int k, int comp, int i) {
  const int j = i >> 1;
  if (j >= k) return 0.0;
  if (comp == 1) return (i & 1) ? 0.0 : dt;
  if (i & 1) return w.wd[j];
  return dt * dt / kL * (w.S[k] - w.S[j + 1]);
}
template <int NMAX> KKT_HD inline double col_entry(const Work<NMAX>& w, double dt, int q, int i) {
  const int e = w.node[q];
  const double r = node_row(w, dt, e >> 2, (e >> 1) & 1, i);
  return (e & 1) ? -r : r;                       // lower bound x - lb >= 0: +row; upper ub - x >= 0: -row
}
template <int NMAX> KKT_HD inline bool eliminated(const Work<NMAX>& w, int i) {
  return w.cs[i] == 2 || (w.cs[i] != 0 && w.pc[i]);
}

// r = g - sum_q nu_q a_q - sum_i sigma_i mu_i e_i at the current iterate, with the coordinates of both-sided control
// bounds zeroed (their two columns span the axis)
template <int NMAX> KKT_HD void residual_vec(const Work<NMAX>& w, int n, double dt, double* r) {
  for (int i = 0; i < n; ++i) {
    double v = w.g[i];
    for (int q = 0; q < w.nq; ++q)
      if (w.nu[q] != 0.0) v -= w.nu[q] * col_entry(w, dt, q, i);
    if (w.cs[i] == 2) v = 0.0;
    else if (w.cs[i] != 0) v -= double(w.cs[i]) * w.mu[i];
    r[i] = v;
  }
}

// Least squares on the passive set: node multipliers z (into sq) minimise || (g - A_Q z) || over the coordinates that
// no passive control column removes; the passive control columns take the rest exactly (into sc).  Returns false when
// the normal matrix is singular (the newest passive column depends on the others) or would exceed cap.
template <int NMAX> KKT_HD bool passive_ls(Work<NMAX>& w, int n, double dt, double* G, int cap) {
  const int m = w.m;
  if (m > cap) return false;
  for (int a = 0; a < m; ++a) {
    const int qa = w.Q[a];
    double h = 0.0;
    for (int b = 0; b <= a; ++b) {
      const int qb = w.Q[b];
      double s = 0.0;
      for (int i = 0; i < n; ++i)
        if (!eliminated(w, i)) s += col_entry(w, dt, qa, i) * col_entry(w, dt, qb, i);
      G[a * cap + b] = s;
    }
    for (int i = 0; i < n; ++i)
      if (!eliminated(w, i)) h += col_entry(w, dt, qa, i) * w.g[i];
    w.sq[qa] = h;
  }
  // Cholesky in place (lower triangle)
  for (int a = 0; a < m; ++a) {
    const double d0 = G[a * cap + a];
    double d = d0;
    for (int c = 0; c < a; ++c) d -= G[a * cap + c] * G[a * cap + c];
    if (!(d > 1e-12 * d0) || !(d0 > 0.0)) return false;
    d = sqrt(d);
    G[a * cap + a] = d;
    for (int b = a + 1; b < m; ++b) {
      double s = G[b * cap + a];
      for (int c = 0; c < a; ++c) s -= G[b * cap + c] * G[a * cap + c];
      G[b * cap + a] = s / d;
    }
  }
  for (int a = 0; a < m; ++a) {                  // L y = h
    double s = w.sq[w.Q[a]];
    for (int c = 0; c < a; ++c) s -= G[a * cap + c] * w.sq[w.Q[c]];
    w.sq[w.Q[a]] = s / G[a * cap + a];
  }
  for (int a = m - 1; a >= 0; --a) {             // L^T z = y
    double s = w.sq[w.Q[a]];
    for (int c = a + 1; c < m; ++c) s -= G[c * cap + a] * w.sq[w.Q[c]];
    w.sq[w.Q[a]] = s / G[a * cap + a];
  }
  for (int i = 0; i < n; ++i) {
    if (w.cs[i] == 2 || w.cs[i] == 0 || !w.pc[i]) continue;
    double v = w.g[i];
    for (int a = 0; a < m; ++a) v -= w.sq[w.Q[a]] * col_entry(w, dt, w.Q[a], i);
    w.sc[i] = double(w.cs[i]) * v;
  }
  return true;
}

template <int NMAX> KKT_HD void drop_passive_node(Work<NMAX>& w, int a) {
  w.pq[w.Q[a]] = 0;
  for (int b = a + 1; b < w.m; ++b) w.Q[b - 1] = w.Q[b];
  --w.m;
}

// Lawson-Hanson NNLS over the control columns (unit vectors) and the node columns.  r is scratch of n doubles.
template <int NMAX> KKT_HD void nnls(Work<NMAX>& w, int n, double dt, double gnorm, double* G, int cap, double* r) {
  const int ncols = n + w.nq;
  const double tol = 1e-14 * (1.0 + gnorm);
  w.m = 0;
  for (int it = 0; it < 3 * ncols + 10; ++it) {
    residual_vec(w, n, dt, r);
    // the most positive dual among the columns outside the passive set
    int pick = -1;
    double best = tol;
    for (int i = 0; i < n; ++i) {
      if ((w.cs[i] != 1 && w.cs[i] != -1) || w.pc[i] || w.bc[i]) continue;
      const double d = double(w.cs[i]) * r[i];
      if (d > best) { best = d; pick = i; }
    }
    for (int q = 0; q < w.nq; ++q) {
      if (w.pq[q] || w.ban[q]) continue;
      double d = 0.0;
      for (int i = 0; i < n; ++i) d += col_entry(w, dt, q, i) * r[i];
      if (d > best) { best = d; pick = n + q; }
    }
    if (pick < 0) return;
    if (pick < n) { w.pc[pick] = 1; w.mu[pick] = 0.0; }
    else { const int q = pick - n; w.pq[q] = 1; w.nu[q] = 0.0; w.Q[w.m++] = (int16_t)q; }
    // inner loop: step towards the unconstrained least-squares point of the passive set, stopping at the first
    // multiplier that would turn negative
    bool moved = false;
    for (int inner = 0; inner < ncols + 1; ++inner) {
      if (!passive_ls(w, n, dt, G, cap)) {
        // the newest column depends on the passive set: take it out again and keep it out until the iterate moves
        if (pick < n) { w.pc[pick] = 0; w.bc[pick] = 1; }
        else { w.ban[pick - n] = 1; drop_passive_node(w, w.m - 1); }
        break;
      }
      bool all_pos = true;
      double alpha = 1.0;
      for (int i = 0; i < n; ++i)
        if (w.cs[i] != 2 && w.cs[i] != 0 && w.pc[i] && !(w.sc[i] > 0.0)) {
          all_pos = false;
          const double den = w.mu[i] - w.sc[i];
          const double al = den > 0.0 ? w.mu[i] / den : 0.0;
          if (al < alpha) alpha = al;
        }
      for (int a = 0; a < w.m; ++a) {
        const int q = w.Q[a];
        if (!(w.sq[q] > 0.0)) {
          all_pos = false;
          const double den = w.nu[q] - w.sq[q];
          const double al = den > 0.0 ? w.nu[q] / den : 0.0;
          if (al < alpha) alpha = al;
        }
      }
      if (all_pos) {
        for (int i = 0; i < n; ++i)
          if (w.cs[i] != 2 && w.cs[i] != 0 && w.pc[i]) w.mu[i] = w.sc[i];
        for (int a = 0; a < w.m; ++a) w.nu[w.Q[a]] = w.sq[w.Q[a]];
        moved = true;
        break;
      }
      // interpolate and drop every passive column that reached zero
      for (int i = 0; i < n; ++i)
        if (w.cs[i] != 2 && w.cs[i] != 0 && w.pc[i]) {
          w.mu[i] += alpha * (w.sc[i] - w.mu[i]);
          if (!(w.mu[i] > 0.0)) { w.mu[i] = 0.0; w.pc[i] = 0; }
        }
      for (int a = w.m - 1; a >= 0; --a) {
        const int q = w.Q[a];
        w.nu[q] += alpha * (w.sq[q] - w.nu[q]);
        if (!(w.nu[q] > 0.0)) { w.nu[q] = 0.0; drop_passive_node(w, a); }
      }
      moved = moved || alpha > 0.0;
    }
    if (moved) {
      for (int q = 0; q < w.nq; ++q) w.ban[q] = 0;
      for (int i = 0; i < n; ++i) w.bc[i] = 0;
    }
  }
}

// The certificate of one problem.  U: the problem's [N][2] float controls.  mult (may be null): [N][4] = mu of a_k,
// mu of delta_k, nu of theta_{k+1}, nu of v_{k+1}; > 0 at an upper bound, < 0 at a lower bound, 0 when inactive.
// G: cap x cap doubles for the normal matrix of the passive node columns; cap = 2N always suffices (the passive node
// columns stay linearly independent).  Returns false, having written nothing but res->n_active, when the problem has
// more than defer_above active node bounds (the caller then retries where a larger G fits).
template <int NMAX>
KKT_HD bool certify(const Config& cfg, const Problem& p, const float* U, double act_tol, Work<NMAX>& w, double* G, int cap,
                    int defer_above, Result* res, float* mult) {
  const int N = cfg.N, n = 2 * N;
  const double dt = cfg.dt;
  // ---- rollout (FP64, no clamping), steering terms of every stage
  for (int c = 0; c < 4; ++c) w.X[0][c] = p.s0[c];
  w.S[0] = 0.0;
  bool fin = true;
  for (int k = 0; k < N; ++k) {
    const double a = (double)U[2 * k], d = (double)U[2 * k + 1];
    fin = fin && finite_(a) && finite_(d);
    const double t = tan(d);
    const double beta = atan(0.5 * t);
    const double db = 0.5 * (1.0 + t * t) / (1.0 + 0.25 * t * t);
    const double* x = w.X[k];
    const double sb = sin(beta);
    w.wd[k] = dt * (x[3] / kL) * cos(beta) * db;
    w.S[k + 1] = w.S[k] + sb;
    w.X[k + 1][0] = x[0] + dt * x[3] * cos(x[2] + beta);
    w.X[k + 1][1] = x[1] + dt * x[3] * sin(x[2] + beta);
    w.X[k + 1][2] = x[2] + dt * (x[3] / kL) * sb;
    w.X[k + 1][3] = x[3] + dt * a;
  }
  // ---- active set and violation
  double viol = 0.0;
  int n_active = 0;
  for (int i = 0; i < n; ++i) {
    const double u = (double)U[i], lim = (i & 1) ? kDMax : kAMax;
    viol = fmax(viol, fmax(-lim - u, u - lim));
    const bool lo = u - (-lim) <= act_tol, hi = lim - u <= act_tol;
    w.cs[i] = (int8_t)(lo && hi ? 2 : lo ? 1 : hi ? -1 : 0);
    n_active += (int)lo + (int)hi;
    w.pc[i] = 0;
    w.bc[i] = 0;
    w.mu[i] = 0.0;
  }
  int nq = 0;
  for (int k = 1; k <= N; ++k) {
    const double v = w.X[k][3], th = w.X[k][2];
    viol = fmax(viol, fmax(kVMin - v, v - kVMax));
    viol = fmax(viol, fmax(-kThMax - th, th - kThMax));
    const bool act[4] = {v - kVMin <= act_tol, kVMax - v <= act_tol, th + kThMax <= act_tol, kThMax - th <= act_tol};
    for (int c = 0; c < 4; ++c)
      if (act[c]) {
        if (nq < 4 * NMAX) w.node[nq] = (uint16_t)(k << 2 | (c < 2 ? 1 : 0) << 1 | (c & 1));
        ++nq;
      }
  }
  n_active += nq;
  res->n_active = n_active;
  if (nq > defer_above) return false;
  w.nq = nq;
  for (int q = 0; q < nq; ++q) { w.pq[q] = 0; w.nu[q] = 0.0; w.ban[q] = 0; }
  // ---- gradient: one reverse sweep
  double lam[4] = {0.0, 0.0, 0.0, 0.0};                 // adjoint of X[k+1]; X[N] carries no cost
  const bool track = !cfg.literal_no_collision;
  for (int k = N - 1; k >= 0; --k) {
    const double* x = w.X[k];
    const double t = tan((double)U[2 * k + 1]);
    const double beta = atan(0.5 * t);
    const double db = 0.5 * (1.0 + t * t) / (1.0 + 0.25 * t * t);
    const double c = cos(x[2] + beta), sn = sin(x[2] + beta), v = x[3];
    // B^T lam
    w.g[2 * k] = dt * lam[3];
    w.g[2 * k + 1] = (-dt * v * sn * db) * lam[0] + (dt * v * c * db) * lam[1] + (dt * (v / kL) * cos(beta) * db) * lam[2];
    if (k == 0) break;
    // lam_k = l_x(k) + A^T lam_{k+1}
    double lx[4] = {0.0, 0.0, 0.0, 0.0};
    if (track) {
      int j = p.ego_index + k;
      j = j < kNRefRows - 1 ? j : kNRefRows - 1;
      const double rx = cfg.ref[4 * j], ry = cfg.ref[4 * j + 1], rh = cfg.ref[4 * j + 3];
      const double sh = sin(rh), ch = cos(rh);
      const double dx = x[0] - rx, dy = x[1] - ry;
      const double perp = dx * sh - dy * ch, para = dx * ch + dy * sh;
      const double rv = k < p.vr_n ? p.vr_a + double(k) * p.vr_slope : p.vr_b;
      lx[0] = 10.0 * (8.0 * perp * sh + 4.0 * para * ch);
      lx[1] = 10.0 * (-8.0 * perp * ch + 4.0 * para * sh);
      lx[2] = 10.0 * (x[2] - rh);
      lx[3] = 10.0 * 2.0 * p.w_speed * (x[3] - rv);
      if (cfg.w_distance != 0.0)                     // obstacle m as seen by stage k: k steps of its increment
        for (int mo = 0; mo < p.n_obs; ++mo) {
          const float* o = p.obstacles + (long long)mo * 4 * p.obs_stride;
          const double ox = (double)o[0], oy = (double)o[p.obs_stride];
          const double ix = (double)o[2 * p.obs_stride], iy = (double)o[3 * p.obs_stride];
          const double ex = x[0] - (ox + double(k) * ix), ey = x[1] - (oy + double(k) * iy);
          const double dd = hypot(ex, ey);
          const double cc = dd < 1.0 ? 1000.0 : 100.0;
          const double e1 = dd + 1e-6;
          const double coef = cfg.w_distance * (-2.0 * cc / (e1 * e1 * e1)) / fmax(dd, 1e-300);
          lx[0] += coef * ex;
          lx[1] += coef * ey;
        }
      if (cfg.w_collision != 0.0 && p.is_collide) lx[3] += cfg.w_collision * 6000.0 * x[3];
    }
    const double A02 = -dt * v * sn, A03 = dt * c, A12 = dt * v * c, A13 = dt * sn, A23 = dt * sin(beta) / kL;
    const double l2 = lam[2] + A02 * lam[0] + A12 * lam[1];
    const double l3 = lam[3] + A03 * lam[0] + A13 * lam[1] + A23 * lam[2];
    lam[0] = lx[0] + lam[0];
    lam[1] = lx[1] + lam[1];
    lam[2] = lx[2] + l2;
    lam[3] = lx[3] + l3;
  }
  for (int k = 0; k < N; ++k)
    for (int c = 0; c < 2; ++c) {
      const double u = (double)U[2 * k + c];
      double gu = p.w_control * 0.02 * u;
      if (k > 0) gu += p.w_diff * 0.02 * (u - (double)U[2 * (k - 1) + c]);
      if (k < N - 1) gu -= p.w_diff * 0.02 * ((double)U[2 * (k + 1) + c] - u);
      w.g[2 * k + c] += gu;
    }
  double gn = 0.0;
  for (int i = 0; i < n; ++i) gn += w.g[i] * w.g[i];
  gn = sqrt(gn);
  for (int k = 0; k <= N; ++k)
    for (int c = 0; c < 4; ++c) fin = fin && finite_(w.X[k][c]);
  fin = fin && finite_(gn);
  res->grad_norm = gn;
  if (!fin) {                                          // non-finite controls or rollout: no certificate
    const double qnan = nan("");
    res->residual = qnan; res->violation = qnan;
    if (mult) for (int i = 0; i < 4 * N; ++i) mult[i] = (float)qnan;
    return true;
  }
  res->violation = viol;
  // ---- NNLS
  double* r = w.r;
  nnls(w, n, dt, gn, G, cap, r);
  residual_vec(w, n, dt, r);
  double rn = 0.0;
  for (int i = 0; i < n; ++i) rn += r[i] * r[i];
  res->residual = sqrt(rn);
  if (mult) {
    for (int i = 0; i < 4 * N; ++i) mult[i] = 0.f;
    for (int i = 0; i < n; ++i) {
      double lam_i = 0.0;
      if (w.cs[i] == 2) {                                // both bounds: the two columns take g - A nu on this axis
        double v = w.g[i];
        for (int q = 0; q < nq; ++q)
          if (w.nu[q] != 0.0) v -= w.nu[q] * col_entry(w, dt, q, i);
        lam_i = -v;
      } else if (w.cs[i] != 0) {
        lam_i = -double(w.cs[i]) * w.mu[i];
      }
      mult[(i >> 1) * 4 + (i & 1)] = (float)lam_i;
    }
    for (int q = 0; q < nq; ++q) {
      const int e = w.node[q], k = e >> 2, comp = (e >> 1) & 1;
      const double s = (e & 1) ? 1.0 : -1.0;            // reported > 0 at an upper bound
      mult[(k - 1) * 4 + 2 + comp] += (float)(s * w.nu[q]);
    }
  }
  return true;
}

}  // namespace kkt
}  // namespace mpcb
