// TEST-ONLY host harness for the solution sensitivity (tests/test_sensitivity.py): the host harness of hostsim_kkt.cpp
// (hostsim.cpp plus hs_kkt, included so that its helpers are shared, not copied) plus
//   hs_sens        the per-problem sweep of csrc/mpc_sens.cuh that k_sens runs, compiled for the CPU;
//   hs_sens_dense  an independent dense method on the same inputs, a second reference for the sweep: H and d(grad)/dp
//                  column by column from dual-number passes through sens::lagrangian_grad, the node rows factored by
//                  Householder QR on the free coordinates, SOSC from the Cholesky factorisation of Z^T H Z.
// Built by the test into a temporary directory; the package never loads it.
#include "hostsim_kkt.cpp"
#include "../../mpc-rl_for_avs_b200/csrc/mpc_sens.cuh"

namespace mpcb {
namespace sens {

struct Dual {
  double v, d;
};
inline Dual operator+(Dual a, Dual b) { return {a.v + b.v, a.d + b.d}; }
inline Dual operator-(Dual a, Dual b) { return {a.v - b.v, a.d - b.d}; }
inline Dual operator*(Dual a, Dual b) { return {a.v * b.v, a.d * b.v + a.v * b.d}; }
inline Dual operator/(Dual a, Dual b) { return {a.v / b.v, (a.d * b.v - a.v * b.d) / (b.v * b.v)}; }
inline Dual operator+(Dual a, double b) { return {a.v + b, a.d}; }
inline Dual operator+(double a, Dual b) { return {a + b.v, b.d}; }
inline Dual operator-(Dual a, double b) { return {a.v - b, a.d}; }
inline Dual operator-(double a, Dual b) { return {a - b.v, -b.d}; }
inline Dual operator*(Dual a, double b) { return {a.v * b, a.d * b}; }
inline Dual operator*(double a, Dual b) { return {a * b.v, a * b.d}; }
inline Dual operator/(Dual a, double b) { return {a.v / b, a.d / b}; }
inline Dual operator/(double a, Dual b) { return {a / b.v, -a * b.d / (b.v * b.v)}; }
inline double val(Dual a) { return a.v; }
inline Dual s_sin(Dual a) { return {sin(a.v), cos(a.v) * a.d}; }
inline Dual s_cos(Dual a) { return {cos(a.v), -sin(a.v) * a.d}; }
inline Dual s_tan(Dual a) { const double t = tan(a.v); return {t, (1.0 + t * t) * a.d}; }
inline Dual s_atan(Dual a) { return {atan(a.v), a.d / (1.0 + a.v * a.v)}; }
inline Dual s_hypot(Dual a, Dual b) {
  const double h = hypot(a.v, b.v);
  return {h, h > 0.0 ? (a.v * a.d + b.v * b.d) / h : 0.0};
}
inline Dual s_floor(Dual a, double lo) { return a.v > lo ? a : Dual{lo, 0.0}; }


// caller-provided dense storage: element e at base[e * stride]
struct Scratch {
  double* base;
  long long stride;
  double& operator[](long long e) const { return base[e * stride]; }
};
inline long long scratch_doubles(int N) { return 8LL * N * N + 8LL * N; }

// Per-problem work arrays for horizons up to NMAX.
template <int NMAX> struct DenseWork {
  double X[NMAX + 1][4];
  Dual Xt[NMAX + 1][4];
  double U[2 * NMAX], g[2 * NMAX], r[2 * NMAX], beta[2 * NMAX], rdiag[2 * NMAX], nu[2 * NMAX];
  Dual Ut[2 * NMAX], gt[2 * NMAX];
  double wth[NMAX + 1], wv[NMAX + 1];
  double wd[NMAX], S[NMAX + 1];
  int8_t cs[2 * NMAX];          // control coordinate: 0 free, +1 lower bound active, -1 upper, 2 both
  int16_t F[2 * NMAX];          // free coordinates
  uint16_t node[2 * NMAX];      // active node bound q: k << 2 | comp << 1 | upper   (comp 0 = theta, 1 = v)
};

// signed entry of node row e at coordinate i (+ row at a lower bound, - at an upper bound)
template <int NMAX> inline double node_entry(const DenseWork<NMAX>& w, double dt, int e, int i) {
  const int k = e >> 2, comp = (e >> 1) & 1, j = i >> 1;
  double r = 0.0;
  if (j < k) r = comp == 1 ? ((i & 1) ? 0.0 : dt) : ((i & 1) ? w.wd[j] : dt * dt / kkt::kL * (w.S[k] - w.S[j + 1]));
  return (e & 1) ? -r : r;
}

// jac: [2][4] dU_0/dp (NaN unless the flags allow it).  mult (may be null): [N][4] in the layout of mpc_kkt's
// multipliers (> 0 at an upper bound, < 0 at a lower bound, 0 when inactive), written when the multipliers exist.
// Returns the flag bits.
template <int NMAX>
int sensitivity_dense(const Config& cfg, const Problem& p, const float* Uf, double act_tol, double stat_tol, DenseWork<NMAX>& w,
                       Scratch s, double* jac, float* mult) {
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
  // ---- active set; closed-form node rows (theta, v do not depend on x, y)
  int nF = 0;
  bool dup = false;
  for (int i = 0; i < n; ++i) {
    const double u = w.U[i], lim = (i & 1) ? kkt::kDMax : kkt::kAMax;
    const bool lo = u + lim <= act_tol, hi = lim - u <= act_tol;
    w.cs[i] = (int8_t)(lo && hi ? 2 : lo ? 1 : hi ? -1 : 0);
    dup = dup || (lo && hi);
    if (!lo && !hi) w.F[nF++] = (int16_t)i;
  }
  w.S[0] = 0.0;
  for (int k = 0; k < N; ++k) {
    const double t = tan(w.U[2 * k + 1]);
    const double beta = atan(0.5 * t);
    const double db = 0.5 * (1.0 + t * t) / (1.0 + 0.25 * t * t);
    w.wd[k] = dt * (w.X[k][3] / kkt::kL) * cos(beta) * db;
    w.S[k + 1] = w.S[k] + sin(beta);
  }
  int mq = 0;
  for (int k = 1; k <= N; ++k) {
    const double v = w.X[k][3], th = w.X[k][2];
    const bool act[4] = {v - kkt::kVMin <= act_tol, kkt::kVMax - v <= act_tol, th + kkt::kThMax <= act_tol,
                         kkt::kThMax - th <= act_tol};
    for (int c = 0; c < 4; ++c)
      if (act[c]) {
        if (mq >= nF) dup = true;                         // more node rows than free coordinates
        else w.node[mq++] = (uint16_t)(k << 2 | (c < 2 ? 1 : 0) << 1 | (c & 1));
      }
  }
  if (dup) return kDegenerate;
  // ---- Householder QR of A_F^T: row q of A at s[n*n + q*n + f]; reflector j kept in row j from column j on, R above
  const long long oA = (long long)n * n, oG = 2LL * n * n;
  for (int q = 0; q < mq; ++q)
    for (int f = 0; f < nF; ++f) s[oA + q * n + f] = node_entry(w, dt, w.node[q], w.F[f]);
  for (int j = 0; j < mq; ++j) {
    double full = 0.0;
    for (int i = 0; i < n; ++i) { const double e = node_entry(w, dt, w.node[j], i); full += e * e; }
    double sig = 0.0;
    for (int f = j; f < nF; ++f) sig += s[oA + j * n + f] * s[oA + j * n + f];
    sig = sqrt(sig);
    if (!(sig > kLicqTol * sqrt(full))) return kDegenerate;
    const double x0 = s[oA + j * n + j];
    const double alpha = x0 > 0.0 ? -sig : sig;
    s[oA + j * n + j] = x0 - alpha;
    double vv = 0.0;
    for (int f = j; f < nF; ++f) vv += s[oA + j * n + f] * s[oA + j * n + f];
    w.beta[j] = 2.0 / vv;
    w.rdiag[j] = alpha;
    for (int q = j + 1; q < mq; ++q) {
      double d = 0.0;
      for (int f = j; f < nF; ++f) d += s[oA + j * n + f] * s[oA + q * n + f];
      d *= w.beta[j];
      for (int f = j; f < nF; ++f) s[oA + q * n + f] -= d * s[oA + j * n + f];
    }
  }
  // x <- Q^T x (forward) or Q x (backward) for a vector of nF entries x(f)
  auto apply_q = [&](auto x, bool transpose) {
    for (int jj = 0; jj < mq; ++jj) {
      const int j = transpose ? jj : mq - 1 - jj;
      double d = 0.0;
      for (int f = j; f < nF; ++f) d += s[oA + j * n + f] * x(f);
      d *= w.beta[j];
      for (int f = j; f < nF; ++f) x(f) -= d * s[oA + j * n + f];
    }
  };
  auto rvec = [&](int f) -> double& { return w.r[f]; };
  auto strided = [&](long long off, long long step) { return [=](int f) -> double& { return s[off + f * step]; }; };
  // ---- multipliers and stationarity
  for (int f = 0; f < nF; ++f) w.r[f] = w.g[w.F[f]];
  apply_q(rvec, true);
  double res = 0.0;
  for (int f = mq; f < nF; ++f) res += w.r[f] * w.r[f];
  res = sqrt(res);
  for (int j = mq - 1; j >= 0; --j) {
    double v = w.r[j];
    for (int q = j + 1; q < mq; ++q) v -= s[oA + q * n + j] * w.nu[q];
    w.nu[j] = v / w.rdiag[j];
  }
  const double tau = stat_tol * (1.0 + fabs(J));
  int flags = res > tau ? kNotStationary : 0;
  double mmin = 1e300;
  if (mult) for (int i = 0; i < 4 * N; ++i) mult[i] = 0.f;
  for (int i = 0; i < n; ++i) {
    if (w.cs[i] == 0) continue;
    double v = w.g[i];
    for (int q = 0; q < mq; ++q) v -= w.nu[q] * node_entry(w, dt, w.node[q], i);
    const double mu = double(w.cs[i]) * v;               // row +e_i at a lower bound, -e_i at an upper one
    mmin = fmin(mmin, mu);
    if (mult) mult[(i >> 1) * 4 + (i & 1)] = (float)(-double(w.cs[i]) * mu);
  }
  for (int q = 0; q < mq; ++q) {
    const int e = w.node[q], k = e >> 2, comp = (e >> 1) & 1;
    const double sg = (e & 1) ? -1.0 : 1.0;
    mmin = fmin(mmin, w.nu[q]);
    if (mult) mult[(k - 1) * 4 + 2 + comp] = (float)(-sg * w.nu[q]);
    (comp ? w.wv : w.wth)[k] -= sg * w.nu[q];            // L = J - sum nu_q c_q, c_q = sg (x_k[comp] - bound)
  }
  const double tw = kWeakTol * (1.0 + fabs(J));
  if (mmin < -tw) flags |= kNotStationary;
  else if (mmin <= tw) flags |= kWeaklyActive;
  // ---- H_FF (Lagrangian) and G_F by forward-mode passes through the gradient
  Dual pt[4];
  for (int f = 0; f <= nF + 4; ++f) {             // nF columns of H, then 4 of G
    if (f == nF) continue;
    for (int i = 0; i < n; ++i) w.Ut[i] = Dual{w.U[i], 0.0};
    for (int c = 0; c < 4; ++c) pt[c] = Dual{prm[c], 0.0};
    if (f < nF) w.Ut[w.F[f]].d = 1.0;
    else pt[f - nF - 1].d = 1.0;
    lagrangian_grad<Dual>(cfg, p, w.Ut, pt, w.wth, w.wv, w.Xt, w.gt);
    for (int a = 0; a < nF; ++a) {
      if (f < nF) s[(long long)a * n + f] = w.gt[w.F[a]].d;
      else s[oG + a * 4 + (f - nF - 1)] = w.gt[w.F[a]].d;
    }
  }
  double hmax = 1.0;
  for (int a = 0; a < nF; ++a) {
    hmax = fmax(hmax, fabs(s[(long long)a * n + a]));
    for (int b = 0; b < a; ++b) {
      const double m = 0.5 * (s[(long long)a * n + b] + s[(long long)b * n + a]);
      s[(long long)a * n + b] = m;
      s[(long long)b * n + a] = m;
    }
  }
  for (int f = 0; f < nF; ++f) apply_q(strided(f, n), true);           // Q^T H Q: columns, then rows
  for (int a = 0; a < nF; ++a) apply_q(strided((long long)a * n, 1), true);
  for (int c = 0; c < 4; ++c) apply_q(strided(oG + c, 4), true);
  // ---- Cholesky of Z^T H Z (the trailing block), in its lower triangle
  for (int a = mq; a < nF; ++a) {
    double d = s[(long long)a * n + a];
    for (int c = mq; c < a; ++c) d -= s[(long long)a * n + c] * s[(long long)a * n + c];
    if (!(d > kSoscTol * hmax)) { flags |= kNotSosc; break; }
    d = sqrt(d);
    s[(long long)a * n + a] = d;
    for (int b = a + 1; b < nF; ++b) {
      double v = s[(long long)b * n + a];
      for (int c = mq; c < a; ++c) v -= s[(long long)b * n + c] * s[(long long)a * n + c];
      s[(long long)b * n + a] = v / d;
    }
  }
  if (flags & (kNotStationary | kNotSosc)) return flags;
  // ---- dU_F = Q [0; y], (Z^T H Z) y = -Z^T G, per parameter column
  for (int c = 0; c < 4; ++c) {
    for (int f = 0; f < mq; ++f) w.r[f] = 0.0;
    for (int a = mq; a < nF; ++a) {                      // L z = -Z^T G
      double v = -s[oG + a * 4 + c];
      for (int b = mq; b < a; ++b) v -= s[(long long)a * n + b] * w.r[b];
      w.r[a] = v / s[(long long)a * n + a];
    }
    for (int a = nF - 1; a >= mq; --a) {                 // L^T y = z
      double v = w.r[a];
      for (int b = a + 1; b < nF; ++b) v -= s[(long long)b * n + a] * w.r[b];
      w.r[a] = v / s[(long long)a * n + a];
    }
    apply_q(rvec, false);
    jac[c] = jac[4 + c] = 0.0;                           // a pinned u_0 coordinate does not move
    for (int f = 0; f < nF && w.F[f] < 2; ++f) jac[w.F[f] * 4 + c] = w.r[f];
  }
  return flags;
}

}  // namespace sens
}  // namespace mpcb

extern "C" {

static kkt::Config sens_config(const SolverConfig* cfg, const double* ref85x4) {
  kkt::Config kc;
  kc.N = cfg->N;
  kc.dt = 1.0 / (double)(long long)(1.0 / (double)cfg->dt + 0.5);
  kc.w_distance = cfg->w_distance; kc.w_collision = cfg->w_collision;
  kc.literal_no_collision = cfg->literal_no_collision;
  kc.ref = ref85x4;
  return kc;
}

// dU_0/dp of the controls U [B][N][2]: jac [B][2][4] (FP64), flags [B], multipliers [B][N][4] (may be null; the layout
// of hs_kkt's).  dt is the double 1 / policy_frequency of cfg->dt, the path table ref85x4 the one of that dt.
int hs_sens(const SolverConfig* cfg, const double* ref85x4, const HsBatch* b, int B, const float* U, double act_tol,
            double stat_tol, double* jac, int* flags, float* mult) {
  if (cfg->N > 64) return -1;
  const kkt::Config kc = sens_config(cfg, ref85x4);
  const int N = cfg->N;
  std::vector<sens::Sweep<64>> w(1);
  for (int i = 0; i < B; ++i) {
    const kkt::Problem p = kkt::load_problem(*b, B, i, cfg->M);
    flags[i] = sens::sensitivity(kc, p, U + (size_t)i * N * 2, act_tol, stat_tol, w[0], jac + (size_t)i * 8,
                                 mult ? mult + (size_t)i * N * 4 : nullptr);
  }
  return 0;
}

// the same quantity by the dense method
int hs_sens_dense(const SolverConfig* cfg, const double* ref85x4, const HsBatch* b, int B, const float* U, double act_tol,
                  double stat_tol, double* jac, int* flags, float* mult) {
  if (cfg->N > 64) return -1;
  const kkt::Config kc = sens_config(cfg, ref85x4);
  const int N = cfg->N;
  std::vector<sens::DenseWork<64>> w(1);
  // stride 3, as if interleaved with two other problems' scratch
  std::vector<double> scratch(3 * sens::scratch_doubles(N));
  for (int i = 0; i < B; ++i) {
    const kkt::Problem p = kkt::load_problem(*b, B, i, cfg->M);
    flags[i] = sens::sensitivity_dense(kc, p, U + (size_t)i * N * 2, act_tol, stat_tol, w[0],
                                       sens::Scratch{scratch.data(), 3}, jac + (size_t)i * 8,
                                       mult ? mult + (size_t)i * N * 4 : nullptr);
  }
  return 0;
}

}  // extern "C"
