// TEST-ONLY host harness.  Compiles the kernel's per-problem device functions
// (mpc-rl_for_avs_b200/csrc/mpc_core.cuh) with g++ so that the solver LOGIC can be exercised
// against the oracle on machines without a GPU (`pytest -m "not gpu"`), in float (the
// device arithmetic) and in double (to separate algorithmic from rounding effects).
// It is NOT part of the product: the package never loads this library and has no CPU path.
#include <cstring>
#include <vector>

#include "../../mpc-rl_for_avs_b200/csrc/mpc_core.cuh"
#include "../../mpc-rl_for_avs_b200/csrc/ref_path.h"

using namespace mpcb;

struct HsBatch {               // same SoA layout as MpcProblemBatch (include/mpc_b200.h), host memory
  const float* s0;             // [4][B]
  const int* ego_index;        // [B]
  const float* w_speed;        // [B]
  const float* w_control;      // [B]
  const float* w_diff;         // [B]
  const float* vr_a;           // [B]
  const float* vr_slope;       // [B]
  const float* vr_b;           // [B]
  const int* vr_n;             // [B]
  const unsigned char* is_collide;  // [B]
  const int* n_obs;            // [B]
  const float* obstacles;      // [M][4][B]
};

template <typename T, typename SL>
static void load_problem(const HsBatch& b, int B, int i, const SolverConfig& cfg, ProblemScalars<T>& p, SL& sl) {
  p.ego_index = b.ego_index[i];
  p.n_obs = b.n_obs ? b.n_obs[i] : 0;
  if (p.n_obs > cfg.M) p.n_obs = cfg.M;
  p.is_collide = b.is_collide ? b.is_collide[i] : 0;
  p.w_speed = T(b.w_speed[i]);
  p.w_control = T(b.w_control[i]);
  p.w_diff = T(b.w_diff[i]);
  p.vr_a = T(b.vr_a[i]); p.vr_slope = T(b.vr_slope[i]); p.vr_b = T(b.vr_b[i]); p.vr_n = b.vr_n[i];
  p.x0 = (double)b.s0[i];
  p.y0 = (double)b.s0[(size_t)B + i];
  sl.X(0, 0) = T(0); sl.X(0, 1) = T(0);
  sl.X(0, 2) = T(b.s0[(size_t)2 * B + i]);
  sl.X(0, 3) = T(b.s0[(size_t)3 * B + i]);
  for (int m = 0; m < cfg.M; ++m) {
    if (b.obstacles) {
      sl.O(m, 0) = T((double)b.obstacles[((size_t)m * 4 + 0) * B + i] - p.x0);
      sl.O(m, 1) = T((double)b.obstacles[((size_t)m * 4 + 1) * B + i] - p.y0);
      sl.O(m, 2) = T(b.obstacles[((size_t)m * 4 + 2) * B + i]);
      sl.O(m, 3) = T(b.obstacles[((size_t)m * 4 + 3) * B + i]);
    } else {
      for (int c = 0; c < 4; ++c) sl.O(m, c) = T(0);
    }
  }
}

template <typename T> struct HostTables {
  std::vector<T> hsc;
  std::vector<double> xy;
  RefTab<T> tab() const { return RefTab<T>{hsc.data(), xy.data()}; }
};
template <typename T>
static void make_ref(const double* ref85x4, HostTables<T>& out) {
  out.hsc.resize(kNRef * kRefStride);
  out.xy.resize(kNRef * 2);
  for (int j = 0; j < kNRef; ++j) {
    out.xy[2 * j] = ref85x4[j * 4 + 0];
    out.xy[2 * j + 1] = ref85x4[j * 4 + 1];
    out.hsc[j * kRefStride + 0] = T(ref85x4[j * 4 + 3]);
    out.hsc[j * kRefStride + 1] = T(sin(ref85x4[j * 4 + 3]));
    out.hsc[j * kRefStride + 2] = T(cos(ref85x4[j * 4 + 3]));
  }
}

template <typename T, bool kPack>
static void run_solve(const SolverConfig& cfg, const double* ref, const HsBatch& b, int B, float* actions,
                      int* status, int* iters, float* cost, float* U_out, int* outer_out, const float* u_init = nullptr,
                      int n_starts = 1) {
  HostTables<T> rt;
  make_ref(ref, rt);
  std::vector<T> buf(slots_per_problem(cfg.N, cfg.M, kPack));
  for (int i = 0; i < B; ++i) {
    // start portfolio as in the product (k_solve + k_select): every start is an independent solve, the lowest
    // FP objective wins (ties: lowest start), `iters` is the total over the starts
    float best = 0.f;
    int it_total = 0;
    for (int st = 0; st < n_starts; ++st) {
      Slots<T, kPack> sl{buf.data(), 1, cfg.N, cfg.M};
      ProblemScalars<T> p;
      load_problem(b, B, i, cfg, p, sl);
      SolveState<T> s;
      solve_one(cfg, p, rt.tab(), sl, s, u_init ? u_init + (size_t)i * cfg.N * 2 : nullptr, st);
      it_total += s.iter;
      const float J = float(s.J);
      if (st > 0 && !(J < best) && !(!(best == best) && J == J)) continue;
      best = J;
      actions[2 * i] = float(sl.U(0, 0));
      actions[2 * i + 1] = float(sl.U(0, 1));
      status[i] = s.status;
      if (outer_out) outer_out[i] = s.fails;
      cost[i] = J;
      if (U_out)
        for (int k = 0; k < cfg.N; ++k) { U_out[((size_t)i * cfg.N + k) * 2] = float(sl.U(k, 0)); U_out[((size_t)i * cfg.N + k) * 2 + 1] = float(sl.U(k, 1)); }
    }
    iters[i] = it_total;
  }
}

template <typename T>
static void run_rollout_cost(const SolverConfig& cfg, const double* ref, const HsBatch& b, int B, const float* U,
                             const float* ref_v /*[N][B] or null*/, float* X_out, float* cost6, float* total) {
  HostTables<T> rt;
  make_ref(ref, rt);
  std::vector<T> buf(slots_per_problem(cfg.N, cfg.M, false));
  for (int i = 0; i < B; ++i) {
    Slots<T, false> sl{buf.data(), 1, cfg.N, cfg.M};
    ProblemScalars<T> p;
    load_problem(b, B, i, cfg, p, sl);
    for (int k = 0; k < cfg.N; ++k) {
      sl.U(k, 0) = T(U[((size_t)i * cfg.N + k) * 2]);
      sl.U(k, 1) = T(U[((size_t)i * cfg.N + k) * 2 + 1]);
    }
    (void)ref_v;
    T comp[6] = {0, 0, 0, 0, 0, 0};
    T J = rollout_nominal(cfg, p, rt.tab(), sl, comp);
    comp[2] = final_state_component(cfg, p, rt.tab(), sl);
    for (int c = 0; c < 6; ++c) cost6[(size_t)i * 6 + c] = float(comp[c]);
    total[i] = float(J);
    for (int k = 0; k <= cfg.N; ++k) {
      float* xo = X_out + ((size_t)i * (cfg.N + 1) + k) * 4;
      xo[0] = float(p.x0 + double(sl.X(k, 0))); xo[1] = float(p.y0 + double(sl.X(k, 1)));
      xo[2] = float(sl.X(k, 2)); xo[3] = float(sl.X(k, 3));
    }
  }
}

extern "C" {

int hs_solve(const SolverConfig* cfg, const double* ref85x4, const HsBatch* b, int B, int use_double, float* actions,
             int* status, int* iters, float* cost, float* U_out, int* outer_out) {
  // use_double: 1 = double; 0 = float with bf16-packed gains (exactly the device arithmetic);
  // 2 = float with full-precision gains (to isolate the effect of the packing)
  if (use_double == 1) run_solve<double, false>(*cfg, ref85x4, *b, B, actions, status, iters, cost, U_out, outer_out);
  else if (use_double == 2) run_solve<float, false>(*cfg, ref85x4, *b, B, actions, status, iters, cost, U_out, outer_out);
  else run_solve<float, true>(*cfg, ref85x4, *b, B, actions, status, iters, cost, U_out, outer_out);
  return 0;
}

// opt-in warm start (the product's mpc_set_warm_start): u_init [B][N][2]
int hs_solve_init(const SolverConfig* cfg, const double* ref85x4, const HsBatch* b, int B, int use_double, const float* u_init,
                  int n_starts, float* actions, int* status, int* iters, float* cost, float* U_out) {
  if (use_double == 1) run_solve<double, false>(*cfg, ref85x4, *b, B, actions, status, iters, cost, U_out, nullptr, u_init, n_starts);
  else run_solve<float, true>(*cfg, ref85x4, *b, B, actions, status, iters, cost, U_out, nullptr, u_init, n_starts);
  return 0;
}

int hs_rollout_cost(const SolverConfig* cfg, const double* ref85x4, const HsBatch* b, int B, int use_double,
                    const float* U, float* X_out, float* cost6, float* total) {
  if (use_double) run_rollout_cost<double>(*cfg, ref85x4, *b, B, U, nullptr, X_out, cost6, total);
  else run_rollout_cost<float>(*cfg, ref85x4, *b, B, U, nullptr, X_out, cost6, total);
  return 0;
}

int hs_sizeof_config() { return (int)sizeof(SolverConfig); }

// the library's path-table generator (what mpc_create builds from the handle's dt): out [85][4]
void hs_reference_path(double dt, double* out) { build_reference_path(dt, reinterpret_cast<double (*)[4]>(out)); }
}

// debugging aid: model-vs-actual merit along the DDP step from a given nominal U
extern "C" int hs_linesearch_probe(const SolverConfig* cfg, const double* ref, const HsBatch* b, int B, int i, const float* U,
                                   double mu, int n_alpha, const double* alphas, double* out /* J0,d1,d2,J(a)... */) {
  HostTables<double> rt;
  make_ref(ref, rt);
  std::vector<double> buf(slots_per_problem(cfg->N, cfg->M, false));
  Slots<double, false> sl{buf.data(), 1, cfg->N, cfg->M};
  ProblemScalars<double> p;
  load_problem(*b, B, i, *cfg, p, sl);
  for (int k = 0; k < cfg->N; ++k) { sl.U(k, 0) = U[2 * k]; sl.U(k, 1) = U[2 * k + 1]; }
  out[0] = rollout_nominal(*cfg, p, rt.tab(), sl, (double*)nullptr);
  backward_pass(*cfg, p, rt.tab(), sl, mu, 1.0, &out[1], &out[2]);
  for (int a = 0; a < n_alpha; ++a) { double md, al = alphas[a]; forward_pass<double, 1>(*cfg, p, rt.tab(), sl, &al, false, true, false, &out[3 + a], &md); }
  for (int k = 0; k < cfg->N; ++k) { double f0, f1, Kr[12]; sl.load_gains(k, f0, f1, Kr); out[3 + n_alpha + 2 * k] = f0; out[3 + n_alpha + 2 * k + 1] = f1; }
  return 0;
}
