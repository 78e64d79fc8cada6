// TEST-ONLY host harness for the optimality certificate (tests/test_kkt.py): the whole host harness (hostsim.cpp,
// included so that its helpers are shared, not copied) plus hs_kkt, the per-problem functions of csrc/mpc_kkt.cuh that
// k_kkt runs, compiled for the CPU.  Built by the test into a temporary directory; the package never loads it.
#include "hostsim.cpp"
#include "../../mpc-rl_for_avs_b200/csrc/mpc_kkt.cuh"

extern "C" {

// Certificate of the controls U [B][N][2] at act_tol, in FP64: residual, |g|, violation, active-row count, multipliers
// [B][N][4] and the gradient g [B][2N] (any output but residual may be null).  dt is the double 1 / policy_frequency
// of cfg->dt, the path table ref85x4 the one of that dt.
int hs_kkt(const SolverConfig* cfg, const double* ref85x4, const HsBatch* b, int B, const float* U, double act_tol,
           double* residual, double* grad_norm, double* violation, int* n_active, float* mult, double* g_out) {
  if (cfg->N > 64) return -1;
  kkt::Config kc;
  kc.N = cfg->N;
  kc.dt = 1.0 / (double)(long long)(1.0 / (double)cfg->dt + 0.5);
  kc.w_distance = cfg->w_distance; kc.w_collision = cfg->w_collision;
  kc.literal_no_collision = cfg->literal_no_collision;
  kc.ref = ref85x4;
  const int N = cfg->N;
  std::vector<kkt::Work<64>> w(1);
  std::vector<double> G(4 * N * N);
  std::vector<float> m(4 * N);
  for (int i = 0; i < B; ++i) {
    const kkt::Problem p = kkt::load_problem(*b, B, i, cfg->M);
    kkt::Result r;
    kkt::certify(kc, p, U + (size_t)i * N * 2, act_tol, w[0], G.data(), 2 * N, 1 << 30, &r, m.data());
    residual[i] = r.residual;
    if (grad_norm) grad_norm[i] = r.grad_norm;
    if (violation) violation[i] = r.violation;
    if (n_active) n_active[i] = r.n_active;
    if (mult) memcpy(mult + (size_t)i * N * 4, m.data(), sizeof(float) * 4 * N);
    if (g_out) memcpy(g_out + (size_t)i * N * 2, w[0].g, sizeof(double) * 2 * N);
  }
  return 0;
}

}  // extern "C"
