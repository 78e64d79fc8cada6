// TEST-ONLY host harness for the adaptive start portfolio (tests/test_adaptive_starts.py): the whole host harness
// (hostsim.cpp, included so that its helpers are shared, not copied) plus one entry point that reports every start of
// the portfolio separately.  Built by the test into a temporary directory; the package never loads it.
#include "hostsim.cpp"

extern "C" {

// every start of the portfolio on its own (float, bf16-packed gains: the device arithmetic): cost, status, iterations
// and first control of start st of problem i at [st * B + i] -- the candidate arrays of the product
int hs_solve_starts(const SolverConfig* cfg, const double* ref85x4, const HsBatch* b, int B, int n_starts, float* cost,
                    int* status, int* iters, float* u0) {
  HostTables<float> rt;
  make_ref(ref85x4, rt);
  std::vector<float> buf(slots_per_problem(cfg->N, cfg->M, true));
  for (int st = 0; st < n_starts; ++st)
    for (int i = 0; i < B; ++i) {
      Slots<float, true> sl{buf.data(), 1, cfg->N, cfg->M};
      ProblemScalars<float> p;
      load_problem(*b, B, i, *cfg, p, sl);
      SolveState<float> s;
      solve_one(*cfg, p, rt.tab(), sl, s, nullptr, st);
      const size_t w = (size_t)st * B + i;
      cost[w] = s.J;
      status[w] = s.status;
      iters[w] = s.iter;
      u0[2 * w] = sl.U(0, 0);
      u0[2 * w + 1] = sl.U(0, 1);
    }
  return 0;
}

}  // extern "C"
