// mpc_sens.cu -- k_sens: the FP64 sensitivity dU_0/dp of given controls (mpc_sensitivity), one problem per thread.  The
// per-problem sweep is in mpc_sens.cuh (shared with the host harness); its state is O(N) per thread.
// Compiled with -fmad=false so that the results stay within rounding of the host build's.
#include "mpc_internal.h"
#include "mpc_sens.cuh"

namespace mpcb {

template <int NMAX> __global__ void __launch_bounds__(128) k_sens(SensLaunch L) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L.B) return;
  kkt::Config c;
  c.N = L.N; c.dt = L.dt; c.w_distance = L.w_distance; c.w_collision = L.w_collision;
  c.literal_no_collision = L.literal_no_collision; c.ref = L.ref;
  sens::Sweep<NMAX> w;
  const kkt::Problem p = kkt::load_problem(L.batch, L.B, i, L.M);
  double jac[8];
  L.out.flags[i] = sens::sensitivity(c, p, L.U + (size_t)i * L.N * 2, L.act_tol, L.stat_tol, w, jac, nullptr);
  for (int e = 0; e < 8; ++e) L.out.jac[(size_t)i * 8 + e] = (float)jac[e];
}

cudaError_t launch_sens(const SensLaunch& L, cudaStream_t st) {
  const int tpb = 128, grid = (L.B + tpb - 1) / tpb;
  if (L.N <= 32) k_sens<32><<<grid, tpb, 0, st>>>(L);
  else k_sens<64><<<grid, tpb, 0, st>>>(L);
  return cudaGetLastError();
}

}  // namespace mpcb
