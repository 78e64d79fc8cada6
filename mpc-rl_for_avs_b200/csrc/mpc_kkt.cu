// mpc_kkt.cu -- k_kkt: the FP64 optimality certificate (KKT residual, bound multipliers) of given controls, one
// problem per thread.  The per-problem functions are in mpc_kkt.cuh (shared with the host harness).
//
// A problem with at most kFastCap active node bounds keeps the normal matrix of its passive node columns in registers /
// local memory (kFastCap^2 doubles).  The others -- a stopped ego has v = 0 active at every node -- are appended to a
// list and certified by k_kkt_deferred, one problem per single-thread block with a (2N)^2-double matrix in shared
// memory (128 KB at N = 64).  Both kernels run the same code, so the result does not depend on which one took a problem.
#include "mpc_internal.h"
#include "mpc_kkt.cuh"

namespace mpcb {

constexpr int kFastCap = 24;

template <int NMAX> __device__ __forceinline__ void kkt_store(const KktLaunch& L, int i, const kkt::Result& r) {
  L.out.residual[i] = (float)r.residual;
  if (L.out.grad_norm) L.out.grad_norm[i] = (float)r.grad_norm;
  if (L.out.violation) L.out.violation[i] = (float)r.violation;
}

template <int NMAX> __device__ __forceinline__ kkt::Config kkt_config(const KktLaunch& L) {
  kkt::Config c;
  c.N = L.N; c.dt = L.dt; c.w_distance = L.w_distance; c.w_collision = L.w_collision;
  c.literal_no_collision = L.literal_no_collision; c.ref = L.ref;
  return c;
}

template <int NMAX> __global__ void __launch_bounds__(128) k_kkt(KktLaunch L) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L.B) return;
  kkt::Work<NMAX> w;
  double G[kFastCap * kFastCap];
  const kkt::Problem p = kkt::load_problem(L.batch, L.B, i, L.M);
  kkt::Result r;
  float* mult = L.out.multipliers ? L.out.multipliers + (size_t)i * L.N * 4 : nullptr;
  const bool done = kkt::certify(kkt_config<NMAX>(L), p, L.U + (size_t)i * L.N * 2, L.act_tol, w, G, kFastCap, kFastCap, &r, mult);
  if (L.out.n_active) L.out.n_active[i] = r.n_active;
  if (!done) {
    L.deferred[atomicAdd(L.n_deferred, 1)] = i;
    return;
  }
  kkt_store<NMAX>(L, i, r);
}

template <int NMAX> __global__ void __launch_bounds__(1) k_kkt_deferred(KktLaunch L) {
  extern __shared__ double G[];                        // (2N)^2
  const int n = *L.n_deferred;
  for (int s = blockIdx.x; s < n; s += gridDim.x) {
    const int i = L.deferred[s];
    kkt::Work<NMAX> w;
    const kkt::Problem p = kkt::load_problem(L.batch, L.B, i, L.M);
    kkt::Result r;
    float* mult = L.out.multipliers ? L.out.multipliers + (size_t)i * L.N * 4 : nullptr;
    kkt::certify(kkt_config<NMAX>(L), p, L.U + (size_t)i * L.N * 2, L.act_tol, w, G, 2 * L.N, 1 << 30, &r, mult);
    kkt_store<NMAX>(L, i, r);
  }
}

template <int NMAX> static cudaError_t launch_kkt_n(const KktLaunch& L, cudaStream_t st) {
  const int tpb = 128;
  k_kkt<NMAX><<<(L.B + tpb - 1) / tpb, tpb, 0, st>>>(L);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  const size_t smem = (size_t)4 * L.N * L.N * sizeof(double);
  e = cudaFuncSetAttribute(k_kkt_deferred<NMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k_kkt_deferred<NMAX><<<L.grid_deferred, 1, smem, st>>>(L);
  return cudaGetLastError();
}

cudaError_t launch_kkt(const KktLaunch& L, cudaStream_t st) {
  return L.N <= 32 ? launch_kkt_n<32>(L, st) : launch_kkt_n<64>(L, st);
}

}  // namespace mpcb
