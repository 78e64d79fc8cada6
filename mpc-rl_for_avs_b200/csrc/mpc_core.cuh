// mpc_core.cuh -- per-problem numerics of the batched nonlinear MPC (sm_100a).
//
// One problem lives in ONE thread: horizon arrays (controls, nominal states, feedback
// gains, multipliers, obstacle tracks) sit in a strided shared-memory "slot file"
// (slot * blockDim + tid -> conflict-free), the 6x6 value-function block sits in
// registers.  The functions are templated on the scalar type and on nothing
// CUDA-specific so the test-only host harness (tests/hostsim) can instantiate them
// with double/float on the CPU; the product library instantiates float on device only.
//
// What is computed (reference: SaeedRahmani/MPC-RL_for_AVs, cited as file:line):
//   dynamics   kinematic bicycle + explicit Euler        agents/pure_mpc.py:220-228,252-254
//   tracking   4 perp^2 + 2 para^2 + w_v dv^2 + .5 dth^2 agents/pure_mpc.py:128-156
//   control    0.01 (a^2 + delta^2); input diff          agents/pure_mpc.py:161-165
//   distance   (1000|100)/(d+1e-6)^2 vs moving obstacles agents/archive/pure_mpc.py:189-206
//   collision  3000 v^2 when is_collide                  agents/pure_mpc.py:179-183
//   objective  10 state + w_c control + w_d diff (+...)  agents/pure_mpc.py:204-212
//   bounds     a, delta, v, theta                        agents/pure_mpc.py:272-280
// The NLP that the reference hands to CasADi/IPOPT (pure_mpc.py:285-300) is solved here
// in single-shooting form by a control-limited second-order DDP (exact dynamics Hessian,
// per-stage 2x2 box QP, saddle-free eigenvalue modification).  The v / theta node bounds
// have relative degree one under Euler, so they are enforced exactly as state-dependent
// control boxes (see control_box).  The previous control is carried as two extra state
// coordinates so the input-difference cost stays stage-wise (state z = x,y,th,v,a-,d-).
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define MPC_HD __host__ __device__ __forceinline__
#else
#define MPC_HD inline
#endif

// obstacle loops: the per-obstacle chain (LDS -> FMA -> MUFU.RSQ -> FMA) is long and serial; unrolling
// overlaps several obstacles' chains (the kernel is latency bound)
#ifndef MPC_OBS_UNROLL
#define MPC_OBS_UNROLL 4
#endif
#ifndef MPC_LOOKAHEAD
#define MPC_LOOKAHEAD 1         // look-ahead bound in the backward sweep (see backward_pass)
#endif
#define MPC_STR2(x) #x
#define MPC_STR(x) MPC_STR2(x)
#define MPC_PRAGMA_UNROLL_OBS _Pragma(MPC_STR(unroll MPC_OBS_UNROLL))

namespace mpcb {

constexpr int kNRef = 85;          // agents/base_agent.py:127-152 (40 + 20 + 25 rows)
constexpr int kRefStride = 3;      // heading, sin h, cos h (float table); x, y live in an FP64 table
constexpr int kMaxObstacles = 16;

template <typename T> struct Lim {
  static MPC_HD T a_max() { return T(5); }                        // pure_mpc.py:279-280
  static MPC_HD T d_max() { return T(1.0471975511965976); }       // pi/3
  static MPC_HD T v_min() { return T(0); }                        // pure_mpc.py:273-274
  static MPC_HD T v_max() { return T(30); }
  static MPC_HD T th_max() { return T(3.14159265358979323846); }  // +-pi
};

// ---- scalar math dispatch ---------------------------------------------------------
#if defined(__CUDACC__)
#define MPC_NOINLINE __host__ __device__ __noinline__
#else
#define MPC_NOINLINE __attribute__((noinline))
#endif

// sin and cos for |x| <= ~4 rad (headings live in [-pi, pi] plus one Euler step, steering in
// [-pi/3, pi/3]): one Cody-Waite step to |r| <= pi/4 and the Cephes single-precision kernels
// (~1 ulp).  The general-purpose sincosf drags a Payne-Hanek slow path into every call site and
// the kernel is instruction-cache bound, so the lean version is worth ~10% of the code size.
MPC_HD void sincos_(float x, float* s, float* c) {
  const float kf = rintf(x * 0.636619772367581343f);           // nearest multiple of pi/2
  float r = fmaf(-kf, 1.57079601287841796875f, x);             // pi/2 split hi / lo
  r = fmaf(-kf, 3.1391647326017846353352069854736e-7f, r);
  const float z = r * r;
  const float sp = r + r * z * fmaf(z, fmaf(z, -1.9515295891e-4f, 8.3321608736e-3f), -1.6666654611e-1f);
  const float cp = fmaf(z * z, fmaf(z, fmaf(z, 2.443315711809948e-5f, -1.388731625493765e-3f), 4.166664568298827e-2f),
                        fmaf(-0.5f, z, 1.0f));
  const int q = (int)kf & 3;
  const float ss = (q & 1) ? cp : sp, cc = (q & 1) ? sp : cp;
  *s = (q & 2) ? -ss : ss;
  *c = ((q + 1) & 2) ? -cc : cc;
}
MPC_HD void sincos_(double x, double* s, double* c) { *s = sin(x); *c = cos(x); }
// 1/x and a/b: the device path uses the 2-ulp hardware approximations (MUFU + no slow path);
// every quantity they touch is either a search direction or carries 1e-5 relative tolerance
MPC_HD float rcp_(float x) {
#if defined(__CUDA_ARCH__)
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));     // one MUFU.RCP, no range fix-up code
  return r;
#else
  return 1.0f / x;
#endif
}
MPC_HD double rcp_(double x) { return 1.0 / x; }
MPC_HD float rsqrt_(float x) {
#if defined(__CUDA_ARCH__)
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));   // one MUFU.RSQ
  return r;
#else
  return 1.0f / sqrtf(x);
#endif
}
MPC_HD double rsqrt_(double x) { return 1.0 / sqrt(x); }
MPC_HD float sqrt_(float x) { return sqrtf(x); }
MPC_HD double sqrt_(double x) { return sqrt(x); }
MPC_HD float abs_(float x) { return fabsf(x); }
MPC_HD double abs_(double x) { return fabs(x); }
// ---- two lanes of one expression: the line search's two candidates (forward_pass<T, 2>) -------------------
// On the device a float pair is evaluated by one packed FP32 instruction per operation (sm_100 FADD2 / FMUL2 / FFMA2,
// round-to-nearest, no flush to zero): per lane it is the same IEEE operation as the scalar code.  The packed forms are
// never contracted by the compiler, so an expression is written with fma2 exactly where the scalar code's multiply-add
// was fused, and with mul2 + add2 where it was not.  The host (and T = double) evaluates two plain scalar expressions,
// as it compiles the scalar code: no std::fma.
template <typename T> struct Pair { T a, b; };
template <typename T> MPC_HD Pair<T> splat(T x) { return {x, x}; }
template <typename T> MPC_HD Pair<T> add2(Pair<T> x, Pair<T> y) { return {x.a + y.a, x.b + y.b}; }
template <typename T> MPC_HD Pair<T> mul2(Pair<T> x, Pair<T> y) { return {x.a * y.a, x.b * y.b}; }
template <typename T> MPC_HD Pair<T> fma2(Pair<T> x, Pair<T> y, Pair<T> z) { return {x.a * y.a + z.a, x.b * y.b + z.b}; }
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ float2 f2_(Pair<float> x) { return make_float2(x.a, x.b); }
__device__ __forceinline__ Pair<float> add2(Pair<float> x, Pair<float> y) { const float2 r = __fadd2_rn(f2_(x), f2_(y)); return {r.x, r.y}; }
__device__ __forceinline__ Pair<float> mul2(Pair<float> x, Pair<float> y) { const float2 r = __fmul2_rn(f2_(x), f2_(y)); return {r.x, r.y}; }
__device__ __forceinline__ Pair<float> fma2(Pair<float> x, Pair<float> y, Pair<float> z) {
  const float2 r = __ffma2_rn(f2_(x), f2_(y), f2_(z));
  return {r.x, r.y};
}
#endif
// x - y as x + (-y): the same IEEE result
template <typename T> MPC_HD Pair<T> sub2(Pair<T> x, Pair<T> y) { return add2(x, Pair<T>{-y.a, -y.b}); }

template <typename T> MPC_HD T min_(T a, T b) { return a < b ? a : b; }
template <typename T> MPC_HD T max_(T a, T b) { return a > b ? a : b; }
template <typename T> MPC_HD T clamp_(T x, T lo, T hi) { return min_(max_(x, lo), hi); }

// ---- configuration shared by the whole batch ----------------------------------------
struct SolverConfig {
  int N;                  // horizon (cfg.yaml:90 ships 16; benchmark 20)
  int M;                  // obstacle slots per problem
  float dt;               // 1 / policy_frequency  (base_agent.py:43)
  float w_distance;       // cfg.yaml:105 (10) in the archive objective; 0 = live agent
  float w_collision;      // cfg.yaml:106; 0 = live agent
  int literal_no_collision;  // 1: objective of pure_mpc_no_collision.py:146-151
  int max_iter;           // DDP iterations per problem (reference: ipopt.max_iter 1000, pure_mpc.py:294)
  float tol_step;         // convergence: max |du| of the accepted full step
  float reg_min;          // floor on |eigenvalue| of the regularised Quu
  float stall_tol;        // relative objective decrease per 6 iterations below which a problem is declared stalled
  float kink_tol;         // relative objective decrease per 6 iterations below which small steps count as converged
};

// ---- per-problem scalars -------------------------------------------------------------
template <typename T> struct ProblemScalars {
  // Positions are carried RELATIVE to the ego's initial position (x0, y0): the rollout then starts
  // at 0 and stays within ~25 m, and path / obstacle offsets are formed in FP64 before rounding,
  // so FP32 tracking and distance residuals keep ~1e-7 m accuracy instead of ulp(50 m).
  double x0, y0;
  int ego_index;          // nearest reference row (pure_mpc.py:106-109)
  int n_obs;              // present obstacles (<= M)
  int is_collide;
  T w_speed;              // already 100 when is_collide (pure_mpc.py:143-147)
  T w_control, w_diff;    // weights_from_RL or cfg defaults (pure_mpc.py:96-104)
  // reference-speed profile seen by stage k: k < vr_n ? vr_a + k*vr_slope : vr_b
  // (constant profile: vr_n = 0; regenerated ramp pure_mpc.py:707-716: vr_a = v_ego,
  //  slope = -v_ego/(n-1), vr_n = n, vr_b = 0)
  T vr_a, vr_slope, vr_b;
  int vr_n;
};

// reference path: FP64 positions (85 x 2) and a scalar-typed (heading, sin h, cos h) table
template <typename T> struct RefTab {
  const T* hsc;
  const double* xy;
};
template <typename T> struct RefPoint { T x, y, h, sh, ch; };
// The heading is constant on the two straights of the path (rows 0..39: -pi/2, rows 59..84: -pi, agents/base_agent.py:127-152),
// so every row of a straight reads the SAME table entry: lanes whose problems sit on a straight -- most of them -- then
// hit one shared-memory address (a broadcast) instead of 32 divergent rows (bank-conflict replays).  Same values bit for bit.
MPC_HD int heading_row(int j) { return j < 39 ? 39 : (j > 59 ? 59 : j); }
template <typename T> MPC_HD RefPoint<T> ref_point(const RefTab<T>& rt, const ProblemScalars<T>& p, int k) {
  int j = p.ego_index + k;                              // j(k) = min(ego_index + k, 84), pure_mpc.py:129
  j = j < kNRef - 1 ? j : kNRef - 1;
  RefPoint<T> r;
  r.x = T(rt.xy[2 * j] - p.x0);
  r.y = T(rt.xy[2 * j + 1] - p.y0);
  const int jh = heading_row(j);
  r.h = rt.hsc[jh * kRefStride]; r.sh = rt.hsc[jh * kRefStride + 1]; r.ch = rt.hsc[jh * kRefStride + 2];
  return r;
}

// same, with the positions taken from the problem's own column where the slot file stages them (bit-identical values:
// the column holds exactly T(xy - x0) of the rows j(k))
template <typename T, typename SL>
MPC_HD RefPoint<T> ref_point(const RefTab<T>& rt, const ProblemScalars<T>& p, const SL& sl, int k) {
  if constexpr (SL::kRefStaged) {
    int j = p.ego_index + k;
    j = j < kNRef - 1 ? j : kNRef - 1;
    RefPoint<T> r;
    r.x = sl.R(k, 0); r.y = sl.R(k, 1);
    const int jh = heading_row(j);
    r.h = rt.hsc[jh * kRefStride]; r.sh = rt.hsc[jh * kRefStride + 1]; r.ch = rt.hsc[jh * kRefStride + 2];
    return r;
  } else {
    return ref_point(rt, p, k);
  }
}

template <typename T> MPC_HD T ref_speed_at(const ProblemScalars<T>& p, int k) {
  return (k < p.vr_n) ? p.vr_a + T(k) * p.vr_slope : p.vr_b;
}

// ---- strided slot file ----------------------------------------------------------------
// base already points at this thread's lane; consecutive slots are `stride` apart.
// Gains: the 2x6 feedback matrix and the feed-forward pair of a stage are only ever used as a
// search direction (the step is validated by the line search on the exact objective), so on the
// device they are stored as bf16 pairs -- 7 words per stage instead of 14.  That is what lets 192
// instead of 128 problems stay resident per SM.  kPack = false keeps them in the scalar type
// (host harness, double).
MPC_HD uint32_t f2bf_bits(float f) {            // round-to-nearest-even float -> bf16 (finite inputs)
  uint32_t u;
  memcpy(&u, &f, 4);
  return (u + 0x7FFFu + ((u >> 16) & 1u)) >> 16;
}
MPC_HD uint32_t pack_bf16x2(float lo, float hi) {   // word = hi:bf16 << 16 | lo:bf16
#if defined(__CUDA_ARCH__)
  uint32_t w;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w) : "f"(hi), "f"(lo));
  return w;
#else
  return f2bf_bits(lo) | (f2bf_bits(hi) << 16);
#endif
}
MPC_HD float bf_bits2f(uint32_t h) {
  uint32_t u = h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
// kStride > 0: the stride is a compile-time constant (= block size on the device), so every slot
// address is base + immediate and no address arithmetic is issued; kStride = 0: run-time stride.
template <typename T, bool kPack, int kStride = 0> struct Slots {
  T* base;
  int stride;
  int N, M;
  MPC_HD T& at(int s) const { return base[(unsigned)s * (unsigned)(kStride > 0 ? kStride : stride)]; }
  static constexpr int kGainWords = kPack ? 7 : 14;
  static constexpr bool kRefStaged = false;      // path positions are read from the block's table at every use
  // layout
  MPC_HD int oU() const { return 0; }                       // 2N
  MPC_HD int oX() const { return 2 * N; }                   // 4(N+1)
  MPC_HD int oG() const { return 2 * N + 4 * (N + 1); }     // gains + feed-forward
  MPC_HD int oO() const { return oG() + kGainWords * N; }   // 4M obstacles x,y,incx,incy
  MPC_HD T& U(int k, int i) const { return at(oU() + 2 * k + i); }
  MPC_HD T& X(int k, int i) const { return at(oX() + 4 * k + i); }
  MPC_HD T& O(int m, int i) const { return at(oO() + 4 * m + i); }
  // Kg[r][c]: rows (accel, steer), columns dz = (x, y, theta, v, a_prev, d_prev)
  MPC_HD void store_gains(int k, T k0, T k1, const T (&Kg)[2][6]) const {
    const int o = oG() + kGainWords * k;
    if (kPack) {
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        uint32_t w = pack_bf16x2(float(Kg[0][c]), float(Kg[1][c]));
        memcpy(&at(o + c), &w, 4);
      }
      uint32_t w = pack_bf16x2(float(k0), float(k1));
      memcpy(&at(o + 6), &w, 4);
    } else {
#pragma unroll
      for (int c = 0; c < 6; ++c) { at(o + c) = Kg[0][c]; at(o + 6 + c) = Kg[1][c]; }
      at(o + 12) = k0; at(o + 13) = k1;
    }
  }
  MPC_HD void gains_fence() const {}
  MPC_HD void load_gains(int k, T& k0, T& k1, T (&Kr)[12]) const {
    const int o = oG() + kGainWords * k;
    if (kPack) {
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        uint32_t w;
        memcpy(&w, &at(o + c), 4);
        Kr[c] = T(bf_bits2f(w & 0xFFFFu)); Kr[6 + c] = T(bf_bits2f(w >> 16));
      }
      uint32_t w;
      memcpy(&w, &at(o + 6), 4);
      k0 = T(bf_bits2f(w & 0xFFFFu)); k1 = T(bf_bits2f(w >> 16));
    } else {
#pragma unroll
      for (int c = 0; c < 12; ++c) Kr[c] = at(o + c);
      k0 = at(o + 12); k1 = at(o + 13);
    }
  }
};
#if defined(__CUDACC__)
// ---- slot file with the gains in TENSOR MEMORY (Blackwell TMEM, 256 KB / SM) ------------------------
// tcgen05.ld/st with shape 32x32b give every thread of a warp a private 32-bit cell per TMEM column
// (lane = 32 (warp % 4) + laneid), i.e. TMEM is usable as a per-thread scratchpad with 12-cycle loads.  The
// 7 gain words of a stage live in 8 consecutive columns of the warp's own column range, so the shared-
// memory footprint of a problem drops from 296 to 156 words and 352 instead of 192 problems stay
// resident per SM.  The instructions are warp-collective (.sync.aligned, one column address for the
// warp): the kernel that uses this type runs every sweep with all 32 lanes (k_solve_tmem).
template <int kStride> struct SlotsTmem {
  float* base;
  uint32_t taddr;        // (lane quarter << 16) | first column of this warp's range
  int N, M;
  static constexpr bool kTmem = true;
  // the ego-relative path positions of the problem's N stages live in its own column (written once when the problem is
  // loaded): the per-lane table reads at divergent rows ego_index + k -- an FP64 pair per stage in every sweep -- were a
  // quarter of the kernel's shared-memory wavefronts (bank conflicts, profiles/r01_k_solve_ncu_full.json)
  static constexpr bool kRefStaged = true;
  __device__ __forceinline__ float& at(int s) const { return base[(unsigned)s * (unsigned)kStride]; }
  __device__ __forceinline__ int oU() const { return 0; }
  __device__ __forceinline__ int oX() const { return 2 * N; }
  __device__ __forceinline__ int oO() const { return 2 * N + 4 * (N + 1); }
  __device__ __forceinline__ int oR() const { return 2 * N + 4 * (N + 1) + 4 * M; }
  __device__ __forceinline__ float& R(int k, int i) const { return at(oR() + 2 * k + i); }
  __device__ __forceinline__ float& U(int k, int i) const { return at(oU() + 2 * k + i); }
  __device__ __forceinline__ float& X(int k, int i) const { return at(oX() + 4 * k + i); }
  __device__ __forceinline__ float& O(int m, int i) const { return at(oO() + 4 * m + i); }
  __device__ __forceinline__ void store_gains(int k, float k0, float k1, const float (&Kg)[2][6]) const {
    uint32_t w[8];
#pragma unroll
    for (int c = 0; c < 6; ++c) w[c] = pack_bf16x2(Kg[0][c], Kg[1][c]);
    w[6] = pack_bf16x2(k0, k1);
    w[7] = 0u;
    __syncwarp();
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n"
                 :: "r"(taddr + 8u * (uint32_t)k), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
  }
  __device__ __forceinline__ void load_gains(int k, float& k0, float& k1, float (&Kr)[12]) const {
    uint32_t w[8];
    __syncwarp();
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
                 : "r"(taddr + 8u * (uint32_t)k) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int c = 0; c < 6; ++c) { Kr[c] = bf_bits2f(w[c] & 0xFFFFu); Kr[6 + c] = bf_bits2f(w[c] >> 16); }
    k0 = bf_bits2f(w[6] & 0xFFFFu); k1 = bf_bits2f(w[6] >> 16);
  }
  __device__ __forceinline__ void gains_fence() const {
    __syncwarp();
    asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
  }
};
MPC_HD int slots_per_problem_tmem(int N, int M) { return 2 * N + 4 * (N + 1) + 4 * M + 2 * N; }
#endif

MPC_HD int slots_per_problem(int N, int M, bool pack) { return 2 * N + 4 * (N + 1) + (pack ? 7 : 14) * N + 4 * M; }

// ---- steering terms -------------------------------------------------------------------
// beta = atan(0.5 tan delta) (pure_mpc.py:221) expressed without atan/tan:
// q = cos^2 d + 0.25 sin^2 d, cos b = cos d / sqrt q, sin b = 0.5 sin d / sqrt q,
// beta' = 0.5 / q, beta'' = 0.75 sin d cos d / q^2.
template <typename T> struct Steer { T sb, cb, g, h; };
template <typename T> MPC_HD Steer<T> steer_terms(T delta, bool second) {
  T sd, cd;
  sincos_(delta, &sd, &cd);
  T q = T(1) - T(0.75) * sd * sd;
  T r = rsqrt_(q);
  Steer<T> o;
  o.cb = cd * r;
  o.sb = T(0.5) * sd * r;
  T iq = rcp_(q);
  o.g = T(0.5) * iq;
  o.h = second ? T(0.75) * sd * cd * iq * iq : T(0);
  return o;
}

// one Euler step (pure_mpc.py:252-254) given sin/cos of theta and the steering terms
template <typename T>
MPC_HD void euler_step(T& x, T& y, T& th, T& v, T a, const Steer<T>& st, T dt, T* c_out = nullptr, T* s_out = nullptr) {
  T sth, cth;
  sincos_(th, &sth, &cth);
  T c = cth * st.cb - sth * st.sb;     // cos(theta + beta)
  T s = sth * st.cb + cth * st.sb;     // sin(theta + beta)
  if (c_out) { *c_out = c; *s_out = s; }
  x += dt * v * c;
  y += dt * v * s;
  th += dt * v * st.sb * T(1.0 / 2.5);  // agents/utils.py:18 wheelbase 2.5
  v += dt * a;
}

// ---- stage cost (value only) ------------------------------------------------------------
// comp[0..5] accumulate the reference's six un-weighted components (pure_mpc.py:215-216);
// returns the weighted stage objective (pure_mpc.py:204-212 + archive terms).
template <typename T, typename SL>
MPC_HD T stage_cost(const SolverConfig& cfg, const ProblemScalars<T>& p, const RefTab<T>& ref,
                    const SL& sl, int k, T x, T y, T th, T v, T a, T d, T ap, T dp, T* comp) {
  const RefPoint<T> r = ref_point(ref, p, sl, k);
  T dx = x - r.x, dy = y - r.y;
  T perp = dx * r.sh - dy * r.ch;
  T para = dx * r.ch + dy * r.sh;
  T dv = v - ref_speed_at(p, k);
  T dth = th - r.h;
  T st = T(4) * perp * perp + T(2) * para * para + p.w_speed * dv * dv + T(0.5) * dth * dth;
  T ct = T(0.01) * (a * a + d * d);
  T df = T(0);
  if (k > 0) { T ea = a - ap, ed = d - dp; df = T(0.01) * (ea * ea + ed * ed); }
  T dist = T(0);
  if (cfg.w_distance != 0.f || comp) {
    // c / (d + 1e-6)^2 with 1/(d + eps) = (1/d)(1 - eps/d + ...): one MUFU.RSQ per obstacle, the
    // dropped (eps/d)^2 term is < 1e-12 relative for d > 1 mm
    const T kf = T(k);
MPC_PRAGMA_UNROLL_OBS
    for (int m = 0; m < p.n_obs; ++m) {
      T ex = (x - sl.O(m, 0)) - kf * sl.O(m, 2);
      T ey = (y - sl.O(m, 1)) - kf * sl.O(m, 3);
      T d2 = ex * ex + (ey * ey + T(1e-30));
      T idd = rsqrt_(d2);
      T c = d2 < T(1) ? T(1000) : T(100);
      dist += c * (idd * idd) * (T(1) - T(2e-6) * idd);
    }
  }
  T col = p.is_collide ? T(3000) * v * v : T(0);
  if (comp) { comp[0] += st; comp[1] += ct; comp[3] += df; comp[4] += dist; comp[5] += col; }
  if (cfg.literal_no_collision) return p.w_control * ct + p.w_diff * df;
  return T(10) * st + p.w_control * ct + p.w_diff * df + T(cfg.w_distance) * dist + T(cfg.w_collision) * col;
}

// stage_cost of the line search's two candidates at once (no components): the same operations on each lane, with the
// multiply-adds fused exactly where the device build of stage_cost fuses them inside forward_pass<T, 2> (read from its
// SASS of every solve kernel; e.g. the input-difference sum is fma(ed, ed, ea^2) there but fma(ea, ea, ed^2) in the
// single-candidate sweep).  The scalar code fuses `para` differently per slot type: fma(dy, sh, dx ch) where the path
// positions are staged in the problem's column (SlotsTmem, k_solve_tmem), fma(dx, ch, dy sh) where they are read from
// the block's table (Slots, k_solve).  The shared operands (reference point, reference speed, obstacle tracks) are
// broadcast once per stage and obstacle; rsqrt_ and the selects stay per lane.
template <typename T, typename SL>
MPC_HD Pair<T> stage_cost2(const SolverConfig& cfg, const ProblemScalars<T>& p, const RefTab<T>& ref, const SL& sl, int k,
                           Pair<T> x, Pair<T> y, Pair<T> th, Pair<T> v, Pair<T> a, Pair<T> d, Pair<T> ap, Pair<T> dp) {
  const RefPoint<T> r = ref_point(ref, p, sl, k);
  const Pair<T> sh = splat(r.sh), ch = splat(r.ch);
  const Pair<T> dx = add2(x, splat(-r.x)), dy = add2(y, splat(-r.y));
  const Pair<T> perp = fma2(dx, sh, mul2(dy, splat(-r.ch)));     // dx sh - dy ch
  const Pair<T> para = SL::kRefStaged ? fma2(dy, sh, mul2(dx, ch)) : fma2(dx, ch, mul2(dy, sh));   // dx ch + dy sh
  const Pair<T> dv = add2(v, splat(-ref_speed_at(p, k)));
  const Pair<T> dth = add2(th, splat(-r.h));
  Pair<T> st = fma2(perp, mul2(perp, splat(T(4))), mul2(para, add2(para, para)));
  st = fma2(dv, mul2(splat(p.w_speed), dv), st);
  st = fma2(dth, mul2(dth, splat(T(0.5))), st);
  const Pair<T> ct = mul2(fma2(a, a, mul2(d, d)), splat(T(0.01)));
  Pair<T> df = splat(T(0));
  if (k > 0) { const Pair<T> ea = sub2(a, ap), ed = sub2(d, dp); df = mul2(fma2(ed, ed, mul2(ea, ea)), splat(T(0.01))); }
  Pair<T> dist = splat(T(0));
  if (cfg.w_distance != 0.f) {
    const Pair<T> nkf = splat(-T(k));
    const Pair<T> tiny = splat(T(1e-30)), one = splat(T(1)), neps = splat(-T(2e-6));
MPC_PRAGMA_UNROLL_OBS
    for (int m = 0; m < p.n_obs; ++m) {
      const Pair<T> ex = fma2(nkf, splat(sl.O(m, 2)), add2(x, splat(-sl.O(m, 0))));
      const Pair<T> ey = fma2(nkf, splat(sl.O(m, 3)), add2(y, splat(-sl.O(m, 1))));
      const Pair<T> d2 = fma2(ex, ex, fma2(ey, ey, tiny));
      const Pair<T> idd = {rsqrt_(d2.a), rsqrt_(d2.b)};
      const Pair<T> c = {d2.a < T(1) ? T(1000) : T(100), d2.b < T(1) ? T(1000) : T(100)};
      dist = fma2(mul2(c, mul2(idd, idd)), fma2(idd, neps, one), dist);
    }
  }
  const Pair<T> col = p.is_collide ? mul2(mul2(v, splat(T(3000))), v) : splat(T(0));
  if (cfg.literal_no_collision) return fma2(splat(p.w_control), ct, mul2(splat(p.w_diff), df));
  Pair<T> J = fma2(splat(p.w_control), ct, mul2(st, splat(T(10))));
  J = fma2(splat(p.w_diff), df, J);
  J = fma2(dist, splat(T(cfg.w_distance)), J);
  return fma2(col, splat(T(cfg.w_collision)), J);
}

// ---- state bounds as state-dependent control boxes ------------------------------------------
// The reference bounds every shooting node: 0 <= v_k <= 30, |theta_k| <= pi (pure_mpc.py:272-274).
// With Euler dynamics both have relative degree one: v_{k+1} = v_k + dt a_k and
// theta_{k+1} = theta_k + dt (v_k / L) sin beta(delta_k), so "node k+1 inside its bounds" is the
// same set as a box on u_k whose edges depend on (theta_k, v_k).  The forward pass clamps to
// that box exactly (every iterate is feasible); the backward pass treats a control sitting on a
// state-dependent edge as the affine policy du = d(edge)/dx dx, i.e. the active-set SQP step.
// The steering edge is kept in sin(beta) space (theta+ is affine in sin beta): the inverse map to a
// steering angle (asinf) is only evaluated when a candidate control actually violates the edge.
template <typename T> struct Box {
  T lo_a, hi_a;         // acceleration bounds at this node
  T sb_lo, sb_hi;       // bounds on sin(beta(delta)) at this node, within +-sin(beta(pi/3))
  bool sa_lo, sa_hi, sd_lo, sd_hi;   // edge comes from a state bound (not the constant limit)
};
template <typename T> MPC_HD T sb_max() { return T(0.6546536707079771); }   // sin beta(pi/3)
MPC_HD float asin_(float x) { return asinf(x); }
MPC_HD double asin_(double x) { return asin(x); }
// inverse of sin beta(delta) = 0.5 sin d / sqrt(1 - 0.75 sin^2 d); out of line: asinf is long and rare
template <typename T> MPC_NOINLINE T delta_of_sinbeta(T sb) {
  sb = clamp_(sb, -sb_max<T>(), sb_max<T>());
  return asin_(sb * rsqrt_(T(0.25) + T(0.75) * sb * sb));
}
template <typename T> MPC_HD Box<T> control_box(T th, T v, T dt) {
  Box<T> b;
  b.lo_a = -Lim<T>::a_max(); b.hi_a = Lim<T>::a_max();
  b.sb_lo = -sb_max<T>(); b.sb_hi = sb_max<T>();
  b.sa_lo = b.sa_hi = b.sd_lo = b.sd_hi = false;
  const T idt = rcp_(dt);
  T ha = (Lim<T>::v_max() - v) * idt, la = (Lim<T>::v_min() - v) * idt;
  if (ha < b.hi_a) { b.hi_a = ha; b.sa_hi = true; }
  if (la > b.lo_a) { b.lo_a = la; b.sa_lo = true; }
  if (b.hi_a < b.lo_a) { b.hi_a = b.lo_a; }                 // v0 outside [0, 30]: keep a defined box
  const T gain = dt * v * T(1.0 / 2.5);                      // d theta+ / d sin beta
  const T reach = gain * sb_max<T>();
  if (th + reach > Lim<T>::th_max()) { b.sb_hi = (Lim<T>::th_max() - th) * rcp_(gain); b.sd_hi = true; }
  if (th - reach < -Lim<T>::th_max()) { b.sb_lo = (-Lim<T>::th_max() - th) * rcp_(gain); b.sd_lo = true; }
  if (b.sb_hi < b.sb_lo) { b.sb_hi = b.sb_lo; }
  return b;
}
// clamp a steering angle to the node's box; returns the steering terms of the clamped angle
template <typename T> MPC_HD Steer<T> clamp_steer(const Box<T>& b, T& delta, bool second) {
  delta = clamp_(delta, -Lim<T>::d_max(), Lim<T>::d_max());
  Steer<T> st = steer_terms(delta, second);
  if (st.sb > b.sb_hi || st.sb < b.sb_lo) {
    delta = delta_of_sinbeta(clamp_(st.sb, b.sb_lo, b.sb_hi));
    st = steer_terms(delta, second);
  }
  return st;
}

// ---- open-loop rollout of the stored controls; fills X, returns the objective ----------------
// Controls are used as stored (no clamping): this is also the parity entry point for
// "rollout + six cost components" (mpc_rollout_cost).
template <typename T, typename SL>
MPC_HD T rollout_nominal(const SolverConfig& cfg, const ProblemScalars<T>& p, const RefTab<T>& ref,
                         const SL& sl, T* comp /*6 or null*/) {
  const int N = cfg.N;
  T x = sl.X(0, 0), y = sl.X(0, 1), th = sl.X(0, 2), v = sl.X(0, 3);
  T J = T(0), ap = T(0), dp = T(0);
  for (int k = 0; k < N; ++k) {
    T a = sl.U(k, 0), d = sl.U(k, 1);
    J += stage_cost(cfg, p, ref, sl, k, x, y, th, v, a, d, ap, dp, comp);
    Steer<T> st = steer_terms(d, false);
    euler_step(x, y, th, v, a, st, T(cfg.dt));
    sl.X(k + 1, 0) = x; sl.X(k + 1, 1) = y; sl.X(k + 1, 2) = th; sl.X(k + 1, 3) = v;
    ap = a; dp = d;
  }
  return J;
}

// final_state component of the reference's cost_fn (agents/pure_mpc.py:195-202; note the
// (y + y_ref) sign) -- reported, never optimised.  Needs absolute y: formed in FP64.
template <typename T, typename SL>
MPC_HD T final_state_component(const SolverConfig& cfg, const ProblemScalars<T>& p, const RefTab<T>& ref, const SL& sl) {
  const int N = cfg.N;
  const RefPoint<T> r = ref_point(ref, p, N);
  int j = p.ego_index + N;
  j = j < kNRef - 1 ? j : kNRef - 1;
  T ex = sl.X(N, 0) - r.x;
  T ey = T((p.y0 + double(sl.X(N, 1))) + ref.xy[2 * j + 1]);
  T ev = sl.X(N, 3) - ref_speed_at(p, N), eth = sl.X(N, 2) - r.h;
  return T(100) * (ex * ex + ey * ey + T(20) * ev * ev + eth * eth);
}

// ---- 2x2 box QP --------------------------------------------------------------------------
// min 1/2 d'Hd + g'd, lo <= d <= hi, H positive definite.  Exact: the Newton point if it is
// inside, otherwise the best of the four edge minimisers.  side[i] = 0 free, -1 at lo, +1 at hi.
template <typename T>
MPC_HD void box_qp2(T h00, T h01, T h11, T g0, T g1, T lo0, T hi0, T lo1, T hi1, T* d0, T* d1, int* side0, int* side1) {
  T idet = rcp_(h00 * h11 - h01 * h01);
  T n0 = -(h11 * g0 - h01 * g1) * idet;
  T n1 = -(h00 * g1 - h01 * g0) * idet;
  if (n0 >= lo0 && n0 <= hi0 && n1 >= lo1 && n1 <= hi1) { *d0 = n0; *d1 = n1; *side0 = 0; *side1 = 0; return; }
  T best = T(1e30), b0 = T(0), b1 = T(0);
  int s0 = 0, s1 = 0;
  const T ih11 = rcp_(h11), ih00 = rcp_(h00);
#pragma unroll
  for (int e = 0; e < 2; ++e) {          // coordinate 0 pinned to an edge
    T f0 = e ? hi0 : lo0;
    T u1 = -(g1 + h01 * f0) * ih11;
    int t1 = u1 <= lo1 ? -1 : (u1 >= hi1 ? 1 : 0);
    u1 = clamp_(u1, lo1, hi1);
    T val = T(0.5) * (h00 * f0 * f0 + T(2) * h01 * f0 * u1 + h11 * u1 * u1) + g0 * f0 + g1 * u1;
    if (val < best) { best = val; b0 = f0; b1 = u1; s0 = e ? 1 : -1; s1 = t1; }
  }
#pragma unroll
  for (int e = 0; e < 2; ++e) {          // coordinate 1 pinned to an edge
    T f1 = e ? hi1 : lo1;
    T u0 = -(g0 + h01 * f1) * ih00;
    int t0 = u0 <= lo0 ? -1 : (u0 >= hi0 ? 1 : 0);
    u0 = clamp_(u0, lo0, hi0);
    T val = T(0.5) * (h00 * u0 * u0 + T(2) * h01 * u0 * f1 + h11 * f1 * f1) + g0 * u0 + g1 * f1;
    if (val < best) { best = val; b0 = u0; b1 = f1; s0 = t0; s1 = e ? 1 : -1; }
  }
  *d0 = b0; *d1 = b1; *side0 = s0; *side1 = s1;
}

// symmetric 6x6 in 21 registers, upper triangle, row-major
MPC_HD constexpr int sym6(int i, int j) { return i <= j ? (i * (13 - i)) / 2 + (j - i) : (j * (13 - j)) / 2 + (i - j); }

// ---- look-ahead half-plane (see backward_pass) ---------------------------------------------------------------------
// Minimiser of the stage model 1/2 du'H du + qu'du on the line n'du = r inside the control box, its multiplier, and the
// feedback gains that keep the line under a perturbation dz of the stage's state (n'du = r - m'dz, m = A'c).  Rare, so
// kept out of line: the hot sweep only tests  n'k < r.
template <typename T> struct LaIO {
  T n0, n1, r, jump, h00, h01, h11, qu0, qu1, lo0, hi0, lo1, hi1, m2, m3, a34;
  T e03_lo, e03_hi, e12_lo, e12_hi;     // gains of the box edges that come from a node bound (0 = constant limit)
  T Rz[2][6];
  T k0, k1;                             // in: box minimiser; out: constrained minimiser
  T Kg[2][6];
  int s0, s1;
  bool applied;
};
template <typename T> MPC_NOINLINE void la_constrain(LaIO<T>& io) {
  io.applied = false;
  const T n0 = io.n0, n1 = io.n1, nn = n0 * n0 + n1 * n1;
  if (!(nn > T(1e-20))) return;
  const T inn = rcp_(nn);
  const T p0 = io.r * n0 * inn, p1 = io.r * n1 * inn, t0 = -n1, t1 = n0;
  const T Ht0 = io.h00 * t0 + io.h01 * t1, Ht1 = io.h01 * t0 + io.h11 * t1;
  const T tHt = t0 * Ht0 + t1 * Ht1;
  T tlo = T(-1e30), thi = T(1e30);
  bool feas = tHt > T(0);
  if (abs_(t0) > T(1e-12)) { const T it = rcp_(t0), u = (io.lo0 - p0) * it, w = (io.hi0 - p0) * it; tlo = max_(tlo, min_(u, w)); thi = min_(thi, max_(u, w)); }
  else feas = feas && p0 >= io.lo0 - T(1e-6) && p0 <= io.hi0 + T(1e-6);
  if (abs_(t1) > T(1e-12)) { const T it = rcp_(t1), u = (io.lo1 - p1) * it, w = (io.hi1 - p1) * it; tlo = max_(tlo, min_(u, w)); thi = min_(thi, max_(u, w)); }
  else feas = feas && p1 >= io.lo1 - T(1e-6) && p1 <= io.hi1 + T(1e-6);
  if (!feas || tlo > thi) return;                        // the line misses the box (this stage is saturated too)
  const T tau = -((Ht0 * p0 + Ht1 * p1) + io.qu0 * t0 + io.qu1 * t1) * rcp_(tHt);
  const T tc = clamp_(tau, tlo, thi);
  const T c0 = p0 + tc * t0, c1 = p1 + tc * t1;
  const T lam = (n0 * (io.h00 * c0 + io.h01 * c1 + io.qu0) + n1 * (io.h01 * c0 + io.h11 * c1 + io.qu1)) * inn;
  if (lam > io.jump) return;                             // crossing the line is worth its price: no constraint this sweep
  io.applied = true;
  io.k0 = clamp_(c0, io.lo0, io.hi0); io.k1 = clamp_(c1, io.lo1, io.hi1);
  for (int jc = 0; jc < 6; ++jc) { io.Kg[0][jc] = T(0); io.Kg[1][jc] = T(0); }
  if (tc == tau) {                                       // free along the line
    const T tHn = (Ht0 * n0 + Ht1 * n1) * inn, itHt = rcp_(tHt);
    for (int jc = 0; jc < 6; ++jc) {
      const T mj = jc == 2 ? io.m2 : (jc == 3 ? io.m3 : T(0));
      const T along = (tHn * mj - (t0 * io.Rz[0][jc] + t1 * io.Rz[1][jc])) * itHt;
      io.Kg[0][jc] = -n0 * inn * mj + t0 * along;
      io.Kg[1][jc] = -n1 * inn * mj + t1 * along;
    }
    io.s0 = 0; io.s1 = 0;
  } else {                                               // corner of the line and the box: nothing left to choose
    const bool pin0 = (io.k0 <= io.lo0 || io.k0 >= io.hi0);
    if (pin0 && abs_(n1) > T(1e-12)) {
      io.s0 = io.k0 <= io.lo0 ? -1 : 1; io.s1 = 0;
      io.Kg[0][3] = io.s0 > 0 ? io.e03_hi : io.e03_lo;
      const T in1 = rcp_(n1);
      io.Kg[1][2] = -io.m2 * in1; io.Kg[1][3] = -(io.m3 + n0 * io.Kg[0][3]) * in1;
    } else if (!pin0 && abs_(n0) > T(1e-12)) {
      io.s1 = io.k1 <= io.lo1 ? -1 : 1; io.s0 = 0;
      const T e = io.s1 > 0 ? io.e12_hi : io.e12_lo;
      io.Kg[1][2] = e; io.Kg[1][3] = io.a34 * e;
      const T in0 = rcp_(n0);
      io.Kg[0][2] = -(io.m2 + n1 * io.Kg[1][2]) * in0; io.Kg[0][3] = -(io.m3 + n1 * io.Kg[1][3]) * in0;
    } else {
      io.s0 = 0; io.s1 = 0;
    }
  }
}

// ---- backward pass -------------------------------------------------------------------------
// Fills K (2x6 per stage) and F (feed-forward) from the nominal (X, U); returns the two
// coefficients of the predicted objective change  dJ(alpha) = alpha*d1 + alpha^2*d2.
template <typename T, typename SL>
MPC_HD void backward_pass(const SolverConfig& cfg, const ProblemScalars<T>& p, const RefTab<T>& ref,
                          const SL& sl, T mu, T hs, T* d1_out, T* d2_out) {
  // hs in [0,1] scales the second-order dynamics terms and the negative (tangential) obstacle
  // curvature: 0 = Gauss-Newton/iLQR model (robust far from the solution), 1 = exact Hessian.
  const int N = cfg.N;
  const T dt = T(cfg.dt);
  const T iL = T(1.0 / 2.5);
  T P[21], pv[6];                 // value function of stage k+1 (x_N carries no cost: pure_mpc.py:128,204-212)
#pragma unroll
  for (int i = 0; i < 21; ++i) P[i] = T(0);
#pragma unroll
  for (int i = 0; i < 6; ++i) pv[i] = T(0);
  T d1 = T(0), d2 = T(0);
  const T cc2 = T(0.02) * p.w_control;
#if MPC_LOOKAHEAD
  // Look-ahead bound (round 2).  When the steering of stage k+1 is pinned on its CONSTANT limit, stage k+1 cannot
  // absorb a perturbation of its own state any more, so the bound of node k+2,
  //   theta_{k+2} = theta_{k+1} + dt (v_{k+1} / L) sin beta(-+pi/3)  within [-pi, pi],
  // is a linear inequality  c_theta dtheta_{k+1} + c_v dv_{k+1} >= la_r  on the state that stage k produces -- a
  // half-plane for du_k (c is one of four sign patterns, la_mode).  The mirror case -- steering riding the node bound's
  // own edge, a model that is only valid while that edge stays inside the constant limit -- gives the opposite half-plane.  Without it the model of stage k happily steps across that line, the forward pass then lifts
  // delta_{k+1} off its limit to stay feasible (a different smooth piece), the step is rejected, and the iteration creeps
  // onto the kink instead of moving ALONG it (status "settled on a kink").  la_jump = the first-order price of lifting
  // delta_{k+1} per radian of violation: if the multiplier of the half-plane exceeds it, crossing the line is worth it
  // and the constraint is dropped for this sweep.
  int la_mode = 0;
  T la_r = T(0), la_jump = T(0);
#endif
  for (int k = N - 1; k >= 0; --k) {
    const T x = sl.X(k, 0), y = sl.X(k, 1), th = sl.X(k, 2), v = sl.X(k, 3);
    const T a = sl.U(k, 0), d = sl.U(k, 1);
    const T cd2 = k > 0 ? T(0.02) * p.w_diff : T(0);
    T ap = T(0), dp = T(0);
    if (k > 0) { ap = sl.U(k - 1, 0); dp = sl.U(k - 1, 1); }
    // ---- dynamics derivatives
    Steer<T> st = steer_terms(d, true);
    T sth, cth;
    sincos_(th, &sth, &cth);
    const T c = cth * st.cb - sth * st.sb, s = sth * st.cb + cth * st.sb;
    const T a13 = -dt * v * s, a14 = dt * c, a23 = dt * v * c, a24 = dt * s, a34 = dt * st.sb * iL;
    const T b1 = a13 * st.g, b2 = a23 * st.g, b3 = dt * v * iL * st.cb * st.g;
    // ---- stage cost derivatives wrt state
    T lx = T(0), ly = T(0), lth = T(0), lv = T(0);
    T lxx = T(0), lxy = T(0), lyy = T(0), lthth = T(0), lvv = T(0);
    if (!cfg.literal_no_collision) {
      const RefPoint<T> r = ref_point(ref, p, sl, k);
      const T sh = r.sh, ch = r.ch;
      T dx = x - r.x, dy = y - r.y;
      T perp = dx * sh - dy * ch, para = dx * ch + dy * sh;
      lx = T(80) * perp * sh + T(40) * para * ch;
      ly = -T(80) * perp * ch + T(40) * para * sh;
      lth = T(10) * (th - r.h);
      T wv = T(20) * p.w_speed;
      lv = wv * (v - ref_speed_at(p, k));
      lxx = T(80) * sh * sh + T(40) * ch * ch;
      lxy = -T(40) * sh * ch;
      lyy = T(80) * ch * ch + T(40) * sh * sh;
      lthth = T(10);
      lvv = wv;
      if (cfg.w_distance != 0.f) {
        const T wd = T(cfg.w_distance);
        const T kf = T(k);
MPC_PRAGMA_UNROLL_OBS
        for (int m = 0; m < p.n_obs; ++m) {
          T ex = (x - sl.O(m, 0)) - kf * sl.O(m, 2);
          T ey = (y - sl.O(m, 1)) - kf * sl.O(m, 3);
          T d2_ = ex * ex + (ey * ey + T(1e-30));
          T idd = rsqrt_(d2_);
          T cw = wd * (d2_ < T(1) ? T(1000) : T(100));
          T ie = idd * (T(1) - T(1e-6) * idd);      // 1/(d + 1e-6) to first order in 1e-6/d
          T ie2 = ie * ie;
          T f1 = -T(2) * cw * ie2 * ie;          // phi'(d)
          T f2 = T(6) * cw * ie2 * ie2;          // phi''(d)
          T nx = ex * idd, ny = ey * idd;
          T tang = hs * f1 * idd;                 // phi'/d  (negative: tangential curvature)
          lx += f1 * nx; ly += f1 * ny;
          T rad = f2 - tang;
          lxx += rad * nx * nx + tang;
          lxy += rad * nx * ny;
          lyy += rad * ny * ny + tang;
        }
      }
      if (cfg.w_collision != 0.f && p.is_collide) {
        lv += T(6000) * T(cfg.w_collision) * v;
        lvv += T(6000) * T(cfg.w_collision);
      }
    }
    // ---- contractions with the next-stage costate (second-order DDP terms)
    const T p1 = pv[0], p2 = pv[1], p3 = pv[2], p4 = pv[3];
    const T mm = p1 * c + p2 * s, nn = -p1 * s + p2 * c;
    const T Hthth = hs * (-dt * v * mm);
    const T Hthv = hs * (dt * nn);
    const T Hthd = hs * (-dt * v * st.g * mm);
    const T Hvd = hs * (dt * st.g * nn + p3 * dt * iL * st.cb * st.g);
    const T Hdd = hs * (dt * v * (-st.g * st.g * mm + st.h * nn) + p3 * dt * v * iL * (-st.sb * st.g * st.g + st.cb * st.h));
    // ---- Qz, Qu
    T Qz[6], Qu[2];
    Qz[0] = lx + p1;
    Qz[1] = ly + p2;
    Qz[2] = lth + p3 + dt * v * nn;
    Qz[3] = lv + p4 + dt * mm + p3 * a34;
    Qz[4] = -cd2 * (a - ap);
    Qz[5] = -cd2 * (d - dp);
    Qu[0] = cc2 * a + cd2 * (a - ap) + dt * p4 + pv[4];
    Qu[1] = cc2 * d + cd2 * (d - dp) + b1 * p1 + b2 * p2 + b3 * p3 + pv[5];
    // ---- M = Pss A (4x4), W = Pus A (2x4)
    T Mx[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      T pi0 = P[sym6(i, 0)], pi1 = P[sym6(i, 1)], pi2 = P[sym6(i, 2)], pi3 = P[sym6(i, 3)];
      Mx[i][0] = pi0;
      Mx[i][1] = pi1;
      Mx[i][2] = pi2 + a13 * pi0 + a23 * pi1;
      Mx[i][3] = pi3 + a14 * pi0 + a24 * pi1 + a34 * pi2;
    }
    T W[2][4];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      T q0 = P[sym6(4 + r, 0)], q1 = P[sym6(4 + r, 1)], q2 = P[sym6(4 + r, 2)], q3 = P[sym6(4 + r, 3)];
      W[r][0] = q0;
      W[r][1] = q1;
      W[r][2] = q2 + a13 * q0 + a23 * q1;
      W[r][3] = q3 + a14 * q0 + a24 * q1 + a34 * q2;
    }
    // ---- Quz (2x6)
    T Quz[2][6];
#pragma unroll
    for (int jc = 0; jc < 4; ++jc) {
      Quz[0][jc] = dt * Mx[3][jc] + W[0][jc];
      Quz[1][jc] = b1 * Mx[0][jc] + b2 * Mx[1][jc] + b3 * Mx[2][jc] + W[1][jc];
    }
    Quz[1][2] += Hthd;
    Quz[1][3] += Hvd;
    Quz[0][4] = -cd2; Quz[0][5] = T(0);
    Quz[1][4] = T(0); Quz[1][5] = -cd2;
    // ---- Quu
    T PBd[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) PBd[i] = b1 * P[sym6(i, 0)] + b2 * P[sym6(i, 1)] + b3 * P[sym6(i, 2)];
    T BPa0 = dt * P[sym6(3, 4)], BPa1 = dt * P[sym6(3, 5)];
    T BPd0 = b1 * P[sym6(0, 4)] + b2 * P[sym6(1, 4)] + b3 * P[sym6(2, 4)];
    T BPd1 = b1 * P[sym6(0, 5)] + b2 * P[sym6(1, 5)] + b3 * P[sym6(2, 5)];
    const T luu = cc2 + cd2;
    T Quu00 = luu + dt * dt * P[sym6(3, 3)] + T(2) * BPa0 + P[sym6(4, 4)];
    T Quu01 = dt * PBd[3] + BPa1 + BPd0 + P[sym6(4, 5)];
    T Quu11 = luu + b1 * PBd[0] + b2 * PBd[1] + b3 * PBd[2] + T(2) * BPd1 + P[sym6(5, 5)] + Hdd;
    // ---- Qzz (sym 6x6): state block A'M + lss + H, (up,up) = cd2 I
    T Qzz[21];
#pragma unroll
    for (int i = 0; i < 21; ++i) Qzz[i] = T(0);
    Qzz[sym6(0, 0)] = Mx[0][0] + lxx;
    Qzz[sym6(0, 1)] = Mx[0][1] + lxy;
    Qzz[sym6(0, 2)] = Mx[0][2];
    Qzz[sym6(0, 3)] = Mx[0][3];
    Qzz[sym6(1, 1)] = Mx[1][1] + lyy;
    Qzz[sym6(1, 2)] = Mx[1][2];
    Qzz[sym6(1, 3)] = Mx[1][3];
    Qzz[sym6(2, 2)] = Mx[2][2] + a13 * Mx[0][2] + a23 * Mx[1][2] + lthth + Hthth;
    Qzz[sym6(2, 3)] = Mx[2][3] + a13 * Mx[0][3] + a23 * Mx[1][3] + Hthv;
    Qzz[sym6(3, 3)] = Mx[3][3] + a14 * Mx[0][3] + a24 * Mx[1][3] + a34 * Mx[2][3] + lvv;
    Qzz[sym6(4, 4)] = cd2;
    Qzz[sym6(5, 5)] = cd2;
    // ---- regularise Quu: replace its eigenvalues l by max(|l|, reg_min) + mu (saddle-free
    // modification; a uniform shift would cripple the healthy direction whenever the
    // second-order dynamics terms make the other one strongly negative)
    T h00 = Quu00, h01 = Quu01, h11 = Quu11;
    {
      T hm = T(0.5) * (h00 + h11), hd = T(0.5) * (h00 - h11);
      T rr = sqrt_(hd * hd + h01 * h01);
      T l1 = hm - rr, l2 = hm + rr;
      T n1 = max_(abs_(l1), T(cfg.reg_min)), n2 = max_(abs_(l2), T(cfg.reg_min));
      if (rr > T(1e-12) * (abs_(hm) + T(1e-30))) {
        T i2r = T(0.5) * rcp_(rr);
        T c0 = (n1 * l2 - n2 * l1) * i2r, c1 = (n2 - n1) * i2r;
        h00 = c0 + c1 * h00; h01 = c1 * h01; h11 = c0 + c1 * h11;
      } else {
        h00 = n1; h01 = T(0); h11 = n1;
      }
    }
    // ---- Levenberg term on the *next state* (mu |dz'|^2): keeps the new trajectory near the
    // nominal where the expansion holds; dz' = A dz + B du, plus the carried control
    const T f00 = h00, f01 = h01, f11 = h11;   // modified Quu without the Levenberg term
    T Rz[2][6];
#pragma unroll
    for (int jc = 0; jc < 6; ++jc) { Rz[0][jc] = Quz[0][jc]; Rz[1][jc] = Quz[1][jc]; }
    if (mu > T(0)) {
      h00 += mu * (dt * dt + T(1));
      h11 += mu * (b1 * b1 + b2 * b2 + b3 * b3 + T(1));
      Rz[0][3] += mu * dt;
      Rz[1][0] += mu * b1;
      Rz[1][1] += mu * b2;
      Rz[1][2] += mu * (b1 * a13 + b2 * a23 + b3);
      Rz[1][3] += mu * (b1 * a14 + b2 * a24 + b3 * a34);
    }
    // ---- box QP for the feed-forward on the (state-dependent) control box of this node
    const Box<T> bx = control_box(th, v, dt);
    // steering edges for the QP in delta space, linearised at the nominal (exact when the nominal
    // sits on the edge, which is the case that matters; the forward pass clamps exactly)
    const T isl = rcp_(st.cb * st.g);                       // d delta / d sin beta
    T hi_dd = Lim<T>::d_max() - d, lo_dd = -Lim<T>::d_max() - d;
    bool sd_hi = false, sd_lo = false;
    if (bx.sd_hi) { T e = max_((bx.sb_hi - st.sb) * isl, T(0)); if (e < hi_dd) { hi_dd = e; sd_hi = true; } }
    if (bx.sd_lo) { T e = min_((bx.sb_lo - st.sb) * isl, T(0)); if (e > lo_dd) { lo_dd = e; sd_lo = true; } }
    T k0, k1;
    int s0, s1;
    box_qp2(h00, h01, h11, Qu[0], Qu[1], bx.lo_a - a, bx.hi_a - a, lo_dd, hi_dd, &k0, &k1, &s0, &s1);
    // ---- gains: pinned coordinates follow their edge (constant edge: zero gain; edge that
    // comes from a node bound: d(edge)/dx), free coordinates minimise the model given those.
    // E = the control Hessian of the model that is actually minimised: the modified matrix on
    // the free block, the true curvature along pinned coordinates.  The same E is used in the
    // value recursion, otherwise negative curvature compounds backwards through the horizon.
    T Kg[2][6];
#pragma unroll
    for (int jc = 0; jc < 6; ++jc) { Kg[0][jc] = T(0); Kg[1][jc] = T(0); }
    if (s0 != 0 && ((s0 > 0) ? bx.sa_hi : bx.sa_lo)) Kg[0][3] = -rcp_(dt);          // keeps v+ on its bound
    if (s1 != 0 && ((s1 > 0) ? sd_hi : sd_lo) && b3 > T(1e-12)) {              // keeps theta+ on its bound
      T ib3 = rcp_(b3);
      Kg[1][2] = -ib3;
      Kg[1][3] = -a34 * ib3;
    }
    // pinned coordinates: true curvature along the edge policy, negative part dropped (the
    // edge's own curvature is not modelled, so a negative value is not trustworthy)
    T E00 = max_(Quu00, T(0)), E01 = Quu01, E11 = max_(Quu11, T(0));
    if (s0 == 0 && s1 == 0) {
      E00 = f00; E01 = f01; E11 = f11;
      T idet = rcp_(h00 * h11 - h01 * h01);
#pragma unroll
      for (int jc = 0; jc < 6; ++jc) {
        Kg[0][jc] = -(h11 * Rz[0][jc] - h01 * Rz[1][jc]) * idet;
        Kg[1][jc] = -(h00 * Rz[1][jc] - h01 * Rz[0][jc]) * idet;
      }
    } else if (s0 == 0) {
      E00 = max_(abs_(Quu00), T(cfg.reg_min)) + mu * (dt * dt + T(1));
      T ih = rcp_(E00);
      k0 = clamp_(-(Qu[0] + E01 * k1) * ih, bx.lo_a - a, bx.hi_a - a);
#pragma unroll
      for (int jc = 0; jc < 6; ++jc) Kg[0][jc] = -(Rz[0][jc] + E01 * Kg[1][jc]) * ih;
    } else if (s1 == 0) {
      E11 = max_(abs_(Quu11), T(cfg.reg_min)) + mu * (b1 * b1 + b2 * b2 + b3 * b3 + T(1));
      T ih = rcp_(E11);
      k1 = clamp_(-(Qu[1] + E01 * k0) * ih, lo_dd, hi_dd);
#pragma unroll
      for (int jc = 0; jc < 6; ++jc) Kg[1][jc] = -(Rz[1][jc] + E01 * Kg[0][jc]) * ih;
    }
#if MPC_LOOKAHEAD
    {
      // la_mode: 0 = none; else the half-plane  c'dx >= la_r  of the stage after this one with
      // c = (c_theta, c_v) = (+1, -gl) [1], (-1, -gl) [2] (steering on its constant limit, lower / upper node bound) or
      // (-1, +gl) [3], (+1, +gl) [4] (steering on the node bound's own edge), gl = dt sin beta(pi/3) / L
      const T gl = dt * sb_max<T>() * iL;
      if (la_mode != 0) {
        const T cth = (la_mode == 1 || la_mode == 4) ? T(1) : T(-1);
        const T cv = (la_mode <= 2) ? -gl : gl;
        const T n0 = cv * dt, n1 = cth * b3;                  // B' c
        if (n0 * k0 + n1 * k1 < la_r) {                       // rare: the box minimiser crosses the line -> out-of-line solve
          LaIO<T> io;
          io.n0 = n0; io.n1 = n1; io.r = la_r; io.jump = la_jump; io.h00 = h00; io.h01 = h01; io.h11 = h11;
          io.qu0 = Qu[0]; io.qu1 = Qu[1]; io.lo0 = bx.lo_a - a; io.hi0 = bx.hi_a - a; io.lo1 = lo_dd; io.hi1 = hi_dd;
          io.m2 = cth; io.m3 = cth * a34 + cv;
          io.e03_lo = bx.sa_lo ? -rcp_(dt) : T(0); io.e03_hi = bx.sa_hi ? -rcp_(dt) : T(0);
          const bool edge_ok = b3 > T(1e-12);
          io.e12_lo = (sd_lo && edge_ok) ? -rcp_(b3) : T(0); io.e12_hi = (sd_hi && edge_ok) ? -rcp_(b3) : T(0);
          io.a34 = a34;
#pragma unroll
          for (int jc = 0; jc < 6; ++jc) { io.Rz[0][jc] = Rz[0][jc]; io.Rz[1][jc] = Rz[1][jc]; }
          io.k0 = k0; io.k1 = k1;
          la_constrain(io);
          if (io.applied) {
            k0 = io.k0; k1 = io.k1; s0 = io.s0; s1 = io.s1;
            E00 = f00; E01 = f01; E11 = f11;
#pragma unroll
            for (int jc = 0; jc < 6; ++jc) { Kg[0][jc] = io.Kg[0][jc]; Kg[1][jc] = io.Kg[1][jc]; }
          }
        }
      }
      // constraint for the stage before this one: steering pinned here.  g = distance of "full steer keeps theta+ inside"
      // from being tight.  Pinned on the CONSTANT limit (model valid while g >= 0): the state of this stage must keep
      // g >= 0.  Pinned on the NODE BOUND's edge (model valid while the edge stays inside the constant limit, g <= 0): it
      // must keep g <= 0.  Either way one half-plane  c'dx >= r  with r <= 0, and the same price for crossing it.
      la_mode = 0;
      if (s1 != 0 && b3 > T(1e-9)) {
        const bool on_edge = (s1 > 0) ? sd_hi : sd_lo;
        const T g = s1 < 0 ? (th - v * gl) + Lim<T>::th_max() : Lim<T>::th_max() - (th + v * gl);
        la_mode = (s1 < 0 ? 1 : 2) + (on_edge ? 2 : 0);
        la_r = min_(on_edge ? g : -g, T(0));
        la_jump = abs_(Qu[1]) * rcp_(b3);
      }
    }
#endif
#if defined(MPC_TRACE2) && !defined(__CUDA_ARCH__)
    printf("  k %d Quu %.4g %.4g %.4g Hdd %.4g Qu %.4g %.4g kff %.4g %.4g side %d %d box d [%.4g %.4g] sd %d %d P22 %.4g P33 %.4g p %.3g %.3g %.3g %.3g\n", k, (double)Quu00, (double)Quu01, (double)Quu11, (double)Hdd,
           (double)Qu[0], (double)Qu[1], (double)k0, (double)k1, s0, s1, (double)lo_dd, (double)hi_dd, (int)sd_lo, (int)sd_hi, (double)P[sym6(2,2)], (double)P[sym6(3,3)], (double)pv[0], (double)pv[1], (double)pv[2], (double)pv[3]);
#endif
    sl.store_gains(k, k0, k1, Kg);
    // ---- predicted change and value update
    T Qk0 = E00 * k0 + E01 * k1, Qk1 = E01 * k0 + E11 * k1;
    d1 += k0 * Qu[0] + k1 * Qu[1];
    d2 += T(0.5) * (k0 * Qk0 + k1 * Qk1);
    T t0 = Qk0 + Qu[0], t1 = Qk1 + Qu[1];
    T Tm[2][6];
#pragma unroll
    for (int jc = 0; jc < 6; ++jc) {
      Tm[0][jc] = E00 * Kg[0][jc] + E01 * Kg[1][jc] + Quz[0][jc];
      Tm[1][jc] = E01 * Kg[0][jc] + E11 * Kg[1][jc] + Quz[1][jc];
      pv[jc] = Qz[jc] + Kg[0][jc] * t0 + Kg[1][jc] * t1 + Quz[0][jc] * k0 + Quz[1][jc] * k1;
    }
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
      for (int jc = i; jc < 6; ++jc)
        P[sym6(i, jc)] = Qzz[sym6(i, jc)] + Kg[0][i] * Tm[0][jc] + Kg[1][i] * Tm[1][jc] +
                         Quz[0][i] * Kg[0][jc] + Quz[1][i] * Kg[1][jc];
  }
  sl.gains_fence();
  *d1_out = d1;
  *d2_out = d2;
}

// ---- control of one stage under the affine policy ----------------------------------------------
// (ac, dc) = u_nom + alpha k + K dz clamped to the box of the node at (th, v); dz = (ex, ey, eth, ev, dap, ddp) is the
// deviation from the nominal state and the previous stage's control change.  Returns the steering terms of dc.
template <typename T>
MPC_HD Steer<T> policy_control(const T (&Kr)[12], T f0, T f1, T alpha, T ex, T ey, T eth, T ev, T dap, T ddp, bool open_loop,
                               T th, T v, T dt, T ua, T ud, T& ac, T& dc) {
  T da = alpha * f0 + Kr[0] * ex + Kr[1] * ey + Kr[2] * eth + Kr[3] * ev + Kr[4] * dap + Kr[5] * ddp;
  T dd = alpha * f1 + Kr[6] * ex + Kr[7] * ey + Kr[8] * eth + Kr[9] * ev + Kr[10] * dap + Kr[11] * ddp;
  if (open_loop) { da = T(0); dd = T(0); }
  const Box<T> bx = control_box(th, v, dt);
  ac = clamp_(ua + da, bx.lo_a, bx.hi_a);
  dc = ud + dd;
  return clamp_steer(bx, dc, false);
}

// ---- closed-loop forward pass -----------------------------------------------------------------
// Rolls the dynamics forward under the affine policy u = u_nom + alpha k + K dz, clamped to the
// node's control box, for NA step lengths AT ONCE (independent dependency chains: the kernel is
// latency bound, so the second candidate is almost free and the gains are loaded once).
// commit (NA == 1 only): overwrite (X, U) in place with the new trajectory.
// with_cost = false skips the objective (the commit of an accepted trial already knows it).
// open_loop = true ignores the stored policy (du = 0): the first rollout of a problem, whose gain slots
// hold whatever the previous problem left there.
// J[a] = objective, maxdu[a] = max |u_new - u_old| over the horizon.
template <typename T, int NA, typename SL>
MPC_HD void forward_pass(const SolverConfig& cfg, const ProblemScalars<T>& p, const RefTab<T>& ref,
                         const SL& sl, const T* alpha, bool commit, bool with_cost, bool open_loop, T* J, T* maxdu) {
  const int N = cfg.N;
  const T dt = T(cfg.dt);
  T x[NA], y[NA], th[NA], v[NA], ap[NA], dp[NA], dap[NA], ddp[NA];
#pragma unroll
  for (int a = 0; a < NA; ++a) {
    x[a] = sl.X(0, 0); y[a] = sl.X(0, 1); th[a] = sl.X(0, 2); v[a] = sl.X(0, 3);
    ap[a] = dp[a] = dap[a] = ddp[a] = T(0);
    J[a] = T(0); maxdu[a] = T(0);
  }
  for (int k = 0; k < N; ++k) {
    const T xn = sl.X(k, 0), yn = sl.X(k, 1), thn = sl.X(k, 2), vn = sl.X(k, 3);
    const T ua = sl.U(k, 0), ud = sl.U(k, 1);
    T f0, f1, Kr[12];
    sl.load_gains(k, f0, f1, Kr);
    if constexpr (NA == 2) {
      // both candidates' controls first, then their stage costs as one packed evaluation, then their Euler steps
      T ac[2], dc[2];
      Steer<T> st[2];
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        st[a] = policy_control(Kr, f0, f1, alpha[a], x[a] - xn, y[a] - yn, th[a] - thn, v[a] - vn, dap[a], ddp[a],
                               open_loop, th[a], v[a], dt, ua, ud, ac[a], dc[a]);
        dap[a] = ac[a] - ua; ddp[a] = dc[a] - ud;
        maxdu[a] = max_(maxdu[a], max_(abs_(dap[a]), abs_(ddp[a])));
      }
      if (with_cost) {
        const Pair<T> c = stage_cost2(cfg, p, ref, sl, k, Pair<T>{x[0], x[1]}, Pair<T>{y[0], y[1]}, Pair<T>{th[0], th[1]},
                                      Pair<T>{v[0], v[1]}, Pair<T>{ac[0], ac[1]}, Pair<T>{dc[0], dc[1]}, Pair<T>{ap[0], ap[1]},
                                      Pair<T>{dp[0], dp[1]});
        const Pair<T> Js = add2(Pair<T>{J[0], J[1]}, c);
        J[0] = Js.a; J[1] = Js.b;
      }
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        euler_step(x[a], y[a], th[a], v[a], ac[a], st[a], dt);
        ap[a] = ac[a]; dp[a] = dc[a];
      }
    } else {
#pragma unroll
      for (int a = 0; a < NA; ++a) {
        T ac, dc;
        const Steer<T> st = policy_control(Kr, f0, f1, alpha[a], x[a] - xn, y[a] - yn, th[a] - thn, v[a] - vn, dap[a], ddp[a],
                                           open_loop, th[a], v[a], dt, ua, ud, ac, dc);
        dap[a] = ac - ua; ddp[a] = dc - ud;
        maxdu[a] = max_(maxdu[a], max_(abs_(dap[a]), abs_(ddp[a])));
        if (with_cost) J[a] += stage_cost(cfg, p, ref, sl, k, x[a], y[a], th[a], v[a], ac, dc, ap[a], dp[a], (T*)nullptr);
        if (NA == 1 && commit) {
          sl.X(k, 0) = x[a]; sl.X(k, 1) = y[a]; sl.X(k, 2) = th[a]; sl.X(k, 3) = v[a];
          sl.U(k, 0) = ac; sl.U(k, 1) = dc;
        }
        euler_step(x[a], y[a], th[a], v[a], ac, st, dt);
        ap[a] = ac; dp[a] = dc;
      }
    }
  }
  if (NA == 1 && commit) { sl.X(N, 0) = x[0]; sl.X(N, 1) = y[0]; sl.X(N, 2) = th[0]; sl.X(N, 3) = v[0]; }
}

// The control that the commit sweep forward_pass<T, 1>(alpha, commit) would store in U(0), without the sweep: the same
// operations on the same operands (the state deviations x - x of stage 0 included), so the same bits, inf / NaN gains too.
template <typename T, typename SL>
MPC_HD void first_control(const SolverConfig& cfg, const SL& sl, T alpha, T& ac, T& dc) {
  const T x = sl.X(0, 0), y = sl.X(0, 1), th = sl.X(0, 2), v = sl.X(0, 3);
  T f0, f1, Kr[12];
  sl.load_gains(0, f0, f1, Kr);
  policy_control(Kr, f0, f1, alpha, x - x, y - y, th - th, v - v, T(0), T(0), false, th, v, T(cfg.dt), sl.U(0, 0), sl.U(0, 1),
                 ac, dc);
}

// status bits returned per problem
enum : int {
  kStatusConverged = 0,
  kStatusMaxIter = 1,        // iteration cap hit (the iterate is still returned, like the reference's print-only failure path pure_mpc.py:303-305)
  kStatusLineSearchFail = 2, // no acceptable step at maximum regularisation
  kStatusNaN = 4,
  kStatusInfeasibleStart = 8, // s0 violates a state bound (the reference NLP is infeasible, SURVEY A.3)
  kStatusStalled = 16,        // objective stopped improving over a window while the steps were still large
  kStatusKink = 32            // settled on a kink of the clamped dynamics: objective stationary to kink_tol over a window with
                              // steps below 10 tol_step, but the un-damped Newton test cannot fire there (not certified)
};

// ---- start portfolio ------------------------------------------------------------------------------
// The NLP is multi-modal (steering costs 0.01, the Euler slip model admits zig-zag minima, 1/d^2 obstacle
// potentials): which local optimum a descent method reaches depends on its path.  Start 0 is the reference's
// own cold start (zero controls, agents/pure_mpc.py:244).  The others are of two kinds:
//   path-following   roll the model forward steering at the path point `look` rows ahead of the stage's own
//                    (the steering angle that turns the heading onto it within the step, clamped to the node box)
//                    with the acceleration that reaches the stage's reference speed within the step (kAccRef) or
//                    full braking (kAccBrake);
//   pulse            a constant acceleration with a short constant steering pulse;
//   slalom           path-following up to the last row of the path, then full steering alternating right / left every
//                    stage.  Past the end of the 85-point path (ego_index + N > 84) the reference point freezes while
//                    the reference speed does not, and the optimum is such a slalom (DESIGN.md 5); no descent from a
//                    smooth start finds it.
// Start 1 is the path-following start for problems whose horizon stays on the path and the slalom for the others;
// start 3 is a pulse for the former and the path-following start for the latter: the first two starts already hold the
// most useful one of each kind of problem, the first four hold the same set for every problem as a fixed table would.
// Picked greedily from 33 candidates by how often they reach a lower optimum than the starts before them on a
// 1024-problem tuning set and checked on a separate hold-out set (tools/experiments/start_selection.py).
// MpcConfig.n_starts of them are solved per problem and the lowest objective wins.
constexpr int kMaxStarts = 8;
enum : int { kStartPulse = 0, kStartPath = 1, kStartPathOrSlalom = 2, kStartPulseOrPath = 3 };
enum : int { kAccRef = 0, kAccBrake = 1 };
struct StartSpec { int kind; float a, d; int n; };    // pulse: (a, d, stages of the pulse); path: (acc mode in n, look-ahead in d)
MPC_HD StartSpec start_spec(int st) {
  switch (st) {
    case 1: return {kStartPathOrSlalom, 0.f, 1.f, kAccRef};
    case 2: return {kStartPath, 0.f, 1.f, kAccBrake};
    case 3: return {kStartPulseOrPath, 0.f, 0.4f, 3};
    case 4: return {kStartPath, 0.f, 2.f, kAccRef};
    case 5: return {kStartPulse, -5.f, -0.4f, 3};
    case 6: return {kStartPath, 0.f, 3.f, kAccRef};
    case 7: return {kStartPulse, 0.f, 0.2f, 3};
    default: return {kStartPulse, 0.f, 0.f, 0};
  }
}
MPC_HD float atan2_(float y, float x) { return atan2f(y, x); }
MPC_HD double atan2_(double y, double x) { return atan2(y, x); }
template <typename T, typename SL>
MPC_HD void apply_start(const SolverConfig& cfg, const ProblemScalars<T>& p, const RefTab<T>& ref, const SL& sl, int st) {
  const StartSpec sp = start_spec(st);
  const int k_end = kNRef - 1 - p.ego_index;            // first stage whose reference row is the frozen last one
  const bool off_path = k_end < cfg.N;
  const bool slalom = sp.kind == kStartPathOrSlalom && off_path;
  if (sp.kind == kStartPulse || (sp.kind == kStartPulseOrPath && !off_path)) {
    for (int k = 0; k < cfg.N; ++k) { sl.U(k, 0) = T(sp.a); sl.U(k, 1) = k < sp.n ? T(sp.d) : T(0); }
    return;
  }
  const T dt = T(cfg.dt);
  const int look = sp.kind == kStartPulseOrPath ? 1 : int(sp.d);
  const bool brake = sp.kind == kStartPath && sp.n == kAccBrake;
  T x = sl.X(0, 0), y = sl.X(0, 1), th = sl.X(0, 2), v = sl.X(0, 3);
  for (int k = 0; k < cfg.N; ++k) {
    const Box<T> bx = control_box(th, v, dt);
    T a = brake ? -Lim<T>::a_max() : (ref_speed_at(p, k) - v) * rcp_(dt);
    a = clamp_(clamp_(a, -Lim<T>::a_max(), Lim<T>::a_max()), bx.lo_a, bx.hi_a);
    T sb;
    if (slalom && k >= k_end) {
      sb = ((k - k_end) & 1) ? sb_max<T>() : -sb_max<T>();
    } else {
      const RefPoint<T> r = ref_point(ref, p, k + look);
      const T ex = r.x - x, ey = r.y - y;
      T dth = ((ex * ex + ey * ey > T(1e-6)) ? atan2_(ey, ex) : r.h) - th;
      if (dth > Lim<T>::th_max()) dth -= T(2) * Lim<T>::th_max();
      if (dth < -Lim<T>::th_max()) dth += T(2) * Lim<T>::th_max();
      const T gain = dt * max_(v, T(1e-3)) * T(1.0 / 2.5);
      sb = clamp_(dth * rcp_(gain), -sb_max<T>(), sb_max<T>());
    }
    const T d = delta_of_sinbeta(clamp_(sb, bx.sb_lo, bx.sb_hi));
    sl.U(k, 0) = a; sl.U(k, 1) = d;
    euler_step(x, y, th, v, a, steer_terms(d, false), dt);
  }
}

// ---- per-thread solver state -------------------------------------------------------------------
template <typename T> struct SolveState {
  T J, mu, hs;
  T J_mark;               // objective at the last progress checkpoint
  T md_last;              // max |du| of the last accepted step
  int iter, status, trials, fails;
  bool done;
};

// Cold start (pure_mpc.py:244: zero controls).  The initial rollout is the commit pass in open-loop mode,
// so there is one rollout code path: solve_init, then forward_pass<T,1>(commit, with_cost, open_loop),
// then solve_init_finish with its objective.
template <typename T, typename SL>
MPC_HD void solve_init(const SolverConfig& cfg, const SL& sl, SolveState<T>& s) {
  for (int k = 0; k < cfg.N; ++k) {
    sl.U(k, 0) = T(0); sl.U(k, 1) = T(0);
    if (k > 0) { sl.X(k, 0) = T(0); sl.X(k, 1) = T(0); sl.X(k, 2) = T(0); sl.X(k, 3) = T(0); }   // 0 * stale memory could be NaN
  }
  s.mu = T(0); s.hs = T(1);
  s.md_last = T(1e30);
  s.iter = 0; s.status = 0; s.trials = 0; s.fails = 0; s.done = false;
  T v0 = sl.X(0, 3), th0 = sl.X(0, 2);
  if (v0 < Lim<T>::v_min() || v0 > Lim<T>::v_max() || abs_(th0) > Lim<T>::th_max() * T(1.000001)) s.status |= kStatusInfeasibleStart;
}
template <typename T> MPC_HD void solve_init_finish(SolveState<T>& s, T J0) {
  s.J = J0;
  s.J_mark = J0;
}

template <typename T> struct Eps;
template <> struct Eps<float> { static MPC_HD float v() { return 1.1920929e-7f; } };
template <> struct Eps<double> { static MPC_HD double v() { return 2.220446049250313e-16; } };


// Armijo test with a floor at the rounding noise of the objective: once the predicted decrease
// is below what the scalar type can resolve, a step that does not make the objective
// measurably worse is accepted (termination is then decided on the step size).
template <typename T> MPC_HD bool accept_step(T J, T Jn, T expected) {
  T noise = T(32) * Eps<T>::v() * (abs_(J) + T(1));
  if (!(Jn == Jn)) return false;
  if (Jn <= J + T(1e-4) * expected) return true;
  return (expected > -noise) && (Jn <= J + noise);
}

// Line search: ONE pass of two candidates (alpha, alpha/4).  A second pass (1/16, 1/64 ...) rescued only
// ~3 % of the iterations but, because a warp waits for its slowest lane, was executed in almost every
// trip: dropping it costs 0.4 % converged problems and saves 22 % of the launch (profiles/r01_solve_kernel_history.md).
#ifndef MPC_LS_NA
#define MPC_LS_NA 2
#endif

#ifndef MPC_LS_RATIO
#define MPC_LS_RATIO 0.25
#endif
#ifndef MPC_LS_PASSES
#define MPC_LS_PASSES 1
#endif
// Levenberg schedule: accepted step -> mu * MPC_MU_DEC (0 below 1e-3), rejected step -> max(mu * MPC_MU_INC, MPC_MU_MIN).
// (A bracketing controller -- bisect in log space between the last rejected and the last accepted damping -- was
//  measured on the golden sets in round 2: same convergence, slightly more iterations; not kept.)
#ifndef MPC_MU_DEC
#define MPC_MU_DEC 0.1
#endif
#ifndef MPC_MU_INC
#define MPC_MU_INC 30
#endif
#ifndef MPC_MU_MIN
#define MPC_MU_MIN 3
#endif
constexpr int kLineSearchPasses = MPC_LS_PASSES;
constexpr int kStallWindow = 6;        // iterations between progress checkpoints
constexpr float kConvDecrease = 2.5e-7f;   // predicted relative decrease of the last Newton step at convergence

// bookkeeping after a line search; sets s.done when converged or failed.
//   (a) converged (status 0): the un-damped full Newton step is accepted, smaller than tol_step, and its predicted
//   decrease is below kConvDecrease relative (a step of 1e-4 can still be worth 3e-5 of the objective when the ego sits
//   centimetres from an obstacle and the curvature of 1000/d^2 is ~1e9: such a solve takes one more Newton step);
//   (b) settled on a kink (kStatusKink): over a window of kStallWindow iterations the objective improved by less than
//   kink_tol relative (floored at the rounding noise of the scalar type) while the last accepted step was below
//   10 tol_step.  This is how the method ends on points that sit on a kink of the clamped dynamics (a control on its
//   constant limit whose node bound becomes active at the same point): the smooth model of either side overshoots,
//   damped steps converge linearly onto the kink, and test (a) can never fire there.  Such points are near-optimal but
//   can usually still be improved a little (median 0.2 % of the cost) by moving ALONG the kink (a coordinated change of
//   several stages that a stage-wise active set cannot represent), so the flag is kept apart from (a).
template <typename T>
MPC_HD void after_line_search(const SolverConfig& cfg, SolveState<T>& s, bool accepted, T alpha, T Jn, T maxdu, T expected) {
  s.iter++;
  if (accepted) {
    s.J = Jn;
    s.md_last = maxdu;
    // a small step only proves stationarity when it is the un-damped Newton step
    if (alpha == T(1) && s.mu == T(0) && maxdu < T(cfg.tol_step) && -expected <= T(kConvDecrease) * (abs_(Jn) + T(1))) s.done = true;
    s.mu = s.mu > T(1e-3) ? s.mu * T(MPC_MU_DEC) : T(0);
  } else {
    s.fails++;
    s.mu = max_(s.mu * T(MPC_MU_INC), T(MPC_MU_MIN));
    if (s.mu > T(1e9)) { s.status |= kStatusLineSearchFail; s.done = true; }
  }
  if (!s.done && s.iter % kStallWindow == 0) {
    const T gain = s.J_mark - s.J;
    const T noise = T(4) * Eps<T>::v() * (abs_(s.J) + T(1));
    if (gain <= max_(T(cfg.kink_tol) * (abs_(s.J) + T(1)), noise) && s.md_last < T(10) * T(cfg.tol_step)) {
      s.status |= kStatusKink; s.done = true;          // (b) settled on a kink
    } else if (gain <= T(cfg.stall_tol) * (abs_(s.J) + T(1))) {
      s.status |= kStatusStalled; s.done = true;       // no progress, but the steps are not small either
    }
    s.J_mark = s.J;
  }
  if (!s.done && s.iter >= cfg.max_iter) { s.status |= kStatusMaxIter; s.done = true; }
}

// one line-search pass: tries alpha and alpha/2 together.  On success `alpha` holds the accepted step
// length and (Jacc, mdacc) its objective and step size; otherwise alpha is divided by 4 for the next pass.
template <typename T, typename SL>
MPC_HD bool line_search_pass(const SolverConfig& cfg, const ProblemScalars<T>& p, const RefTab<T>& ref,
                             const SL& sl, SolveState<T>& s, T d1, T d2, T& alpha, T& Jacc, T& mdacc) {
#if MPC_LS_NA == 1
  T Jt, mt;
  forward_pass<T, 1, SL>(cfg, p, ref, sl, &alpha, false, true, false, &Jt, &mt);
  s.trials += 1;
  if (accept_step(s.J, Jt, alpha * d1 + alpha * alpha * d2)) { Jacc = Jt; mdacc = mt; return true; }
#else
  T al[2] = {alpha, alpha * T(MPC_LS_RATIO)}, Jt[2], mt[2];
  forward_pass<T, 2, SL>(cfg, p, ref, sl, al, false, true, false, Jt, mt);
  s.trials += 2;
  if (accept_step(s.J, Jt[0], al[0] * d1 + al[0] * al[0] * d2)) { alpha = al[0]; Jacc = Jt[0]; mdacc = mt[0]; return true; }
  if (accept_step(s.J, Jt[1], al[1] * d1 + al[1] * al[1] * d2)) { alpha = al[1]; Jacc = Jt[1]; mdacc = mt[1]; return true; }
#endif
  alpha = alpha * T(MPC_LS_RATIO) * T(MPC_LS_RATIO);
  return false;
}

// straight-line single-problem driver (host harness; the kernel runs the same sub-steps with
// a warp-synchronous line search, see mpc_kernels.cu)
template <typename T, typename SL>
MPC_HD void solve_one(const SolverConfig& cfg, const ProblemScalars<T>& p, const RefTab<T>& ref,
                      const SL& sl, SolveState<T>& s, const float* u_init = nullptr, int start = 0) {
  {
    solve_init(cfg, sl, s);
    if (start > 0) apply_start<T>(cfg, p, ref, sl, start);
    if (u_init && start == 0) for (int k = 0; k < cfg.N; ++k) { sl.U(k, 0) = T(u_init[2 * k]); sl.U(k, 1) = T(u_init[2 * k + 1]); }
    T a1 = T(1), J0, md0;
    forward_pass<T, 1, SL>(cfg, p, ref, sl, &a1, true, true, true, &J0, &md0);
    solve_init_finish(s, J0);
  }
  while (!s.done) {
    T d1, d2;
    backward_pass(cfg, p, ref, sl, s.mu, s.hs, &d1, &d2);
    T alpha = T(1), Jn = T(0), md = T(0);
    bool acc = false;
    for (int t = 0; t < kLineSearchPasses && !acc; ++t) {
      acc = line_search_pass(cfg, p, ref, sl, s, d1, d2, alpha, Jn, md);
    }
    if (acc) { T Jc, mdc; forward_pass<T, 1, SL>(cfg, p, ref, sl, &alpha, true, false, false, &Jc, &mdc); }
#if defined(MPC_TRACE) && !defined(__CUDA_ARCH__)
    printf("it %d J %.9g d1 %.4g d2 %.4g alpha %.4g acc %d Jn %.9g maxdu %.3g mu %.3g hs %g u0 %.6f %.6f\n", s.iter, (double)s.J,
           (double)d1, (double)d2, (double)alpha, (int)acc, (double)Jn, (double)md, (double)s.mu, (double)s.hs, (double)sl.U(0, 0), (double)sl.U(0, 1));
#endif
    after_line_search(cfg, s, acc, alpha, Jn, md, alpha * d1 + alpha * alpha * d2);
  }
  if (!(s.J == s.J)) s.status |= kStatusNaN;
}

}  // namespace mpcb
