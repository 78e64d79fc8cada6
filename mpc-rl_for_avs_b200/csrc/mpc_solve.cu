// mpc_solve.cu -- the hot kernels: one persistent launch solves the whole batch of MPC problems.
//
// Mapping (B200, 148 SMs, 227 KB shared memory + 256 KB tensor memory / SM, 64 K registers / SM):
//   * one problem per THREAD.  The horizon recursion (rollout, Riccati sweep) is serial in k and
//     the per-stage blocks are 6x6 / 2x6 -- nothing a warp or a tensor core could share -- so the
//     parallelism that exists is across problems and lanes stay full for the dominant work.
//   * the per-problem horizon arrays U, X and the obstacle tracks (156 words at H=20, M=8) live in a
//     strided shared-memory slot file (slot*blockDim + tid: bank-conflict free); the bf16-packed gains +
//     feed-forward (140 words) live in TENSOR MEMORY in k_solve_tmem (this path issues no MMA, so TMEM is
//     free capacity) and in the same slot file in k_solve; the value-function block (21+6 floats) in
//     registers.
//   * persistent grid, one block per SM.  Iteration counts differ by 10x between problems, so a thread
//     that finishes pulls the next problem index from a global counter (after a static first wave)
//     instead of idling until its warp's slowest problem ends.
//   * one trip of the loop = backward sweep, ONE line-search sweep of two candidates (alpha, alpha/4),
//     commit sweep; a rejected step raises the Levenberg damping for the next trip.
//   * the tail of a launch (k_solve_tmem, 192/256 threads): the surviving problems are packed into the
//     lowest warps, and the freed lanes run the trips the sequential algorithm would run after 1, 2, ...
//     rejections side by side (see the comments at kCompact / kSpec).
//   * HBM traffic is the compulsory ~0.3 KB per problem: these kernels are FP32-issue / latency bound.
#include <mutex>

#include "mpc_internal.h"

#include "ref_table.inc"

namespace mpcb {

__constant__ float c_hsc[kNRef * kRefStride];     // heading, sin h, cos h
__constant__ double c_xy[kNRef * 2];               // path positions, FP64

cudaError_t upload_ref_table_solve() {
  float h[kNRef * kRefStride];
  double xy[kNRef * 2];
  for (int j = 0; j < kNRef; ++j) {
    xy[2 * j] = kRefPath[j][0];
    xy[2 * j + 1] = kRefPath[j][1];
    h[j * kRefStride + 0] = (float)kRefPath[j][3];
    h[j * kRefStride + 1] = (float)sin(kRefPath[j][3]);
    h[j * kRefStride + 2] = (float)cos(kRefPath[j][3]);
  }
  cudaError_t e = cudaMemcpyToSymbol(c_hsc, h, sizeof(h));
  if (e != cudaSuccess) return e;
  return cudaMemcpyToSymbol(c_xy, xy, sizeof(xy));
}

constexpr int kTabFloats = kNRef * 2 * 2 + kNRef * kRefStride + 1;   // FP64 xy (as 2 floats each) + hsc, padded to even
size_t solve_smem_bytes(int N, int M, int tpb) {
  return (size_t)(kTabFloats + slots_per_problem(N, M, true) * tpb) * sizeof(float);
}

// block-shared copy of the path tables at the head of dynamic shared memory
__device__ __forceinline__ RefTab<float> stage_tables(float* smem) {
  double* xy = reinterpret_cast<double*>(smem);
  float* hsc = smem + kNRef * 2 * 2;
#pragma unroll 1
  for (int i = threadIdx.x; i < kNRef * 2; i += blockDim.x) xy[i] = c_xy[i];
#pragma unroll 1
  for (int i = threadIdx.x; i < kNRef * kRefStride; i += blockDim.x) hsc[i] = c_hsc[i];
  __syncthreads();
  return RefTab<float>{hsc, xy};
}

template <typename SL>
__device__ __forceinline__ void load_problem(const MpcProblemBatch& b, int B, int i, const SolverConfig& cfg,
                                             ProblemScalars<float>& p, const SL& sl, const RefTab<float>& ref) {
  p.ego_index = b.ego_index[i];
  int n = b.n_obs ? b.n_obs[i] : 0;
  p.n_obs = n < cfg.M ? n : cfg.M;
  p.is_collide = b.is_collide ? b.is_collide[i] : 0;
  p.w_speed = b.w_speed[i];
  p.w_control = b.w_control[i];
  p.w_diff = b.w_diff[i];
  p.vr_a = b.vr_a[i];
  p.vr_slope = b.vr_slope[i];
  p.vr_b = b.vr_b[i];
  p.vr_n = b.vr_n[i];
  p.x0 = (double)b.s0[i];
  p.y0 = (double)b.s0[(size_t)B + i];
  sl.X(0, 0) = 0.f; sl.X(0, 1) = 0.f;                       // positions are relative to the ego start
  sl.X(0, 2) = b.s0[(size_t)2 * B + i];
  sl.X(0, 3) = b.s0[(size_t)3 * B + i];
#pragma unroll 1
  for (int m = 0; m < cfg.M; ++m) {
    if (b.obstacles) {
      sl.O(m, 0) = (float)((double)b.obstacles[((size_t)m * 4 + 0) * B + i] - p.x0);
      sl.O(m, 1) = (float)((double)b.obstacles[((size_t)m * 4 + 1) * B + i] - p.y0);
      sl.O(m, 2) = b.obstacles[((size_t)m * 4 + 2) * B + i];
      sl.O(m, 3) = b.obstacles[((size_t)m * 4 + 3) * B + i];
    } else {
      sl.O(m, 0) = 0.f; sl.O(m, 1) = 0.f; sl.O(m, 2) = 0.f; sl.O(m, 3) = 0.f;
    }
  }
  if constexpr (SL::kRefStaged) {
#pragma unroll 1
    for (int k = 0; k < cfg.N; ++k) {
      int j = p.ego_index + k;
      j = j < kNRef - 1 ? j : kNRef - 1;
      sl.R(k, 0) = (float)(ref.xy[2 * j] - p.x0);
      sl.R(k, 1) = (float)(ref.xy[2 * j + 1] - p.y0);
    }
  }
}

// work item -> (problem, start); first controls of a fresh item (cold start pure_mpc.py:244, a portfolio start, or the
// opt-in warm start for start 0)
template <typename SL>
__device__ __forceinline__ void begin_item(const SolverConfig& cfg, const MpcProblemBatch& batch, int B, int idx, const float* __restrict__ u_init,
                                           ProblemScalars<float>& p, const SL& sl, SolveState<float>& s, const RefTab<float>& ref) {
  const int st = idx / B, pb = idx - st * B;
  load_problem(batch, B, pb, cfg, p, sl, ref);
  solve_init(cfg, sl, s);
  if (st > 0) {
    apply_start<float>(cfg, p, ref, sl, st);
  } else if (u_init) {                  // opt-in warm start: the first rollout clamps it into the node boxes
#pragma unroll 1
    for (int k = 0; k < cfg.N; ++k) {
      sl.U(k, 0) = u_init[((size_t)pb * cfg.N + k) * 2];
      sl.U(k, 1) = u_init[((size_t)pb * cfg.N + k) * 2 + 1];
    }
  }
}
// result of a finished item: straight to the caller's arrays (one start) or to the candidate arrays (portfolio)
template <typename SL>
__device__ __forceinline__ void finish_item(const SolverConfig& cfg, const MpcSolveOut& out, const SolveCand& cand, int n_starts, int idx,
                                            const SL& sl, SolveState<float>& s) {
  if (!(s.J == s.J)) s.status |= kStatusNaN;
  if (n_starts == 1) {
    out.actions[2 * (size_t)idx] = sl.U(0, 0);
    out.actions[2 * (size_t)idx + 1] = sl.U(0, 1);
    if (out.status) out.status[idx] = s.status;
    if (out.iters) out.iters[idx] = s.iter;
    if (out.cost) out.cost[idx] = s.J;
    if (out.U)
#pragma unroll 1
      for (int k = 0; k < cfg.N; ++k) {
        out.U[((size_t)idx * cfg.N + k) * 2] = sl.U(k, 0);
        out.U[((size_t)idx * cfg.N + k) * 2 + 1] = sl.U(k, 1);
      }
  } else {
    cand.u0[2 * (size_t)idx] = sl.U(0, 0);
    cand.u0[2 * (size_t)idx + 1] = sl.U(0, 1);
    cand.status[idx] = s.status;
    cand.iters[idx] = s.iter;
    cand.cost[idx] = s.J;
    if (out.U)
#pragma unroll 1
      for (int k = 0; k < cfg.N; ++k) {
        cand.U[((size_t)idx * cfg.N + k) * 2] = sl.U(k, 0);
        cand.U[((size_t)idx * cfg.N + k) * 2 + 1] = sl.U(k, 1);
      }
  }
}

// ---- adaptive portfolio: the work queue grows while the launch runs ---------------------------------------------
// A ticket below B * S0 is base item `ticket`; a larger one reads slot ticket - B * S0 of the extra list.  Returns the
// item, kTicketPending (slot not written yet and base items still running: poll again next trip -- never spin inside a
// trip, the sweeps are warp-collective) or kTicketEmpty (definitively nothing left).
constexpr int kTicketPending = -1, kTicketEmpty = -2;
__device__ __forceinline__ int ld_acquire(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ int poll_ticket(const AdaptiveQueue& aq, int B, int n_starts, int ticket) {
  const int n_base = B * n_starts;
  if (ticket < n_base) return ticket;
  const int slot = ticket - n_base;
  if (slot >= (aq.max_starts - n_starts) * B) return kTicketEmpty;   // past the list's capacity: can never be written
  // every base item publishes before it counts itself finished: once all are counted, every reserved slot is written
  const bool all_done = ld_acquire(aq.items_done) == n_base;
  const int v = ld_acquire(aq.extra + slot);
  if (v >= 0) return v;
  if (all_done && slot >= ld_acquire(aq.reserve)) return kTicketEmpty;
  return kTicketPending;
}
// After a base item's candidate is written: count it; the lane that finishes a problem's last base start reads the
// S0 objectives and appends starts S0..S-1 when any is not finite or max - min > rel_gap * max(|min|, 1).
__device__ __forceinline__ void publish_base(const AdaptiveQueue& aq, const SolveCand& cand, int B, int n_starts, int idx) {
  const int b = idx % B;
  __threadfence();                                           // the candidate before the count
  if (atomicAdd(aq.base_done + b, 1) == n_starts - 1) {
    __threadfence();
    float lo = __ldcg(cand.cost + b), hi = lo;               // L2: the other starts were written by other SMs
    bool finite = isfinite(lo);
    for (int st = 1; st < n_starts; ++st) {
      const float J = __ldcg(cand.cost + (size_t)st * B + b);
      finite = finite && isfinite(J);
      lo = fminf(lo, J); hi = fmaxf(hi, J);
    }
    if (!finite || hi - lo > aq.rel_gap * fmaxf(fabsf(lo), 1.f)) {
      const int n_extra = aq.max_starts - n_starts;
      const int r = atomicAdd(aq.reserve, n_extra);
      for (int j = 0; j < n_extra; ++j) aq.extra[r + j] = (n_starts + j) * B + b;
      aq.base_done[b] = n_starts + 1;                        // marks the problem extended for k_select_adaptive
      __threadfence();
    }
  }
  atomicAdd(aq.items_done, 1);
}

// One trip of the loop = [fetch] -> backward sweep -> line-search passes -> commit sweep -> bookkeeping,
// each with exactly ONE call site so the kernel body stays near the instruction-cache size (the
// first profile showed 2.3 stall cycles per issued instruction waiting for instructions).
// A freshly fetched problem joins at the commit sweep (its first rollout is the commit under a zero
// policy) and starts iterating on the next trip.
// kAdaptive: the adaptive portfolio (AdaptiveQueue); a lane whose ticket is not resolved yet is `pending`.
template <int TPB, bool kAdaptive>
__global__ void __launch_bounds__(TPB, 1)
k_solve(const SolverConfig cfg, const MpcProblemBatch batch, const MpcSolveOut out, const int B, int* __restrict__ work_counter,
        const float* __restrict__ u_init, const int n_starts, const SolveCand cand, const AdaptiveQueue aq) {
  extern __shared__ __align__(16) float smem[];
  const RefTab<float> ref = stage_tables(smem);
  using SL = Slots<float, true, TPB>;
  const SL sl{smem + kTabFloats + threadIdx.x, TPB, cfg.N, cfg.M};
  const unsigned full = 0xffffffffu;

  ProblemScalars<float> p;
  SolveState<float> s;
  int idx = -1;
  bool active = false, fresh = false, need_fetch = true, pending = false;

  for (;;) {
    if (need_fetch) {
      need_fetch = false;
      idx = atomicAdd(work_counter, 1);
      if constexpr (kAdaptive) {
        pending = true;
      } else {
        active = idx < B * n_starts;
        if (active) {
          begin_item(cfg, batch, B, idx, u_init, p, sl, s, ref);
          fresh = true;
        }
      }
    }
    if constexpr (kAdaptive) {
      if (pending) {
        const int r = poll_ticket(aq, B, n_starts, idx);
        if (r != kTicketPending) {
          pending = false;
          active = r >= 0;
          if (active) {
            idx = r;
            begin_item(cfg, batch, B, idx, u_init, p, sl, s, ref);
            fresh = true;
          }
        }
      }
    }
    if (!__any_sync(full, active || pending)) break;
    float d1 = 0.f, d2 = 0.f, alpha = 1.f, Jn = 0.f, md = 0.f;
    bool acc = false;
    const bool run = active && !fresh;
    if (run) backward_pass(cfg, p, ref, sl, s.mu, s.hs, &d1, &d2);
    for (int t = 0; t < kLineSearchPasses; ++t) {
      const bool need = run && !acc;
      if (!__any_sync(full, need)) break;
      if (need) acc = line_search_pass(cfg, p, ref, sl, s, d1, d2, alpha, Jn, md);
    }
    if (active && (fresh || acc)) {      // commit sweep; only a fresh problem still needs its objective
      float Jc, mdc;
      forward_pass<float, 1, SL>(cfg, p, ref, sl, &alpha, true, fresh, fresh, &Jc, &mdc);
      if (fresh) Jn = Jc;
    }
    if (active) {
      if (fresh) {
        solve_init_finish(s, Jn);
        fresh = false;
      } else {
        after_line_search(cfg, s, acc, alpha, Jn, md, alpha * d1 + alpha * alpha * d2);
        if (s.done) {
          finish_item(cfg, out, cand, n_starts, idx, sl, s);
          if constexpr (kAdaptive) if (idx < B * n_starts) publish_base(aq, cand, B, n_starts, idx);
          active = false;
          need_fetch = true;
        }
      }
    }
  }
}

// ---- variant with the gains in tensor memory -----------------------------------------------------
// Same trip structure; differences forced by the warp-collective tcgen05.ld/st:
//   * every sweep is executed by all 32 lanes whenever ANY lane needs it.  Lanes without work compute on
//     whatever their slots hold (finite loops only, results discarded); their TMEM stores land in their own
//     cells.  Under SIMT those lanes were waiting anyway.
//   * shared memory per problem is 156 words -> up to 352 problems fit an SM (192 with gains in shared memory);
//     256 are used, which leaves room for the scratch of the tail compaction.
constexpr int kTmemColsPerStage = 8;
// Tail compaction (k_solve_tmem, blocks of <= 256 threads): scratch for moving up to kCompactMax problems'
// register state between lanes, plus one counter per warp.
constexpr int kCompactMax = 128, kCompactWords = 28, kCompactTpbMax = 256;
static constexpr int compact_floats(int tpb) { return (tpb > 128 && tpb <= kCompactTpbMax) ? kCompactMax * kCompactWords + 16 : 0; }
size_t solve_smem_bytes_tmem(int N, int M, int tpb) {
  return (size_t)(kTabFloats + 4 + slots_per_problem_tmem(N, M) * tpb + compact_floats(tpb)) * sizeof(float);
}
bool tmem_layout_fits(int N, int tpb) {
  const int warps = tpb / 32, per_quarter = (warps + 3) / 4;
  return kTmemColsPerStage * N * per_quarter <= 512;
}

#ifndef MPC_COMPACT
#define MPC_COMPACT 1
#endif
#ifndef MPC_SPEC
#define MPC_SPEC 1
#endif
#ifndef MPC_SPEC_LANES
#define MPC_SPEC_LANES 128     // lanes the speculating groups may occupy: 4 warps = one per scheduler
#endif
#ifndef MPC_SPEC_MAXK
#define MPC_SPEC_MAXK 8
#endif

template <int TPB, bool kAdaptive>
__global__ void __launch_bounds__(TPB, 1)
k_solve_tmem(const SolverConfig cfg, const MpcProblemBatch batch, const MpcSolveOut out, const int B, int* __restrict__ work_counter,
             const float* __restrict__ u_init, const int n_starts, const SolveCand cand, const AdaptiveQueue aq) {
  extern __shared__ __align__(16) float smem[];
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + kTabFloats);
  const int warp = threadIdx.x >> 5;
  if (warp == 0) {          // one warp allocates all 512 columns for the CTA (one CTA per SM)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n"
                 :: "r"((uint32_t)__cvta_generic_to_shared(s_tmem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  const RefTab<float> ref = stage_tables(smem);            // contains the __syncthreads()
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tmem_base = *s_tmem;
  using SL = SlotsTmem<TPB>;
  float* const slot0 = smem + kTabFloats + 4;
  SL sl{slot0 + threadIdx.x,
        tmem_base + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(kTmemColsPerStage * cfg.N * (warp >> 2)), cfg.N, cfg.M};
  const unsigned full = 0xffffffffu;
  constexpr bool kCompact = (MPC_COMPACT != 0) && TPB > 128 && TPB <= kCompactTpbMax;   // <= 4 warps already have a scheduler each
  uint32_t* const scratch = reinterpret_cast<uint32_t*>(slot0 + slots_per_problem_tmem(cfg.N, cfg.M) * TPB);
  int* const s_wcnt = reinterpret_cast<int*>(scratch + kCompactMax * kCompactWords);
  int live_warps = TPB / 32;                                // warps that may still hold problems (block-uniform)
  constexpr bool kSpec = kCompact && (MPC_SPEC != 0);
  int spec_k = 1, spec_j = 0;                               // lanes per problem (block-uniform) / this lane's index in its group
  bool drained = false;                                     // some lane of the block found the queue empty (block-uniform)
  bool saw_empty = false;                                   // this lane did

  ProblemScalars<float> p;
  p.x0 = 0.0; p.y0 = 0.0; p.ego_index = 0; p.n_obs = 0; p.is_collide = 0;
  p.w_speed = 1.f; p.w_control = 1.f; p.w_diff = 1.f; p.vr_a = 0.f; p.vr_slope = 0.f; p.vr_b = 0.f; p.vr_n = 0;
  SolveState<float> s;
  s.J = 0.f; s.mu = 0.f; s.hs = 1.f; s.J_mark = 0.f; s.md_last = 1e30f; s.iter = 0; s.status = 0; s.trials = 0; s.fails = 0; s.done = true;
  int idx = -1;
  bool active = false, fresh = false, need_fetch = true, first_wave = true;
  bool pending = false;                                     // kAdaptive: holds a ticket whose slot is not written yet

  for (;;) {
    if (need_fetch) {
      need_fetch = false;
      // first wave: a static, evenly spread assignment (problem b + grid * t to thread t of block b) -- no storm of
      // atomics on one counter, and a small launch lands in the lowest lanes of every block; later: the shared queue
      idx = first_wave ? (int)(blockIdx.x + gridDim.x * threadIdx.x) : (int)(gridDim.x * TPB) + atomicAdd(work_counter, 1);
      first_wave = false;
      if constexpr (kAdaptive) {
        pending = true;
      } else {
        active = idx < B * n_starts;
        if (active) {
          begin_item(cfg, batch, B, idx, u_init, p, sl, s, ref);
          fresh = true;
        } else {
          saw_empty = true;
        }
      }
    }
    if constexpr (kAdaptive) {
      if (pending) {
        const int r = poll_ticket(aq, B, n_starts, idx);
        if (r != kTicketPending) {
          pending = false;
          active = r >= 0;
          if (active) {
            idx = r;
            begin_item(cfg, batch, B, idx, u_init, p, sl, s, ref);
            fresh = true;
          } else {
            saw_empty = true;
          }
        }
      }
    }
    __syncwarp();
    if (kCompact) {
      // ---- one block barrier per trip: count the running problems; once the queue is drained and they fit
      // into half of the warps that still hold any, move them to the lowest lanes.  The launch ends with a
      // tail of a few long problems per SM, and one trip of a warp takes 71 us with two warps per scheduler
      // but 56 us with one: packing the survivors into <= 4 (then 2, then 1) warps shortens every trip of
      // the tail.  A problem's state is 25 registers + its shared-memory column (re-pointed, not copied);
      // the gains in TMEM are rebuilt by the next backward sweep, so nothing else moves.
      //
      // Speculation (kSpec): when <= 64 (<= 32) problems are left, each gets 2 (4) adjacent lanes.  Lane j of a
      // group runs the SAME trip with the damping the sequential algorithm would use after j rejected steps
      // (mu -> max(30 mu, 3), X and U untouched by a rejection), so one trip decides up to 4 sequential trips:
      // the first lane whose step is accepted wins, the rejections before it are replayed in the bookkeeping,
      // the winner commits.  Same iterates, same iteration counts, same results -- fewer trips in the tail,
      // where ~40 % of the trips of the slow problems are rejections.
      const int n_active = __syncthreads_count(active && spec_j == 0);
      // kAdaptive: a pending lane keeps the block alive, and compaction (which reassigns lanes and would drop its
      // ticket) waits until no lane is pending -- once some lane saw the queue empty, pending lanes resolve next trip
      bool settled;
      if constexpr (kAdaptive) {
        const bool any_pending = __syncthreads_or(pending) != 0;
        if (n_active == 0 && !any_pending) break;
        if (!drained) drained = __syncthreads_or(saw_empty) != 0;
        settled = drained && !any_pending;
      } else {
        if (n_active == 0) break;
        if (!drained) drained = __syncthreads_or(saw_empty) != 0;     // every decision below is taken on barrier results only
        settled = drained;
      }
      int k_new = 1;
      if (kSpec && settled) {                                // largest power of two with n_active * k <= MPC_SPEC_LANES, at most MPC_SPEC_MAXK
        while (2 * k_new <= MPC_SPEC_MAXK && n_active * 2 * k_new <= MPC_SPEC_LANES) k_new *= 2;
      }
      if (k_new < spec_k) k_new = spec_k;
      const int warps_new = (n_active * k_new + 31) >> 5;
      if (settled && n_active <= kCompactMax && (k_new > spec_k || (live_warps > 1 && 2 * warps_new <= live_warps))) {
        const bool lead = active && spec_j == 0;
        const unsigned bal = __ballot_sync(full, lead);
        const int lane = threadIdx.x & 31;
        if (lane == 0) s_wcnt[warp] = __popc(bal);
        __syncthreads();
        if (lead) {
          int r = __popc(bal & ((1u << lane) - 1u));
          for (int w = 0; w < warp; ++w) r += s_wcnt[w];
          uint32_t* q = scratch + r * kCompactWords;
          q[0] = (uint32_t)__double2loint(p.x0); q[1] = (uint32_t)__double2hiint(p.x0);
          q[2] = (uint32_t)__double2loint(p.y0); q[3] = (uint32_t)__double2hiint(p.y0);
          q[4] = (uint32_t)p.ego_index; q[5] = (uint32_t)p.n_obs; q[6] = (uint32_t)p.is_collide;
          q[7] = __float_as_uint(p.w_speed); q[8] = __float_as_uint(p.w_control); q[9] = __float_as_uint(p.w_diff);
          q[10] = __float_as_uint(p.vr_a); q[11] = __float_as_uint(p.vr_slope); q[12] = __float_as_uint(p.vr_b);
          q[13] = (uint32_t)p.vr_n;
          q[14] = __float_as_uint(s.J); q[15] = __float_as_uint(s.mu);    // s.hs is the constant 1 in every kernel: kept out of memory so it still folds
          q[16] = __float_as_uint(s.md_last);
          q[17] = __float_as_uint(s.J_mark); q[18] = (uint32_t)s.iter; q[19] = (uint32_t)s.status;
          q[20] = (uint32_t)s.trials; q[21] = (uint32_t)s.fails;
          q[22] = (uint32_t)idx; q[23] = fresh ? 1u : 0u;
          q[24] = (uint32_t)(sl.base - slot0);               // the shared-memory column that holds U, X, obstacles
        }
        __syncthreads();
        const int group = (int)threadIdx.x / k_new;
        spec_k = k_new;
        spec_j = (int)threadIdx.x % k_new;
        active = group < n_active;
        fresh = false;
        if (active) {
          const uint32_t* q = scratch + group * kCompactWords;
          p.x0 = __hiloint2double((int)q[1], (int)q[0]); p.y0 = __hiloint2double((int)q[3], (int)q[2]);
          p.ego_index = (int)q[4]; p.n_obs = (int)q[5]; p.is_collide = (int)q[6];
          p.w_speed = __uint_as_float(q[7]); p.w_control = __uint_as_float(q[8]); p.w_diff = __uint_as_float(q[9]);
          p.vr_a = __uint_as_float(q[10]); p.vr_slope = __uint_as_float(q[11]); p.vr_b = __uint_as_float(q[12]);
          p.vr_n = (int)q[13];
          s.J = __uint_as_float(q[14]); s.mu = __uint_as_float(q[15]); s.md_last = __uint_as_float(q[16]);
          s.J_mark = __uint_as_float(q[17]); s.iter = (int)q[18]; s.status = (int)q[19];
          s.trials = (int)q[20]; s.fails = (int)q[21]; s.done = false;
          idx = (int)q[22]; fresh = q[23] != 0u;
          sl.base = slot0 + q[24];
        } else {
          spec_j = 0;                                        // idle lanes must not look like followers of a group
        }
        live_warps = warps_new;
        __syncthreads();                                     // scratch may be rewritten by the next compaction
      }
      if (warp >= live_warps) continue;                      // parked: nothing to sweep, back to the barrier
    } else {
      if (!__any_sync(full, active || pending)) break;
    }
    float d1 = 0.f, d2 = 0.f, alpha = 1.f, Jn = 0.f, md = 0.f;
    bool ok = false;
    const bool run = active && !fresh;
    const bool any_run = __any_sync(full, run);
    const int trials0 = s.trials;
    if (any_run) {                                          // all 32 lanes sweep; only `run` lanes keep the result
      float mu_j = s.mu;
      if (kSpec) for (int i = 0; i < spec_j; ++i) mu_j = max_(mu_j * float(MPC_MU_INC), float(MPC_MU_MIN));   // damping after i rejected steps (after_line_search)
      backward_pass(cfg, p, ref, sl, mu_j, s.hs, &d1, &d2);
      __syncwarp();
      ok = line_search_pass(cfg, p, ref, sl, s, d1, d2, alpha, Jn, md) && run;
      __syncwarp();
    }
    // ---- bookkeeping of the solver state (before the commit sweep: it only needs the line-search results)
    bool commit_me = false;
    if (!kSpec || spec_k == 1) {
      if (run) { after_line_search(cfg, s, ok, alpha, Jn, md, alpha * d1 + alpha * alpha * d2); commit_me = ok; }
    } else {
      const unsigned okmask = __ballot_sync(full, ok);
      const int gbase = (threadIdx.x & 31) & ~(spec_k - 1);
      const unsigned gm = (okmask >> gbase) & ((1u << spec_k) - 1u);
      const int w = gm ? (__ffs((int)gm) - 1) : spec_k;     // first speculative lane whose step was accepted
      const int src = gbase + (w < spec_k ? w : 0);
      const float a_w = __shfl_sync(full, alpha, src), J_w = __shfl_sync(full, Jn, src), md_w = __shfl_sync(full, md, src);
      const float ex_w = __shfl_sync(full, alpha * d1 + alpha * alpha * d2, src);
      if (run) {
        int t = 0;
        bool reached = false;
        for (; t < spec_k && !s.done; ++t) {
          if (t == w) { after_line_search(cfg, s, true, a_w, J_w, md_w, ex_w); reached = true; ++t; break; }
          after_line_search(cfg, s, false, 1.f, 0.f, 0.f, 0.f);
        }
        s.trials = trials0 + MPC_LS_NA * t;
        commit_me = reached && spec_j == w;
      }
    }
    const bool do_commit = active && (fresh ? spec_j == 0 : commit_me);
    float Jc = 0.f, mdc = 0.f;
    if (__any_sync(full, do_commit)) {
      forward_pass<float, 1, SL>(cfg, p, ref, sl, &alpha, do_commit, fresh, fresh, &Jc, &mdc);
      __syncwarp();
    }
    if (kSpec && spec_k > 1) Jc = __shfl_sync(full, Jc, (threadIdx.x & 31) & ~(spec_k - 1));   // the group leader did the first rollout
    if (active) {
      if (fresh) {
        solve_init_finish(s, Jc);
        fresh = false;
      } else if (s.done) {
        if (spec_j == 0) {
          finish_item(cfg, out, cand, n_starts, idx, sl, s);
          if constexpr (kAdaptive) if (idx < B * n_starts) publish_base(aq, cand, B, n_starts, idx);
        }
        active = false;
        spec_j = 0;
        need_fetch = !drained;                               // nothing left to fetch once a lane of the block saw the queue empty
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" :: "r"(tmem_base) : "memory");
}

// The opt-in dynamic shared memory size is a per-DEVICE function attribute: remember what was set per device (a
// process may hold handles on several GPUs) and per kernel instantiation; guarded for concurrent host threads.
constexpr int kMaxDevices = 64;
struct SmemOptIn {
  std::mutex m;
  size_t configured[kMaxDevices] = {};
  template <typename K> cudaError_t ensure(K kernel, size_t bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> g(m);
    if (dev < 0 || dev >= kMaxDevices || bytes > configured[dev]) {
      e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
      if (e != cudaSuccess) return e;
      if (dev >= 0 && dev < kMaxDevices) configured[dev] = bytes;
    }
    return cudaSuccess;
  }
};

template <int TPB, bool kAdaptive> static cudaError_t launch_solve_tmem_t(const SolveLaunch& s, cudaStream_t stream) {
  static SmemOptIn opt;
  cudaError_t e = opt.ensure(k_solve_tmem<TPB, kAdaptive>, s.smem_bytes);
  if (e != cudaSuccess) return e;
  k_solve_tmem<TPB, kAdaptive><<<s.grid, TPB, s.smem_bytes, stream>>>(s.cfg, s.batch, s.out, s.B, s.work_counter, s.u_init,
                                                                       s.n_starts, s.cand, s.aq);
  return cudaGetLastError();
}
template <int TPB> static cudaError_t launch_solve_tmem_t(const SolveLaunch& s, cudaStream_t stream) {
  return s.aq.max_starts > 0 ? launch_solve_tmem_t<TPB, true>(s, stream) : launch_solve_tmem_t<TPB, false>(s, stream);
}

cudaError_t launch_solve_tmem(const SolveLaunch& s, cudaStream_t stream) {
  switch (s.threads_per_block) {
    case 128: return launch_solve_tmem_t<128>(s, stream);
    case 192: return launch_solve_tmem_t<192>(s, stream);
    case 256: return launch_solve_tmem_t<256>(s, stream);
    case 288: return launch_solve_tmem_t<288>(s, stream);
    case 320: return launch_solve_tmem_t<320>(s, stream);
    case 352: return launch_solve_tmem_t<352>(s, stream);
    case 384: return launch_solve_tmem_t<384>(s, stream);
    default: return cudaErrorInvalidConfiguration;
  }
}

template <int TPB, bool kAdaptive> static cudaError_t launch_solve_t(const SolveLaunch& s, cudaStream_t stream) {
  // handles with different horizon / obstacle counts share the kernel: raise the opt-in limit as needed
  static SmemOptIn opt;
  cudaError_t e = opt.ensure(k_solve<TPB, kAdaptive>, s.smem_bytes);
  if (e != cudaSuccess) return e;
  k_solve<TPB, kAdaptive><<<s.grid, TPB, s.smem_bytes, stream>>>(s.cfg, s.batch, s.out, s.B, s.work_counter, s.u_init, s.n_starts,
                                                                  s.cand, s.aq);
  return cudaGetLastError();
}
template <int TPB> static cudaError_t launch_solve_t(const SolveLaunch& s, cudaStream_t stream) {
  return s.aq.max_starts > 0 ? launch_solve_t<TPB, true>(s, stream) : launch_solve_t<TPB, false>(s, stream);
}

cudaError_t launch_solve(const SolveLaunch& s, cudaStream_t stream) {
  switch (s.threads_per_block) {
    case 32: return launch_solve_t<32>(s, stream);
    case 64: return launch_solve_t<64>(s, stream);
    case 96: return launch_solve_t<96>(s, stream);
    case 128: return launch_solve_t<128>(s, stream);
    case 160: return launch_solve_t<160>(s, stream);
    case 192: return launch_solve_t<192>(s, stream);
    default: return cudaErrorInvalidConfiguration;
  }
}

// ---- start portfolio: per problem, the candidate with the lowest objective wins (ties: lowest start) --------------
__global__ void __launch_bounds__(256)
k_select(const int B, const int S, const int N, const SolveCand cand, const MpcSolveOut out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  int best = 0, it = 0;
  float Jb = 0.f;
  for (int st = 0; st < S; ++st) {
    const float J = cand.cost[(size_t)st * B + b];
    it += cand.iters[(size_t)st * B + b];
    if (st == 0 || J < Jb) { Jb = J; best = st; }       // NaN never wins over a finite start 0; a NaN start 0 is replaced by any finite one
    if (st > 0 && !(Jb == Jb) && J == J) { Jb = J; best = st; }
  }
  const size_t w = (size_t)best * B + b;
  out.actions[2 * (size_t)b] = cand.u0[2 * w];
  out.actions[2 * (size_t)b + 1] = cand.u0[2 * w + 1];
  if (out.status) out.status[b] = cand.status[w];
  if (out.iters) out.iters[b] = it;                     // total over the starts: the work this problem cost
  if (out.cost) out.cost[b] = Jb;
  if (out.U)
    for (int k = 0; k < 2 * N; ++k) out.U[(size_t)b * 2 * N + k] = cand.U[w * 2 * N + k];
}

cudaError_t launch_select(const SolveLaunch& s, cudaStream_t stream) {
  k_select<<<(s.B + 255) / 256, 256, 0, stream>>>(s.B, s.n_starts, s.cfg.N, s.cand, s.out);
  return cudaGetLastError();
}

// Adaptive portfolio: the same selection over starts 0..S0-1, plus S0..S-1 for the problems the solve kernel extended
// (base_done[b] == S0 + 1).  start_cost [S][ld] (NaN for starts that did not run) and extended [B] are optional.
__global__ void __launch_bounds__(256)
k_select_adaptive(const int B, const int S0, const int N, const SolveCand cand, const MpcSolveOut out, const AdaptiveQueue aq,
                  float* __restrict__ start_cost, uint8_t* __restrict__ extended, const int ld) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const bool ext = aq.base_done[b] > S0;
  const int S = ext ? aq.max_starts : S0;
  int best = 0, it = 0;
  float Jb = 0.f;
  for (int st = 0; st < S; ++st) {
    const float J = cand.cost[(size_t)st * B + b];
    it += cand.iters[(size_t)st * B + b];
    if (st == 0 || J < Jb) { Jb = J; best = st; }
    if (st > 0 && !(Jb == Jb) && J == J) { Jb = J; best = st; }
    if (start_cost) start_cost[(size_t)st * ld + b] = J;
  }
  if (start_cost)
    for (int st = S; st < aq.max_starts; ++st) start_cost[(size_t)st * ld + b] = __int_as_float(0x7fc00000);
  if (extended) extended[b] = ext ? 1 : 0;
  const size_t w = (size_t)best * B + b;
  out.actions[2 * (size_t)b] = cand.u0[2 * w];
  out.actions[2 * (size_t)b + 1] = cand.u0[2 * w + 1];
  if (out.status) out.status[b] = cand.status[w];
  if (out.iters) out.iters[b] = it;
  if (out.cost) out.cost[b] = Jb;
  if (out.U)
    for (int k = 0; k < 2 * N; ++k) out.U[(size_t)b * 2 * N + k] = cand.U[w * 2 * N + k];
}

cudaError_t launch_select_adaptive(const SolveLaunch& s, cudaStream_t stream) {
  k_select_adaptive<<<(s.B + 255) / 256, 256, 0, stream>>>(s.B, s.n_starts, s.cfg.N, s.cand, s.out, s.aq, s.start_cost, s.extended, s.ld);
  return cudaGetLastError();
}

// ---- K1 parity entry: rollout + six cost components for given controls -----------------------
__global__ void __launch_bounds__(64)
k_rollout_cost(const SolverConfig cfg, const MpcProblemBatch batch, const int B, const float* __restrict__ U,
               float* __restrict__ X_out, float* __restrict__ cost6, float* __restrict__ total) {
  extern __shared__ __align__(16) float smem[];
  const RefTab<float> ref = stage_tables(smem);
  const Slots<float, true> sl{smem + kTabFloats + threadIdx.x, (int)blockDim.x, cfg.N, cfg.M};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B; i += gridDim.x * blockDim.x) {
    ProblemScalars<float> p;
    load_problem(batch, B, i, cfg, p, sl, ref);
    for (int k = 0; k < cfg.N; ++k) {
      sl.U(k, 0) = U[((size_t)i * cfg.N + k) * 2];
      sl.U(k, 1) = U[((size_t)i * cfg.N + k) * 2 + 1];
    }
    float comp[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float J = rollout_nominal(cfg, p, ref, sl, comp);
    // final_state component (agents/pure_mpc.py:195-202: note the (y + y_ref) sign), reported only
    comp[2] = final_state_component(cfg, p, ref, sl);
    for (int c = 0; c < 6; ++c) cost6[(size_t)i * 6 + c] = comp[c];
    total[i] = J;
    for (int k = 0; k <= cfg.N; ++k) {
      float* xo = X_out + ((size_t)i * (cfg.N + 1) + k) * 4;
      xo[0] = (float)(p.x0 + (double)sl.X(k, 0));
      xo[1] = (float)(p.y0 + (double)sl.X(k, 1));
      xo[2] = sl.X(k, 2);
      xo[3] = sl.X(k, 3);
    }
  }
}

cudaError_t launch_rollout_cost(const SolverConfig& cfg, const MpcProblemBatch& batch, int B, const float* U,
                                float* X_out, float* cost6, float* total, cudaStream_t stream) {
  const int tpb = 64;
  size_t smem = solve_smem_bytes(cfg.N, cfg.M, tpb);
  cudaError_t e = cudaFuncSetAttribute(k_rollout_cost, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  int grid = (B + tpb - 1) / tpb;
  if (grid > 148 * 8) grid = 148 * 8;
  if (grid < 1) grid = 1;
  k_rollout_cost<<<grid, tpb, smem, stream>>>(cfg, batch, B, U, X_out, cost6, total);
  return cudaGetLastError();
}

// ---- FP32 FMA micro-benchmark: the roofline denominator for this (non-tensor, non-HBM) path ----
__global__ void __launch_bounds__(256)
k_fma_peak(float* __restrict__ sink, const int iters) {
  float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f;
  float a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
  const float m = 0.999f, c = 1e-3f;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
      a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
    }
  }
  float r = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (r == 123.456f) sink[0] = r;   // never true; keeps the loop alive
}

cudaError_t launch_fma_peak(float* sink, int iters, int grid, int block, cudaStream_t stream) {
  k_fma_peak<<<grid, block, 0, stream>>>(sink, iters);
  return cudaGetLastError();
}

}  // namespace mpcb
