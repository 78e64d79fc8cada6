// Internal (not installed) declarations shared by the translation units of libmpcb200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mpc_b200.h"
#include "mpc_core.cuh"

namespace mpcb {

// mutable view of the handle's parsed-problem workspace (same layout as MpcProblemBatch)
struct BatchWs {
  float* s0;
  int32_t* ego_index;
  float* w_speed;
  float* w_control;
  float* w_diff;
  float* vr_a;
  float* vr_slope;
  float* vr_b;
  int32_t* vr_n;
  uint8_t* is_collide;
  int32_t* n_obs;
  float* obstacles;
};

struct PrepareParams {
  const float* obs;            // [B][V][8]
  const float* ref_speed;      // [B] or null (NaN = none)
  const float* weights;        // [B][3] or null
  const uint8_t* reset_mask;   // [B] or null
  MpcLatchState latch;         // pointers may be null when collision_check == 0
  MpcCollisionOut col;         // any pointer may be null
  BatchWs ws;
  int B, V, M, N;              // B = environments of the call = stride of the SoA outputs
  int first, count;            // this launch handles environments [first, first + count)
  double dt;
  float w_speed, w_control, w_diff;
  int collision_check;
};

// launches (defined in mpc_prepare.cu, compiled with -fmad=false so that FP64 results are
// bit-identical to the numpy oracle's un-fused arithmetic)
cudaError_t launch_prepare(const PrepareParams& p, cudaStream_t stream);
cudaError_t upload_ref_table_prepare();

// defined in mpc_solve.cu
// Candidate results of the start portfolio: work item w = start * B + problem.  Filled by the solve kernels when
// n_starts > 1, reduced to MpcSolveOut by k_select (lowest objective wins, ties to the lowest start).
struct SolveCand {
  float* cost;            // [S * B]
  float* u0;              // [S * B][2]
  int32_t* status;        // [S * B]
  int32_t* iters;         // [S * B]
  float* U;               // [S * B][N][2]
};
// Adaptive portfolio (mpc_set_adaptive_starts): the base items (start < n_starts) are the tickets below B * n_starts;
// the lane that finishes a problem's last base start appends that problem's extra items (starts n_starts..max_starts-1)
// to `extra` when the base objectives disagree, and a larger ticket t takes slot t - B * n_starts of that list.
// Zeroed / preset to -1 before every launch.
struct AdaptiveQueue {
  int* base_done;         // [B] base starts finished per problem; ends at n_starts, or n_starts + 1 when extended
  int* extra;             // [(max_starts - n_starts) * B] extra items (start * B + problem), -1 = not written yet
  int* reserve;           // slots of `extra` reserved so far
  int* items_done;        // base items finished (each increments it after its publishing)
  int max_starts;         // 0 = fixed portfolio
  float rel_gap;
};
struct SolveLaunch {
  SolverConfig cfg;
  MpcProblemBatch batch;
  MpcSolveOut out;
  int B;                  // problems
  int n_starts;           // work items = B * n_starts (base items of the adaptive portfolio)
  SolveCand cand;         // used when n_starts > 1
  int* work_counter;      // device, zeroed before launch
  const float* u_init;    // [B][N][2] warm start of start 0, or null
  int threads_per_block;
  int grid;
  size_t smem_bytes;
  int use_tmem;           // gains in tensor memory (k_solve_tmem) instead of shared memory (k_solve)
  AdaptiveQueue aq;       // aq.max_starts > 0: adaptive portfolio
  float* start_cost;      // adaptive: [max_starts][ld] per-start objectives or null
  uint8_t* extended;      // adaptive: [B] or null
  int ld;                 // row stride of start_cost
};
cudaError_t launch_solve(const SolveLaunch& s, cudaStream_t stream);
cudaError_t launch_rollout_cost(const SolverConfig& cfg, const MpcProblemBatch& batch, int B, const float* U,
                                float* X_out, float* cost6, float* total, cudaStream_t stream);
cudaError_t upload_ref_table_solve();
cudaError_t launch_fma_peak(float* sink, int iters, int grid, int block, cudaStream_t stream);
size_t solve_smem_bytes(int N, int M, int tpb);
size_t solve_smem_bytes_tmem(int N, int M, int tpb);
bool tmem_layout_fits(int N, int tpb);
cudaError_t launch_solve_tmem(const SolveLaunch& s, cudaStream_t stream);
cudaError_t launch_select(const SolveLaunch& s, cudaStream_t stream);
cudaError_t launch_select_adaptive(const SolveLaunch& s, cudaStream_t stream);

}  // namespace mpcb
