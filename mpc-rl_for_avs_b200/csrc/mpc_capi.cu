// mpc_capi.cu -- extern "C" boundary of libmpcb200.so (see include/mpc_b200.h).
// Host side only: argument checks, workspace ownership, launch sequencing, error text.
// No exception crosses the ABI; there is no CPU compute path anywhere in this library.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "mpc_internal.h"
#include "ref_path.h"

using namespace mpcb;

static thread_local std::string g_create_error;

constexpr int kHostChunks = 4;      // pieces of the observation upload in mpc_predict_host

struct MpcHandle {
  MpcConfig cfg;
  SolverConfig scfg;
  int device = 0;
  int max_batch = 0;
  int sm_count = 0, cc_major = 0, cc_minor = 0, smem_optin = 0;
  int tpb = 0, grid = 0;
  size_t smem = 0;
  int use_tmem = 0;
  int tpb_small = 0;              // TMEM kernel: largest block the per-launch choice may use (<= 256)
  bool tpb_forced = false;
  // device workspace
  void* ref_block = nullptr;      // the path tables built from cfg.dt (RefTables), uploaded once by mpc_create
  RefTables tables{};
  void* ws_block = nullptr;       // one allocation carved into the BatchWs arrays
  BatchWs ws{};
  int* work_counter = nullptr;
  int n_starts = 1;
  SolveCand cand{};                // candidate results of the start portfolio (n_starts > 1)
  int cand_starts = 0;             // starts the candidate arrays hold per problem (n_starts, or max_starts once adaptive)
  // opt-in adaptive portfolio (mpc_set_adaptive_starts); max_starts = 0: off
  int max_starts = 0;
  float rel_gap = 0.f;
  int* aq_block = nullptr;         // [2 + max_batch + (aq_starts - n_starts) * max_batch]: reserve, items_done, base_done, extra
  int aq_starts = 0;
  float* start_cost = nullptr;     // borrowed
  uint8_t* extended = nullptr;     // borrowed
  const float* u_init = nullptr;   // opt-in warm start (device, borrowed)
  float* sink = nullptr;
  // host-call staging (mpc_predict_host)
  float* d_obs = nullptr; float* d_ref_speed = nullptr; float* d_weights = nullptr; uint8_t* d_reset = nullptr;
  float* d_actions = nullptr; int32_t* d_status = nullptr; int32_t* d_iters = nullptr; float* d_cost = nullptr;
  int32_t* d_mem = nullptr; int32_t* d_memo = nullptr; uint8_t* d_iscol = nullptr;
  uint8_t* d_flags = nullptr; int32_t* d_cidx = nullptr; int32_t* d_egoidx = nullptr; int32_t* d_stop = nullptr;
  uint8_t* d_deg = nullptr; float* d_cpt = nullptr;
  cudaStream_t host_stream = nullptr;
  cudaStream_t copy_stream = nullptr;        // uploads of mpc_predict_host
  cudaEvent_t copy_done[kHostChunks] = {};
  // measurement
  int64_t launches = 0;
  bool timing = false;
  std::vector<cudaEvent_t> ev_prepare, ev_solve;   // start/stop pairs
  std::string err;
};

static int fail(MpcHandle* h, int code, const char* what, cudaError_t e = cudaSuccess) {
  char buf[512];
  if (e != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
  else snprintf(buf, sizeof buf, "%s", what);
  if (h) h->err = buf; else g_create_error = buf;
  return code;
}

#define CK(h, call)                                                    \
  do {                                                                 \
    cudaError_t e__ = (call);                                          \
    if (e__ != cudaSuccess) return fail((h), MPC_ERR_CUDA, #call, e__); \
  } while (0)

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// dt arrives as a float (0.1f); the reference's dt is the double 1 / policy_frequency (agents/base_agent.py:43)
static double prep_dt(float dt) { return 1.0 / (double)(long long)(1.0 / (double)dt + 0.5); }

extern "C" {

MPC_API const char* mpc_last_error(const MpcHandle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

MPC_API int mpc_destroy(MpcHandle* h) {
  if (!h) return MPC_OK;
  cudaSetDevice(h->device);
  for (auto e : h->ev_prepare) cudaEventDestroy(e);
  for (auto e : h->ev_solve) cudaEventDestroy(e);
  cudaFree(h->ref_block); cudaFree(h->ws_block); cudaFree(h->work_counter); cudaFree(h->sink); cudaFree(h->aq_block);
  cudaFree(h->cand.cost); cudaFree(h->cand.u0); cudaFree(h->cand.status); cudaFree(h->cand.iters); cudaFree(h->cand.U);
  cudaFree(h->d_obs); cudaFree(h->d_ref_speed); cudaFree(h->d_weights); cudaFree(h->d_reset);
  cudaFree(h->d_actions); cudaFree(h->d_status); cudaFree(h->d_iters); cudaFree(h->d_cost);
  cudaFree(h->d_mem); cudaFree(h->d_memo); cudaFree(h->d_iscol);
  cudaFree(h->d_flags); cudaFree(h->d_cidx); cudaFree(h->d_egoidx); cudaFree(h->d_stop); cudaFree(h->d_deg); cudaFree(h->d_cpt);
  if (h->host_stream) cudaStreamDestroy(h->host_stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  for (auto e : h->copy_done) if (e) cudaEventDestroy(e);
  delete h;
  return MPC_OK;
}

MPC_API int mpc_create(const MpcConfig* cfg, int device, int max_batch, MpcHandle** out) {
  if (!cfg || !out) return fail(nullptr, MPC_ERR_BAD_ARG, "mpc_create: null argument");
  *out = nullptr;
  if (cfg->abi_version != MPC_ABI_VERSION) return fail(nullptr, MPC_ERR_BAD_ARG, "mpc_create: abi_version mismatch");
  if (cfg->horizon < 2 || cfg->horizon > 64) return fail(nullptr, MPC_ERR_BAD_ARG, "mpc_create: horizon must be in 2..64");
  if (cfg->vehicles_count < 1 || cfg->vehicles_count - 1 > MPC_MAX_OBSTACLES)
    return fail(nullptr, MPC_ERR_BAD_ARG, "mpc_create: vehicles_count must be in 1..17");
  if (!(cfg->dt > 0.f)) return fail(nullptr, MPC_ERR_BAD_ARG, "mpc_create: dt must be positive");
  if (max_batch < 1) return fail(nullptr, MPC_ERR_BAD_ARG, "mpc_create: max_batch must be >= 1");
  if (cfg->n_starts < 0 || cfg->n_starts > MPC_MAX_STARTS) return fail(nullptr, MPC_ERR_BAD_ARG, "mpc_create: n_starts must be in 0..8");
  {   // dt enters the collision prediction as the double 1 / policy_frequency (agents/base_agent.py:43) and the dynamics
      // as the float itself: both must be the same time step
    const double f = 1.0 / (double)cfg->dt, fr = (double)(long long)(f + 0.5);
    if (fr < 1.0 || (f - fr > 1e-4 * fr) || (fr - f > 1e-4 * fr))
      return fail(nullptr, MPC_ERR_BAD_ARG, "mpc_create: dt must be 1 / (an integer policy frequency)");
  }
  const int n_starts = cfg->n_starts > 0 ? cfg->n_starts : 4;
  if ((long long)max_batch * n_starts > 0x7fffffffLL / 64) return fail(nullptr, MPC_ERR_BAD_ARG, "mpc_create: max_batch * n_starts too large");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return fail(nullptr, MPC_ERR_NO_DEVICE, "mpc_create: no CUDA device (this library has no CPU path)");
  if (device < 0 || device >= ndev) return fail(nullptr, MPC_ERR_BAD_ARG, "mpc_create: device index out of range");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(nullptr, MPC_ERR_NO_DEVICE, "mpc_create: cannot query device");
  if (prop.major != 10) return fail(nullptr, MPC_ERR_NO_DEVICE, "mpc_create: device is not sm_100 (B200); the kernels are built for sm_100a only");

  MpcHandle* h = new (std::nothrow) MpcHandle();
  if (!h) return fail(nullptr, MPC_ERR_CUDA, "mpc_create: out of host memory");
  h->cfg = *cfg;
  h->device = device;
  h->max_batch = max_batch;
  h->n_starts = n_starts;
  h->sm_count = prop.multiProcessorCount;
  h->cc_major = prop.major; h->cc_minor = prop.minor;
  h->smem_optin = (int)prop.sharedMemPerBlockOptin;
  const int N = cfg->horizon, M = cfg->vehicles_count - 1;
  SolverConfig& s = h->scfg;
  s.N = N; s.M = M; s.dt = cfg->dt;
  s.w_distance = cfg->weight_distance; s.w_collision = cfg->weight_collision;
  s.literal_no_collision = cfg->literal_no_collision;
  s.max_iter = cfg->max_iter > 0 ? cfg->max_iter : 60;
  s.tol_step = cfg->tol_step > 0.f ? cfg->tol_step : 1e-4f;
  s.reg_min = cfg->reg_min > 0.f ? cfg->reg_min : 1e-2f;
  s.stall_tol = 0.f;
  s.kink_tol = 1e-7f;

#define CKC(call)                                                                        \
  do {                                                                                   \
    cudaError_t e__ = (call);                                                            \
    if (e__ != cudaSuccess) { fail(nullptr, MPC_ERR_CUDA, #call, e__); mpc_destroy(h); return MPC_ERR_CUDA; } \
  } while (0)

  CKC(cudaSetDevice(device));
  // grid / block.  Default: gains in tensor memory, at most 256 problems (8 warps, two per scheduler) per SM --
  // up to 352 fit at H=20, M=8 and can be forced with threads_per_block, but measured no faster even at 1 M
  // problems per launch; a horizon whose gains do not fit the 512 TMEM columns selects the shared-memory kernel
  // (192 problems / SM).
  int tpb = 0;
  {
    static const int cand[] = {384, 352, 320, 288, 256, 192, 128};
    const int cap = cfg->threads_per_block > 0 ? cfg->threads_per_block : 256;   // 256 is as fast as 352 at 1 M problems and faster below
    for (int c : cand) {
      if (c > cap) continue;
      if (!tmem_layout_fits(N, c)) continue;
      if (solve_smem_bytes_tmem(N, M, c) > (size_t)h->smem_optin) continue;
      if (65536 / c < 160) continue;                       // registers: the kernel needs ~150 per thread
      tpb = c;
      break;
    }
    if (tpb) {
      h->use_tmem = 1; h->tpb = tpb; h->smem = solve_smem_bytes_tmem(N, M, tpb);
      // Measured (profiles/r01_solve_kernel_history.md): 8 warps / SM (2 per scheduler, evenly) is the fastest
      // block up to ~0.5 M problems per launch -- the launch is bounded by the latency of its longest problems,
      // which grows with the number of resident warps; the largest block only pays off when throughput bound.
      h->tpb_forced = cfg->threads_per_block > 0;
      h->tpb_small = tpb < 256 ? tpb : 256;
    }
  }
  if (!h->use_tmem) {
    tpb = cfg->threads_per_block > 0 ? cfg->threads_per_block : 192;
    tpb = (tpb + 31) / 32 * 32;
    if (tpb > 192) tpb = 192;
    while (tpb > 32 && solve_smem_bytes(N, M, tpb) > (size_t)h->smem_optin) tpb -= 32;
    if (solve_smem_bytes(N, M, tpb) > (size_t)h->smem_optin) { fail(nullptr, MPC_ERR_BAD_ARG, "mpc_create: horizon/obstacle count do not fit shared memory"); mpc_destroy(h); return MPC_ERR_BAD_ARG; }
    h->tpb = tpb;
    h->smem = solve_smem_bytes(N, M, tpb);
  }
  int bps = cfg->blocks_per_sm > 0 ? cfg->blocks_per_sm : (int)((size_t)prop.sharedMemPerMultiprocessor / (h->smem + 1024));
  if (bps < 1) bps = 1;
  if (h->use_tmem) bps = 1;                                 // the CTA owns all 512 TMEM columns of its SM
  h->grid = h->sm_count * bps;
  {   // the path is accumulated with v * dt steps (agents/base_agent.py:118-154): each handle holds its own table, so
      // handles with different policy frequencies coexist in one process
    double ref[kNRef][4], seg[kNRef - 1], xy[kNRef * 2];
    float hsc[kNRef * kRefStride];
    build_reference_path(prep_dt(cfg->dt), ref);
    for (int j = 0; j < kNRef; ++j) {
      xy[2 * j] = ref[j][0];
      xy[2 * j + 1] = ref[j][1];
      hsc[j * kRefStride + 0] = (float)ref[j][3];
      hsc[j * kRefStride + 1] = (float)sin(ref[j][3]);
      hsc[j * kRefStride + 2] = (float)cos(ref[j][3]);
    }
    for (int j = 0; j < kNRef - 1; ++j) {
      double dx = ref[j + 1][0] - ref[j][0], dy = ref[j + 1][1] - ref[j][1];
      volatile double xx = dx * dx, yy = dy * dy;       // volatile: no host-side FMA contraction (np.linalg.norm rounds each)
      seg[j] = sqrt(xx + yy);
    }
    const size_t o_seg = sizeof(ref), o_xy = o_seg + sizeof(seg), o_hsc = o_xy + sizeof(xy);
    CKC(cudaMalloc(&h->ref_block, o_hsc + sizeof(hsc)));
    char* tb = (char*)h->ref_block;
    CKC(cudaMemcpy(tb, ref, sizeof(ref), cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(tb + o_seg, seg, sizeof(seg), cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(tb + o_xy, xy, sizeof(xy), cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(tb + o_hsc, hsc, sizeof(hsc), cudaMemcpyHostToDevice));
    h->tables.ref = (const double*)tb;
    h->tables.seg = (const double*)(tb + o_seg);
    h->tables.solve = RefTab<float>{(const float*)(tb + o_hsc), (const double*)(tb + o_xy)};
  }

  // parsed-problem workspace
  const size_t B = (size_t)max_batch;
  size_t off = 0;
  auto carve = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  size_t o_s0 = carve(4 * B * 4), o_ei = carve(B * 4), o_ws = carve(B * 4), o_wc = carve(B * 4), o_wd = carve(B * 4);
  size_t o_va = carve(B * 4), o_vs = carve(B * 4), o_vb = carve(B * 4), o_vn = carve(B * 4), o_ic = carve(B), o_no = carve(B * 4);
  size_t o_ob = carve((size_t)(M > 0 ? M : 1) * 4 * B * 4);
  CKC(cudaMalloc(&h->ws_block, off));
  CKC(cudaMemset(h->ws_block, 0, off));
  char* base = (char*)h->ws_block;
  h->ws.s0 = (float*)(base + o_s0); h->ws.ego_index = (int32_t*)(base + o_ei); h->ws.w_speed = (float*)(base + o_ws);
  h->ws.w_control = (float*)(base + o_wc); h->ws.w_diff = (float*)(base + o_wd); h->ws.vr_a = (float*)(base + o_va);
  h->ws.vr_slope = (float*)(base + o_vs); h->ws.vr_b = (float*)(base + o_vb); h->ws.vr_n = (int32_t*)(base + o_vn);
  h->ws.is_collide = (uint8_t*)(base + o_ic); h->ws.n_obs = (int32_t*)(base + o_no); h->ws.obstacles = (float*)(base + o_ob);
  CKC(cudaMalloc(&h->work_counter, sizeof(int)));
  if (n_starts > 1) {
    const size_t W = B * (size_t)n_starts;
    CKC(cudaMalloc(&h->cand.cost, W * 4));
    CKC(cudaMalloc(&h->cand.u0, W * 8));
    CKC(cudaMalloc(&h->cand.status, W * 4));
    CKC(cudaMalloc(&h->cand.iters, W * 4));
    CKC(cudaMalloc(&h->cand.U, W * (size_t)N * 8));
    h->cand_starts = n_starts;
  }
  CKC(cudaMalloc(&h->sink, 256));
  // staging for the host-buffer entry point
  CKC(cudaMalloc(&h->d_obs, B * cfg->vehicles_count * 8 * 4));
  CKC(cudaMalloc(&h->d_ref_speed, B * 4));
  CKC(cudaMalloc(&h->d_weights, B * 3 * 4));
  CKC(cudaMalloc(&h->d_reset, B));
  CKC(cudaMalloc(&h->d_actions, B * 2 * 4));
  CKC(cudaMalloc(&h->d_status, B * 4));
  CKC(cudaMalloc(&h->d_iters, B * 4));
  CKC(cudaMalloc(&h->d_cost, B * 4));
  CKC(cudaMalloc(&h->d_mem, B * 4));
  CKC(cudaMalloc(&h->d_memo, B * 4));
  CKC(cudaMalloc(&h->d_iscol, B));
  {
    const size_t Mx = (size_t)(M > 0 ? M : 1);
    CKC(cudaMalloc(&h->d_flags, B * Mx));
    CKC(cudaMalloc(&h->d_cidx, B * Mx * 4));
    CKC(cudaMalloc(&h->d_egoidx, B * 4));
    CKC(cudaMalloc(&h->d_stop, B * 4));
    CKC(cudaMalloc(&h->d_deg, B));
    CKC(cudaMalloc(&h->d_cpt, B * Mx * 8));
  }
  CKC(cudaMemset(h->d_mem, 0, B * 4));
  CKC(cudaMemset(h->d_memo, 0xff, B * 4));
  CKC(cudaMemset(h->d_iscol, 0, B));
  CKC(cudaStreamCreateWithFlags(&h->host_stream, cudaStreamNonBlocking));
  CKC(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  for (int c = 0; c < kHostChunks; ++c) CKC(cudaEventCreateWithFlags(&h->copy_done[c], cudaEventDisableTiming));
  CKC(cudaDeviceSynchronize());
#undef CKC
  *out = h;
  return MPC_OK;
}

MPC_API int mpc_device_info(const MpcHandle* h, int* sm_count, int* cc_major, int* cc_minor, int* smem_per_block_optin) {
  if (!h) return MPC_ERR_BAD_ARG;
  if (sm_count) *sm_count = h->sm_count;
  if (cc_major) *cc_major = h->cc_major;
  if (cc_minor) *cc_minor = h->cc_minor;
  if (smem_per_block_optin) *smem_per_block_optin = h->smem_optin;
  return MPC_OK;
}

MPC_API int mpc_workspace_batch(MpcHandle* h, MpcProblemBatch* out) {
  if (!h || !out) return MPC_ERR_BAD_ARG;
  out->s0 = h->ws.s0; out->ego_index = h->ws.ego_index; out->w_speed = h->ws.w_speed; out->w_control = h->ws.w_control;
  out->w_diff = h->ws.w_diff; out->vr_a = h->ws.vr_a; out->vr_slope = h->ws.vr_slope; out->vr_b = h->ws.vr_b;
  out->vr_n = h->ws.vr_n; out->is_collide = h->ws.is_collide; out->n_obs = h->ws.n_obs; out->obstacles = h->ws.obstacles;
  return MPC_OK;
}

static int check_batch(MpcHandle* h, const MpcProblemBatch* b, int B) {
  if (!h) return MPC_ERR_BAD_ARG;
  if (B == 0) return MPC_OK;
  if (!b || B < 0) return fail(h, MPC_ERR_BAD_ARG, "null batch or negative size");
  if (!b->s0 || !b->ego_index || !b->w_speed || !b->w_control || !b->w_diff || !b->vr_a || !b->vr_slope || !b->vr_b || !b->vr_n)
    return fail(h, MPC_ERR_BAD_ARG, "MpcProblemBatch: a required array is null");
  if (h->scfg.M > 0 && h->scfg.w_distance != 0.f && (!b->obstacles || !b->n_obs))
    return fail(h, MPC_ERR_BAD_ARG, "MpcProblemBatch: obstacles/n_obs required when weight_distance != 0");
  return MPC_OK;
}

MPC_API int mpc_rollout_cost(MpcHandle* h, const MpcProblemBatch* batch, int B, const float* U, float* X_out, float* cost6_out,
                     float* total_out, void* stream) {
  int rc = check_batch(h, batch, B);
  if (rc) return rc;
  if (!U || !X_out || !cost6_out || !total_out) return fail(h, MPC_ERR_BAD_ARG, "mpc_rollout_cost: null output/input");
  if (B == 0) return MPC_OK;
  CK(h, cudaSetDevice(h->device));
  CK(h, launch_rollout_cost(h->scfg, h->tables.solve, *batch, B, U, X_out, cost6_out, total_out, (cudaStream_t)stream));
  h->launches += 1;
  return MPC_OK;
}

static int timed_begin(MpcHandle* h, std::vector<cudaEvent_t>& v, cudaStream_t st) {
  if (!h->timing) return MPC_OK;
  cudaEvent_t a, b;
  CK(h, cudaEventCreate(&a));
  CK(h, cudaEventCreate(&b));
  v.push_back(a); v.push_back(b);
  CK(h, cudaEventRecord(a, st));
  return MPC_OK;
}
static int timed_end(MpcHandle* h, std::vector<cudaEvent_t>& v, cudaStream_t st) {
  if (!h->timing) return MPC_OK;
  CK(h, cudaEventRecord(v.back(), st));
  return MPC_OK;
}

// Block size and kernel of one launch.  The launch lasts as long as its slowest SM, and one solver
// iteration takes longer the more warps share an SM's four schedulers, so: spread the batch over all SMs
// first (one block per SM), and only then grow the block.  Both kernels run the same per-problem code and
// store the gains in the same packed form, so the result of a problem does not depend on the choice
// (tests/test_gpu_parity.py::test_result_independent_of_batch_size).
static void pick_solve_launch(const MpcHandle* h, int B /* work items = problems x starts */, SolveLaunch& s) {
  s.threads_per_block = h->tpb; s.smem_bytes = h->smem; s.use_tmem = h->use_tmem;
  const int N = h->scfg.N, M = h->scfg.M;
  const int per_sm = (B + h->sm_count - 1) / h->sm_count;
  int want = (per_sm + 31) / 32 * 32;
  if (!h->tpb_forced) {
    if (!h->use_tmem) {
      if (want < h->tpb) { s.threads_per_block = want; s.smem_bytes = solve_smem_bytes(N, M, want); }
    } else {
      // the 192/256-thread TMEM kernel at every size: a block that gets fewer problems than lanes packs them
      // into its lowest warps on the first trip and gives each 2-8 lanes to speculate with
      int tpb = (want > 128 && want <= 192) ? 192 : 256;
      if (tpb > h->tpb_small) tpb = h->tpb_small;
      s.threads_per_block = tpb; s.smem_bytes = solve_smem_bytes_tmem(N, M, tpb);
    }
  }
  // grid: one block per SM; small launches still spread over all SMs (>= 8 problems per block)
  int need = (B + s.threads_per_block - 1) / s.threads_per_block;
  if (s.use_tmem) { const int spread = (B + 7) / 8; if (spread > need) need = spread; }
  s.grid = need < h->grid ? need : h->grid;
}

MPC_API int mpc_solve_config(const MpcHandle* h, int B, int* gains_in_tmem, int* threads_per_block) {
  if (!h || B < 0) return MPC_ERR_BAD_ARG;
  SolveLaunch s;
  pick_solve_launch(h, B * h->n_starts, s);
  if (gains_in_tmem) *gains_in_tmem = s.use_tmem;
  if (threads_per_block) *threads_per_block = s.threads_per_block;
  return MPC_OK;
}

MPC_API int mpc_solve(MpcHandle* h, const MpcProblemBatch* batch, int B, const MpcSolveOut* out, void* stream) {
  int rc = check_batch(h, batch, B);
  if (rc) return rc;
  if (!out || !out->actions) return fail(h, MPC_ERR_BAD_ARG, "mpc_solve: actions output is required");
  if (B == 0) return MPC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  CK(h, cudaSetDevice(h->device));
  CK(h, cudaMemsetAsync(h->work_counter, 0, sizeof(int), st));
  SolveLaunch s;
  if (B > h->max_batch && h->n_starts > 1) return fail(h, MPC_ERR_TOO_LARGE, "mpc_solve: B exceeds max_batch of mpc_create");
  s.cfg = h->scfg; s.tables = h->tables.solve; s.batch = *batch; s.out = *out; s.B = B; s.work_counter = h->work_counter;
  s.n_starts = h->n_starts; s.cand = h->cand;
  s.u_init = h->u_init;
  s.aq = AdaptiveQueue{};
  s.start_cost = nullptr; s.extended = nullptr; s.ld = h->max_batch;
  if (h->max_starts > 0) {   // per-launch queue state: counters zeroed, extra list preset to -1 (all on the stream: capturable)
    const size_t n_extra = (size_t)(h->max_starts - h->n_starts) * B;
    s.aq.reserve = h->aq_block; s.aq.items_done = h->aq_block + 1; s.aq.base_done = h->aq_block + 2;
    s.aq.extra = h->aq_block + 2 + h->max_batch;
    s.aq.max_starts = h->max_starts; s.aq.rel_gap = h->rel_gap;
    s.start_cost = h->start_cost; s.extended = h->extended;
    CK(h, cudaMemsetAsync(h->aq_block, 0, (2 + (size_t)B) * sizeof(int), st));
    CK(h, cudaMemsetAsync(s.aq.extra, 0xff, n_extra * sizeof(int), st));
  }
  pick_solve_launch(h, B * h->n_starts, s);
  if ((rc = timed_begin(h, h->ev_solve, st))) return rc;
  CK(h, s.use_tmem ? launch_solve_tmem(s, st) : launch_solve(s, st));
  h->launches += 1;
  if (h->max_starts > 0) { CK(h, launch_select_adaptive(s, st)); h->launches += 1; }
  else if (h->n_starts > 1) { CK(h, launch_select(s, st)); h->launches += 1; }
  if ((rc = timed_end(h, h->ev_solve, st))) return rc;
  return MPC_OK;
}

// launches k_prepare for environments [first, first + count) of a call of B environments
static int prepare_range(MpcHandle* h, const float* obs, const float* ref_speed, const float* weights, const uint8_t* reset_mask,
                         const MpcLatchState* latch, int B, int first, int count, const MpcCollisionOut* col, cudaStream_t st) {
  PrepareParams p{};
  p.obs = obs; p.ref_speed = ref_speed; p.weights = weights; p.reset_mask = reset_mask;
  if (latch) p.latch = *latch;
  if (col) p.col = *col;
  p.ws = h->ws;
  p.B = B; p.first = first; p.count = count;
  p.V = h->cfg.vehicles_count; p.M = h->scfg.M; p.N = h->scfg.N;
  p.dt = prep_dt(h->cfg.dt);
  p.ref = h->tables.ref; p.seg = h->tables.seg;
  p.w_speed = h->cfg.weight_speed; p.w_control = h->cfg.weight_control; p.w_diff = h->cfg.weight_input_diff;
  p.collision_check = h->cfg.collision_check;
  CK(h, launch_prepare(p, st));
  h->launches += 1;
  return MPC_OK;
}

MPC_API int mpc_prepare(MpcHandle* h, const float* obs, const float* ref_speed, const float* weights, const uint8_t* reset_mask,
                const MpcLatchState* latch, int B, const MpcCollisionOut* col, void* stream) {
  if (!h) return MPC_ERR_BAD_ARG;
  if (B == 0) return MPC_OK;
  if (!obs || B < 0) return fail(h, MPC_ERR_BAD_ARG, "mpc_prepare: obs is null or B < 0");
  if (B > h->max_batch) return fail(h, MPC_ERR_TOO_LARGE, "mpc_prepare: B exceeds max_batch of mpc_create");
  if (h->cfg.collision_check && (!latch || !latch->collision_memory || !latch->memo_conflict || !latch->is_collide))
    return fail(h, MPC_ERR_BAD_ARG, "mpc_prepare: latch state is required when collision_check is on");
  cudaStream_t st = (cudaStream_t)stream;
  CK(h, cudaSetDevice(h->device));
  int rc;
  if ((rc = timed_begin(h, h->ev_prepare, st))) return rc;
  if ((rc = prepare_range(h, obs, ref_speed, weights, reset_mask, latch, B, 0, B, col, st))) return rc;
  if ((rc = timed_end(h, h->ev_prepare, st))) return rc;
  return MPC_OK;
}

MPC_API int mpc_predict(MpcHandle* h, const float* obs, const float* ref_speed, const float* weights, const uint8_t* reset_mask,
                const MpcLatchState* latch, int B, const MpcSolveOut* out, const MpcCollisionOut* col, void* stream) {
  int rc = mpc_prepare(h, obs, ref_speed, weights, reset_mask, latch, B, col, stream);
  if (rc) return rc;
  MpcProblemBatch b;
  mpc_workspace_batch(h, &b);
  return mpc_solve(h, &b, B, out, stream);
}

MPC_API int mpc_predict_host(MpcHandle* h, const float* obs_host, const float* ref_speed_host, const float* weights_host,
                     const uint8_t* reset_mask_host, int B, float* actions_host, int32_t* status_host,
                     uint8_t* is_collide_host, const MpcCollisionOut* col_host, int64_t* h2d_bytes, int64_t* d2h_bytes) {
  if (!h) return MPC_ERR_BAD_ARG;
  if (B == 0) return MPC_OK;
  if (!obs_host || !actions_host || B < 0) return fail(h, MPC_ERR_BAD_ARG, "mpc_predict_host: null obs/actions or B < 0");
  if (B > h->max_batch) return fail(h, MPC_ERR_TOO_LARGE, "mpc_predict_host: B exceeds max_batch of mpc_create");
  if (B == 0) return MPC_OK;
  CK(h, cudaSetDevice(h->device));
  cudaStream_t st = h->host_stream;
  int64_t up = 0, down = 0;
  const size_t row = (size_t)h->cfg.vehicles_count * 8 * 4;
  MpcLatchState latch{h->d_mem, h->d_memo, h->d_iscol};
  MpcSolveOut out{h->d_actions, h->d_status, h->d_iters, h->d_cost, nullptr};
  MpcCollisionOut col{};
  if (col_host) {            // device staging for the outputs the caller asked for
    if (col_host->agent_collide) col.agent_collide = h->d_flags;
    if (col_host->conflict_index) col.conflict_index = h->d_cidx;
    if (col_host->ego_index) col.ego_index = h->d_egoidx;
    if (col_host->stop_index) col.stop_index = h->d_stop;
    if (col_host->degenerate) col.degenerate = h->d_deg;
    if (col_host->conflict_point) col.conflict_point = h->d_cpt;
  }
  const float* d_rs = ref_speed_host ? h->d_ref_speed : nullptr;
  const float* d_w = weights_host ? h->d_weights : nullptr;
  const uint8_t* d_rm = reset_mask_host ? h->d_reset : nullptr;
  int rc;
  // The observations are 97 % of the upload.  They go up in kHostChunks pieces on a second stream and
  // k_prepare (independent per environment) starts on each piece as soon as it has landed, so the copy of
  // piece c+1 overlaps the parsing / collision logic of piece c.  Small batches take one piece.
  const int chunks = B >= 8192 ? kHostChunks : 1;
  if (ref_speed_host) { CK(h, cudaMemcpyAsync(h->d_ref_speed, ref_speed_host, (size_t)B * 4, cudaMemcpyHostToDevice, h->copy_stream)); up += (int64_t)B * 4; }
  if (weights_host) { CK(h, cudaMemcpyAsync(h->d_weights, weights_host, (size_t)B * 12, cudaMemcpyHostToDevice, h->copy_stream)); up += (int64_t)B * 12; }
  if (reset_mask_host) { CK(h, cudaMemcpyAsync(h->d_reset, reset_mask_host, (size_t)B, cudaMemcpyHostToDevice, h->copy_stream)); up += B; }
  if ((rc = timed_begin(h, h->ev_prepare, st))) return rc;
  for (int c = 0; c < chunks; ++c) {
    const int lo = (int)((int64_t)B * c / chunks), hi = (int)((int64_t)B * (c + 1) / chunks);
    if (hi <= lo) continue;
    CK(h, cudaMemcpyAsync((char*)h->d_obs + (size_t)lo * row, (const char*)obs_host + (size_t)lo * row, (size_t)(hi - lo) * row,
                          cudaMemcpyHostToDevice, h->copy_stream));
    up += (int64_t)(hi - lo) * (int64_t)row;
    CK(h, cudaEventRecord(h->copy_done[c], h->copy_stream));
    CK(h, cudaStreamWaitEvent(st, h->copy_done[c], 0));
    if ((rc = prepare_range(h, h->d_obs, d_rs, d_w, d_rm, &latch, B, lo, hi - lo, &col, st))) return rc;
  }
  if ((rc = timed_end(h, h->ev_prepare, st))) return rc;
  MpcProblemBatch wb;
  mpc_workspace_batch(h, &wb);
  if ((rc = mpc_solve(h, &wb, B, &out, st))) return rc;
  CK(h, cudaMemcpyAsync(actions_host, h->d_actions, (size_t)B * 8, cudaMemcpyDeviceToHost, st)); down += (int64_t)B * 8;
  if (status_host) { CK(h, cudaMemcpyAsync(status_host, h->d_status, (size_t)B * 4, cudaMemcpyDeviceToHost, st)); down += (int64_t)B * 4; }
  if (is_collide_host) { CK(h, cudaMemcpyAsync(is_collide_host, h->ws.is_collide, (size_t)B, cudaMemcpyDeviceToHost, st)); down += B; }
  if (col_host) {
    const size_t Mx = (size_t)(h->scfg.M > 0 ? h->scfg.M : 1);
    auto back = [&](void* dst, const void* src, size_t bytes) -> cudaError_t {
      if (!dst) return cudaSuccess;
      down += (int64_t)bytes;
      return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st);
    };
    CK(h, back(col_host->agent_collide, h->d_flags, (size_t)B * Mx));
    CK(h, back(col_host->conflict_index, h->d_cidx, (size_t)B * Mx * 4));
    CK(h, back(col_host->ego_index, h->d_egoidx, (size_t)B * 4));
    CK(h, back(col_host->stop_index, h->d_stop, (size_t)B * 4));
    CK(h, back(col_host->degenerate, h->d_deg, (size_t)B));
    CK(h, back(col_host->conflict_point, h->d_cpt, (size_t)B * Mx * 8));
    if (col_host->is_collide) CK(h, back(col_host->is_collide, h->ws.is_collide, (size_t)B));
  }
  CK(h, cudaStreamSynchronize(st));
  if (h2d_bytes) *h2d_bytes = up;
  if (d2h_bytes) *d2h_bytes = down;
  return MPC_OK;
}

MPC_API int mpc_set_warm_start(MpcHandle* h, const float* u_init) {
  if (!h) return MPC_ERR_BAD_ARG;
  h->u_init = u_init;
  return MPC_OK;
}

MPC_API int mpc_set_adaptive_starts(MpcHandle* h, int max_starts, float rel_gap, float* start_cost, uint8_t* extended) {
  if (!h) return MPC_ERR_BAD_ARG;
  if (max_starts == 0) {
    h->max_starts = 0; h->start_cost = nullptr; h->extended = nullptr;
    return MPC_OK;
  }
  if (h->n_starts < 2) return fail(h, MPC_ERR_BAD_ARG, "mpc_set_adaptive_starts: the handle's n_starts must be at least 2");
  if (max_starts <= h->n_starts || max_starts > MPC_MAX_STARTS)
    return fail(h, MPC_ERR_BAD_ARG, "mpc_set_adaptive_starts: max_starts must be in (n_starts, 8]");
  if (rel_gap != rel_gap) return fail(h, MPC_ERR_BAD_ARG, "mpc_set_adaptive_starts: rel_gap is NaN");
  if ((long long)h->max_batch * max_starts > 0x7fffffffLL / 64) return fail(h, MPC_ERR_BAD_ARG, "mpc_set_adaptive_starts: max_batch * max_starts too large");
  CK(h, cudaSetDevice(h->device));
  const size_t B = (size_t)h->max_batch;
  if (max_starts > h->cand_starts) {     // candidate arrays for every start that may run; cudaFree waits for work in flight
    SolveCand c{};
    const size_t W = B * (size_t)max_starts;
    cudaError_t e = cudaMalloc(&c.cost, W * 4);
    if (e == cudaSuccess) e = cudaMalloc(&c.u0, W * 8);
    if (e == cudaSuccess) e = cudaMalloc(&c.status, W * 4);
    if (e == cudaSuccess) e = cudaMalloc(&c.iters, W * 4);
    if (e == cudaSuccess) e = cudaMalloc(&c.U, W * (size_t)h->scfg.N * 8);
    SolveCand& old = e == cudaSuccess ? h->cand : c;
    cudaFree(old.cost); cudaFree(old.u0); cudaFree(old.status); cudaFree(old.iters); cudaFree(old.U);
    if (e != cudaSuccess) return fail(h, MPC_ERR_CUDA, "mpc_set_adaptive_starts: candidate arrays", e);
    h->cand = c;
    h->cand_starts = max_starts;
  }
  if (max_starts > h->aq_starts) {
    int* q = nullptr;
    CK(h, cudaMalloc(&q, (2 + B + (size_t)(max_starts - h->n_starts) * B) * sizeof(int)));
    cudaFree(h->aq_block);
    h->aq_block = q;
    h->aq_starts = max_starts;
  }
  h->max_starts = max_starts;
  h->rel_gap = rel_gap;
  h->start_cost = start_cost;
  h->extended = extended;
  return MPC_OK;
}

MPC_API int64_t mpc_launch_count(const MpcHandle* h) { return h ? h->launches : 0; }

MPC_API int mpc_fp32_peak(MpcHandle* h, int repeats, float* tflops_out) {
  if (!h || !tflops_out) return MPC_ERR_BAD_ARG;
  CK(h, cudaSetDevice(h->device));
  const int block = 256, grid = h->sm_count * 8, iters = 4096;
  cudaEvent_t a, b;
  CK(h, cudaEventCreate(&a));
  CK(h, cudaEventCreate(&b));
  CK(h, launch_fma_peak(h->sink, 64, grid, block, nullptr));   // warm-up
  float best = 0.f;
  if (repeats < 1) repeats = 1;
  for (int r = 0; r < repeats; ++r) {
    CK(h, cudaEventRecord(a, nullptr));
    CK(h, launch_fma_peak(h->sink, iters, grid, block, nullptr));
    CK(h, cudaEventRecord(b, nullptr));
    CK(h, cudaEventSynchronize(b));
    float ms = 0.f;
    CK(h, cudaEventElapsedTime(&ms, a, b));
    const double flops = 2.0 * 16 * 8 * (double)iters * (double)grid * block;
    const float tf = (float)(flops / (ms * 1e-3) / 1e12);
    if (tf > best) best = tf;
    h->launches += 1;
  }
  h->launches += 1;
  cudaEventDestroy(a); cudaEventDestroy(b);
  *tflops_out = best;
  return MPC_OK;
}

MPC_API int mpc_timing_begin(MpcHandle* h) {
  if (!h) return MPC_ERR_BAD_ARG;
  for (auto e : h->ev_prepare) cudaEventDestroy(e);
  for (auto e : h->ev_solve) cudaEventDestroy(e);
  h->ev_prepare.clear(); h->ev_solve.clear();
  h->timing = true;
  return MPC_OK;
}

MPC_API int mpc_timing_end(MpcHandle* h, float* prepare_ms_avg, float* solve_ms_avg, int* n_prepare, int* n_solve) {
  if (!h) return MPC_ERR_BAD_ARG;
  h->timing = false;
  CK(h, cudaSetDevice(h->device));
  CK(h, cudaDeviceSynchronize());
  auto avg = [&](std::vector<cudaEvent_t>& v, float* out_ms, int* out_n) -> int {
    double tot = 0; int n = 0;
    for (size_t i = 0; i + 1 < v.size(); i += 2) {
      float ms = 0.f;
      cudaError_t e = cudaEventElapsedTime(&ms, v[i], v[i + 1]);
      if (e != cudaSuccess) return fail(h, MPC_ERR_CUDA, "cudaEventElapsedTime", e);
      tot += ms; ++n;
    }
    if (out_ms) *out_ms = n ? (float)(tot / n) : 0.f;
    if (out_n) *out_n = n;
    return MPC_OK;
  };
  int rc = avg(h->ev_prepare, prepare_ms_avg, n_prepare);
  if (rc) return rc;
  return avg(h->ev_solve, solve_ms_avg, n_solve);
}

}  // extern "C"
