/* mpc_b200.h -- C ABI of libmpcb200.so: batched nonlinear MPC for the PureMPC_Agent hot path
 * of SaeedRahmani/MPC-RL_for_AVs, NVIDIA B200 (sm_100a) only.
 *
 * The reference has no FFI for this path: it is Python calling CasADi/IPOPT and shapely in
 * process (agents/pure_mpc.py:297-300, :608-609).  The entry points below are what a ctypes
 * binding inside the reference's own `PureMPC_Agent` would call instead; each one cites the
 * reference interface it replaces.  INTEGRATION.md shows that binding.
 *
 * Conventions
 *  - plain pointers and sizes only; every array argument of the *device* entry points is a
 *    CUDA device pointer borrowed for the duration of the call (the caller -- PyTorch -- owns
 *    all memory); `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *  - all work is enqueued on `stream`; nothing synchronises with the host except the
 *    `*_host` entry points, which are synchronous by contract.
 *  - return value: 0 = ok, < 0 = error (see MpcError); `mpc_last_error` gives the text.
 *    Nothing throws across this boundary.  There is NO CPU fallback: without an sm_100
 *    device `mpc_create` fails.
 *  - state order [x, y, theta, v], control order [accel, steer]  (agents/pure_mpc.py:88-89).
 */
#ifndef MPC_B200_H_
#define MPC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MPC_API __attribute__((visibility("default")))
#else
#define MPC_API
#endif

#define MPC_ABI_VERSION 2
#define MPC_MAX_OBSTACLES 16
#define MPC_N_REF 85 /* rows of the reference path, agents/base_agent.py:127-152 */

typedef enum MpcError {
  MPC_OK = 0,
  MPC_ERR_BAD_ARG = -1,
  MPC_ERR_NO_DEVICE = -2,  /* no CUDA device, or compute capability != 10.x */
  MPC_ERR_CUDA = -3,       /* allocation / launch failure, text in mpc_last_error */
  MPC_ERR_TOO_LARGE = -4   /* batch > max_batch given to mpc_create */
} MpcError;

/* per-problem status bits written to MpcSolveOut.status
 * (the reference only prints on solver failure and still applies the iterate,
 *  agents/pure_mpc.py:303-305; here the caller gets the flag) */
#define MPC_STATUS_CONVERGED 0          /* un-damped Newton step below tol_step accepted: a certified local optimum */
#define MPC_STATUS_MAX_ITER 1
#define MPC_STATUS_LINESEARCH_FAIL 2
#define MPC_STATUS_NAN 4
#define MPC_STATUS_INFEASIBLE_START 8   /* s0 violates a state bound: the reference NLP is infeasible */
#define MPC_STATUS_STALLED 16           /* no progress over 6 iterations while the steps were still large */
#define MPC_STATUS_KINK 32              /* settled (objective stationary to 1e-7 over 6 iterations, steps < 10 tol_step) on a
                                         * kink of the bound-clamped dynamics; near-optimal (median 0.2 % of the cost), not certified */
#define MPC_MAX_STARTS 8

/* Configuration = cfg["pure_mpc"] of the reference (config/cfg.yaml:88-106) plus the constants
 * that are hard-coded in agents/pure_mpc.py, and the solver's own knobs. */
typedef struct MpcConfig {
  int32_t abi_version;        /* MPC_ABI_VERSION */
  int32_t horizon;            /* cfg.yaml:90 (16 shipped; benchmark 20); 2..64 */
  int32_t vehicles_count;     /* env observation rows V = ego + others (cfg.yaml:2); M = V-1 <= 16 */
  float dt;                   /* 1 / policy_frequency (agents/base_agent.py:43) */
  float weight_speed;         /* cfg.yaml:101 */
  float weight_control;       /* cfg.yaml:102 */
  float weight_input_diff;    /* cfg.yaml:104 */
  float weight_distance;      /* cfg.yaml:105; 0 = live agent (term disabled, pure_mpc.py:82,204-212) */
  float weight_collision;     /* cfg.yaml:106; 0 = live agent */
  int32_t collision_check;    /* 1: _check_collision + regeneration (agents/pure_mpc.py); 0: agents/pure_mpc_no_collision.py flow */
  int32_t literal_no_collision; /* 1: objective of pure_mpc_no_collision.py:146-151 (control + input diff only) */
  int32_t max_iter;           /* solver iteration cap (reference: ipopt.max_iter 1000) */
  float tol_step;             /* convergence: max |du| of an accepted full step */
  float reg_min;              /* eigenvalue floor of the control Hessian */
  int32_t threads_per_block;  /* 0 = default */
  int32_t blocks_per_sm;      /* 0 = default */
  int32_t n_starts;           /* start portfolio: solves per problem, lowest objective wins; 1 = only the reference's cold
                               * start (zero controls, agents/pure_mpc.py:244); 0 = default (4); <= MPC_MAX_STARTS */
} MpcConfig;

/* One batch of parsed problems, SoA, length B (what _parse_obs + _check_collision +
 * update_reference_states leave behind for _solve: agents/base_agent.py:81-116,
 * agents/pure_mpc.py:552-724).  Produced on device by mpc_prepare / consumed by mpc_solve;
 * callers that already hold parsed problems may fill it themselves. */
typedef struct MpcProblemBatch {
  const float* s0;            /* [4][B]  x, y, theta (wrapped to [-pi,pi]), speed */
  const int32_t* ego_index;   /* [B]     nearest reference row (pure_mpc.py:106-109) */
  const float* w_speed;       /* [B]     100 when is_collide (pure_mpc.py:143-147) else weight_speed / RL */
  const float* w_control;     /* [B] */
  const float* w_diff;        /* [B] */
  /* reference speed seen by stage k: k < vr_n ? vr_a + k*vr_slope : vr_b
   * (constant: vr_n = 0; regenerated ramp of pure_mpc.py:707-716: vr_a = v_ego, vr_b = 0) */
  const float* vr_a;          /* [B] */
  const float* vr_slope;      /* [B] */
  const float* vr_b;          /* [B] */
  const int32_t* vr_n;        /* [B] */
  const uint8_t* is_collide;  /* [B] */
  const int32_t* n_obs;       /* [B]     present other vehicles */
  const float* obstacles;     /* [M][4][B]  x, y, speed*dt*cos(h), speed*dt*sin(h) (base_agent.py:172-174) */
} MpcProblemBatch;

/* Result of a solve.  `actions` is what PureMPC_Agent.predict returns (u_opt[0],
 * agents/pure_mpc.py:311-318).  Optional outputs may be NULL. */
typedef struct MpcSolveOut {
  float* actions;             /* [B][2]  first control (accel, steer) */
  int32_t* status;            /* [B]     MPC_STATUS_* bits */
  int32_t* iters;             /* [B]     iterations used (total over the starts of the portfolio) */
  float* cost;                /* [B]     objective at the returned iterate (pure_mpc.py:204-212) */
  float* U;                   /* [B][N][2] full control sequence, or NULL */
} MpcSolveOut;

/* Per-environment collision latch (agents/pure_mpc.py:38-43, 552-563, 660-676), caller-visible so
 * environments can be reset or sharded.  Read and updated by mpc_prepare / mpc_predict. */
typedef struct MpcLatchState {
  int32_t* collision_memory;  /* [B]  steps left in the 10-step memory (0 = none) */
  int32_t* memo_conflict;     /* [B]  earliest memorised conflict index, -1 = None */
  uint8_t* is_collide;        /* [B]  flag of the last call (kept when detection aborts, pure_mpc.py:582-587) */
} MpcLatchState;

/* Per-call collision outputs (public attributes of the reference agent: is_collide,
 * conflict_index, agent_collide, ego_index, stop_point).  Any pointer may be NULL. */
typedef struct MpcCollisionOut {
  uint8_t* agent_collide;     /* [B][M] */
  int32_t* conflict_index;    /* [B][M]  -1 = None */
  uint8_t* is_collide;        /* [B] */
  int32_t* ego_index;         /* [B] */
  int32_t* stop_index;        /* [B]  regenerated stop row, -1 = none */
  uint8_t* degenerate;        /* [B]  a tested orientation was within 1e-9 (relative) of zero without being zero (robust vs plain predicate may differ) */
  float* conflict_point;      /* [B][M][2]  the intersection point behind each flag (self.conflict_points, pure_mpc.py:656), NaN = None */
} MpcCollisionOut;

typedef struct MpcHandle MpcHandle;

/* Replaces PureMPC_Agent.__init__ (agents/pure_mpc.py:24-63, agents/base_agent.py:14-49).
 * Allocates every workspace for batches up to max_batch on `device`. */
MPC_API int mpc_create(const MpcConfig* cfg, int device, int max_batch, MpcHandle** out);
MPC_API int mpc_destroy(MpcHandle* h);
/* Text of the last error on this handle (h may be NULL: last error of mpc_create). */
MPC_API const char* mpc_last_error(const MpcHandle* h);

/* Device views of the handle's own parsed-problem workspace (filled by mpc_prepare). */
MPC_API int mpc_workspace_batch(MpcHandle* h, MpcProblemBatch* out);

/* K1 parity entry point: rollout + the six cost components of the reference's `cost_fn`
 * (agents/pure_mpc.py:215-216, 220-228, 252-254) for given controls U [B][N][2].
 * X_out [B][N+1][4], cost6_out [B][6] = state, control, final_state, input_diff, distance,
 * collision (un-weighted), total_out [B] = objective of pure_mpc.py:204-212 (+ weighted archive terms). */
MPC_API int mpc_rollout_cost(MpcHandle* h, const MpcProblemBatch* batch, int B, const float* U, float* X_out,
                     float* cost6_out, float* total_out, void* stream);

/* Replaces the NLP build + IPOPT solve of PureMPC_Agent._solve (agents/pure_mpc.py:230-318). */
MPC_API int mpc_solve(MpcHandle* h, const MpcProblemBatch* batch, int B, const MpcSolveOut* out, void* stream);

/* Replaces _parse_obs + _check_collision + update_reference_states
 * (agents/base_agent.py:81-116, agents/pure_mpc.py:552-724): obs [B][V][8] f32 in the Kinematics
 * layout, ref_speed [B] or NULL (NaN entries = no override; pure_mpc.py:683-688), weights [B][3] or
 * NULL (weights_from_RL, pure_mpc.py:96-104), reset_mask [B] or NULL (1 = clear this env's latch
 * first).  Fills the handle's problem workspace; collision outputs optional. */
MPC_API int mpc_prepare(MpcHandle* h, const float* obs, const float* ref_speed, const float* weights,
                const uint8_t* reset_mask, const MpcLatchState* latch, int B, const MpcCollisionOut* col,
                void* stream);

/* Replaces PureMPC_Agent.predict (agents/pure_mpc.py:68-78): mpc_prepare followed by mpc_solve
 * on the handle's workspace.  latch may be NULL only if cfg.collision_check == 0. */
MPC_API int mpc_predict(MpcHandle* h, const float* obs, const float* ref_speed, const float* weights,
                const uint8_t* reset_mask, const MpcLatchState* latch, int B, const MpcSolveOut* out,
                const MpcCollisionOut* col, void* stream);

/* OPT-IN warm start (SURVEY 8-f row N3; the reference always cold-starts from zero controls,
 * agents/pure_mpc.py:240-246): subsequent mpc_solve / mpc_predict calls start each problem from
 * u_init [B][N][2] (device pointer, borrowed until replaced; NULL switches back to the cold start).
 * A warm start changes which local optimum of the multi-modal NLP is found: keep it off for parity runs. */
MPC_API int mpc_set_warm_start(MpcHandle* h, const float* u_init);

/* OPT-IN adaptive portfolio: subsequent mpc_solve / mpc_predict(_host) calls run starts n_starts..max_starts-1 only for
 * problems whose base objectives J_0..J_{n_starts-1} disagree: any of them not finite, or
 * max J - min J > rel_gap * max(|min J|, 1).  Such a problem is "extended"; its results (actions, status, cost, U, iters)
 * are bit-identical to those of a handle with n_starts = max_starts, every other problem's to those of this handle without
 * the mode.  The extra starts are queued inside the running solve launch by the thread that finishes a problem's last
 * base start, so the mode costs no second launch; it may lengthen the launch's tail by up to one more solve.
 * Needs the handle's n_starts >= 2 and max_starts in (n_starts, MPC_MAX_STARTS]; rel_gap must not be NaN (+inf: extend
 * only problems with a non-finite base objective; < 0: extend all).  max_starts = 0 switches the mode off.
 * start_cost [max_starts][max_batch] (row stride max_batch; NaN for starts that did not run) and extended [B] are device
 * pointers or NULL, borrowed until replaced.  Allocates; do not call during stream capture. */
MPC_API int mpc_set_adaptive_starts(MpcHandle* h, int max_starts, float rel_gap, float* start_cost, uint8_t* extended);

/* Same call with HOST buffers (what a numpy caller holds): obs/ref_speed/weights/reset_mask are
 * copied host->device, actions/status (and is_collide) device->host, inside the call; the latch
 * lives in the handle.  col_host (may be NULL, and so may any pointer in it) receives the per-call collision
 * outputs in HOST arrays of the MpcCollisionOut shapes -- the public attributes a drop-in PureMPC_Agent exposes.
 * Synchronous.  Returns bytes moved in *h2d_bytes / *d2h_bytes if non-NULL. */
MPC_API int mpc_predict_host(MpcHandle* h, const float* obs_host, const float* ref_speed_host,
                     const float* weights_host, const uint8_t* reset_mask_host, int B,
                     float* actions_host, int32_t* status_host, uint8_t* is_collide_host,
                     const MpcCollisionOut* col_host, int64_t* h2d_bytes, int64_t* d2h_bytes);

/* Measurement helpers */
/* number of this library's kernel launches since mpc_create (bench.py's gpu_launches) */
MPC_API int64_t mpc_launch_count(const MpcHandle* h);
/* FP32 FMA micro-benchmark on the handle's device: achieved TFLOP/s (FMA = 2 flops), for the roofline denominator */
MPC_API int mpc_fp32_peak(MpcHandle* h, int repeats, float* tflops_out);
/* average duration in ms of the `which` kernel (0 = prepare, 1 = solve) over the launches timed since
 * mpc_timing_begin: CUDA events recorded on the launch stream around every launch */
MPC_API int mpc_timing_begin(MpcHandle* h);
MPC_API int mpc_timing_end(MpcHandle* h, float* prepare_ms_avg, float* solve_ms_avg, int* n_prepare, int* n_solve);
/* which solve kernel a launch of B problems uses: *gains_in_tmem = 1 -> k_solve_tmem (feedback gains in
 * tensor memory), 0 -> k_solve (gains in shared memory); *threads_per_block = its block size (one block per SM).
 * The launch is sized on the B * n_starts base work items; the adaptive portfolio's extra starts do not change it. */
MPC_API int mpc_solve_config(const MpcHandle* h, int B, int* gains_in_tmem, int* threads_per_block);
/* device properties used for grid sizing */
MPC_API int mpc_device_info(const MpcHandle* h, int* sm_count, int* cc_major, int* cc_minor, int* smem_per_block_optin);

/* ---- SURVEY 8-f row N1 (not part of the MPC hot path): one step of the batched synthetic intersection
 * environment of mpc_rl_for_avs_b200.rl as a single kernel.  Replaces nothing in the reference (highway-env's
 * IntersectionEnv.step is third-party Python); rules cited in rl.py (envs/intersection_env__.py:61-129, :395-446).
 * State arrays are updated in place; finished environments are reset in place.  The caller advances
 * *counter by 10 draw steps afterwards (rl.BatchedIntersectionEnv does). */
typedef struct MpcEnvStep {
  float* ego;                 /* [B][4]  x, y, heading, speed                 in/out */
  float* others;              /* [B][M][4]  x, y, speed, heading              in/out */
  int32_t* t;                 /* [B]  policy steps since reset                in/out */
  uint8_t* crashed_state;     /* [B]                                          out    */
  const int64_t* counter;     /* device scalar: draw counter of the env's random numbers */
  const float* action;        /* [B][2]  (accel, steer) as sent by the caller */
  float* obs;                 /* [B][M+1][8]  observation after the step / reset */
  float* terminal_obs;        /* [B][M+1][8]  observation before the reset       */
  float* reward;              /* [B] */
  uint8_t* done;              /* [B] */
  uint8_t* crashed;           /* [B] */
  uint8_t* arrived;           /* [B] */
  uint8_t* truncated;         /* [B] */
  float* speed;               /* [B]  ego speed after the step (before a reset) */
  int32_t B, n_others;
  int32_t substeps;           /* simulation_frequency / policy_frequency */
  int32_t duration_steps;
  int32_t raw_action;         /* 1: clip to [-1, 1] and scale to +-5 m/s^2, +-pi/4 (SB3 raw action path, quirk Q8) */
  float dt_sim;
  float arrive_x, arrive_y;   /* arrival test: x <= arrive_x and |y - arrive_y| < 4 */
} MpcEnvStep;
MPC_API int mpc_env_step(const MpcEnvStep* args, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MPC_B200_H_ */
