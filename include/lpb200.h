/*
 * lpb200.h -- C ABI of liblpb200.so: the B200-native (sm_100a) replacement for the
 * interior-point hot path of the `ripped` LP solver (sebasv/lp).
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  Every entry point cites the
 * reference interface it replaces; paths are relative to /root/reference/src.
 * Plain pointers and sizes only: no C++/torch types cross this boundary, no
 * exceptions, no aborts.  All matrices are row-major IEEE FP64.
 *
 * There is NO CPU fallback behind this API: with no CUDA device every compute
 * entry point returns LPB_ERR_NO_DEVICE.
 *
 * Threading: a context is not thread-safe; use one per host thread (the reference's
 * `solve(&self, &Problem)` is re-entrant because it owns no state; a context is
 * the owned GPU state of ONE solve at a time).
 */
#ifndef LPB200_H_
#define LPB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define LPB_ABI_VERSION 1

/* ------------------------------------------------------------------ status codes
 * 0 = Ok / Optimal, 1..7 = one per `LinearProgramError` variant in declaration
 * order (error.rs:7-29), negative = failures that have no reference counterpart. */
enum {
  LPB_OK = 0,
  LPB_ERR_UNCONSTRAINED = 1,                  /* error.rs:10 */
  LPB_ERR_NUMERICAL_PROBLEM = 2,              /* error.rs:13 */
  LPB_ERR_INVALID_PARAMETER = 3,              /* error.rs:16 */
  LPB_ERR_INCOMPATIBLE_INPUT_DIMENSIONS = 4,  /* error.rs:19 */
  LPB_ERR_INFEASIBLE = 5,                     /* error.rs:22 */
  LPB_ERR_UNBOUNDED = 6,                      /* error.rs:25 */
  LPB_ERR_ITERATION_LIMIT_EXCEEDED = 7,       /* error.rs:28 (x_out is still filled) */
  LPB_ERR_CUDA = -1,
  LPB_ERR_NCCL = -2,
  LPB_ERR_NO_DEVICE = -3,
  LPB_ERR_BAD_ARGUMENT = -4,
  LPB_ERR_UNSUPPORTED = -5                    /* e.g. solver_type != Cholesky, see below */
};

/* EquationSolverType (interior_point/newton_equations.rs:36-46).  Only Cholesky is the
 * accelerated path; Inverse / LeastSquares (the CPU QR/LU/SVD fallback chain,
 * newton_equations.rs:201-209) are rejected with LPB_ERR_UNSUPPORTED, never silently mapped. */
enum { LPB_SOLVER_CHOLESKY = 0, LPB_SOLVER_INVERSE = 1, LPB_SOLVER_LEAST_SQUARES = 2 };

/* InteriorPointBuilder fields (interior_point/mod.rs:41-48), defaults :51-60. */
typedef struct lpb_options {
  double tol;        /* 1e-8 */
  int32_t disp;      /* 0 */
  int32_t ip;        /* 1 */
  int32_t solver_type; /* LPB_SOLVER_CHOLESKY */
  int32_t reserved;
  double alpha0;     /* 0.99995 */
  int64_t max_iter;  /* 1000 */
} lpb_options;

/* InteriorPointBuilder::new (mod.rs:51-60). */
void lpb_options_default(lpb_options* o);
/* InteriorPointBuilder::build validation (mod.rs:118-128): LPB_ERR_INVALID_PARAMETER when
 * !(0 < alpha0 < 1) or tol <= 0; LPB_ERR_UNSUPPORTED when solver_type != Cholesky. */
int lpb_options_validate(const lpb_options* o);

const char* lpb_strerror(int code);   /* Display strings of error.rs:8-28 */
const char* lpb_last_error(void);     /* detail of the last CUDA/NCCL/argument failure on this thread */
int lpb_abi_version(void);
int lpb_device_count(void);           /* 0 when no CUDA device is visible */

/* ------------------------------------------------------------------ problem model (host)
 * ProblemBuilder::build (linear_program.rs:125-169): slack form
 *     A = [[A_ub, I], [A_eq, 0]],  b = [b_ub; b_eq],  c = [c; 0].
 * Shapes are passed as the reference sees them so the two validations are identical:
 * LPB_ERR_UNCONSTRAINED when rows_ub + rows_eq == 0 (:134-136),
 * LPB_ERR_INCOMPATIBLE_INPUT_DIMENSIONS on any mismatch (:137-143).
 * A_ub / A_eq may be NULL when their row count is 0 (then cols_* must still equal n_c,
 * exactly like the reference's (0, n) placeholders, :127-130). */
int lpb_slack_dims(int64_t n_c, int64_t rows_ub, int64_t cols_ub, int64_t len_b_ub,
                   int64_t rows_eq, int64_t cols_eq, int64_t len_b_eq,
                   int64_t* m_out, int64_t* n_out, int64_t* n_slack_out);
int lpb_build_slack_form(const double* c, int64_t n_c,
                         const double* A_ub, int64_t rows_ub, int64_t cols_ub, int64_t ld_ub,
                         const double* b_ub, int64_t len_b_ub,
                         const double* A_eq, int64_t rows_eq, int64_t cols_eq, int64_t ld_eq,
                         const double* b_eq, int64_t len_b_eq,
                         double* A_out, int64_t ld_out, double* b_out, double* c_out);

/* Pinned host memory for the slack-form arrays (so uploads run at PCIe rate). */
int lpb_host_alloc(void** p, uint64_t bytes);
int lpb_host_free(void* p);

/* ------------------------------------------------------------------ context
 * Owns every device buffer of one LP in slack form (Problem, linear_program.rs:24-30;
 * FeasiblePoint, feasible_point.rs:14-21; EquationsSolver::Cholesky{factor,M,Dinv},
 * newton_equations.rs:108-113).  `stream` is a cudaStream_t (NULL = a stream owned by ctx). */
typedef struct lpb_ctx lpb_ctx;

enum {
  LPB_MEM_HOST = 0,     /* A, b, c are host pointers (copied H2D)            */
  LPB_MEM_DEVICE = 1    /* A, b, c are device pointers (copied D2D, padded)  */
};

int lpb_create(lpb_ctx** ctx, int64_t m, int64_t n, const double* A, int64_t lda,
               const double* b, const double* c, double c0, int mem, void* stream);
/* Re-upload a problem of the SAME dims into an existing context. */
int lpb_set_problem(lpb_ctx* ctx, const double* A, int64_t lda, const double* b, const double* c,
                    double c0, int mem);
/* Work-buffers-only context for the lpb_k_* kernel entry points (no problem attached). */
int lpb_create_bare(lpb_ctx** ctx, int64_t m_max, int64_t n_max, void* stream);
int lpb_destroy(lpb_ctx* ctx);

/* Column-sharded multi-GPU context (SURVEY.md 8e; no reference counterpart): this rank owns
 * columns [col0, col0+n_local) of the m x n_global slack-form A.  `nccl_unique_id` is the
 * 128-byte ncclUniqueId every rank received from rank 0 (lpb_nccl_unique_id), or NULL to re-use the
 * process communicator. */
int lpb_nccl_unique_id(void* id128);
/* The NCCL communicator is process-wide (one process per GPU) and outlives contexts: the first
 * lpb_create_sharded with a unique id builds it, later ones pass nccl_unique_id = NULL and share it.
 * lpb_comm_ready: 1 if this process already holds a communicator for (rank, world). */
int lpb_comm_ready(int rank, int world);
int lpb_comm_finalize(void);
int lpb_create_sharded(lpb_ctx** ctx, int64_t m, int64_t n_global, int64_t col0, int64_t n_local,
                       const double* A_local, int64_t lda, const double* b, const double* c_local,
                       double c0, int mem, int rank, int world, const void* nccl_unique_id,
                       void* stream);
/* Fill this rank's column shard of the SURVEY 8(d)-style synthetic LP on the device
 * (counter-based generator keyed by (seed, global row, global column)); A is never on the host. */
int lpb_create_sharded_synthetic(lpb_ctx** ctx, int64_t m, int64_t n_global, int64_t col0,
                                 int64_t n_local, uint64_t seed, int rank, int world,
                                 const void* nccl_unique_id, void* stream);

/* Peer-memory hand-off inside the distributed factorisation (optional; no reference counterpart).  The owner of a
 * panel writes the 128 rows the next owner needs straight into every peer's panel slot over NVLink and raises a flag
 * there, instead of an ncclBroadcast of 128 KB (cholesky.cu: peer_push_kernel / wait_flag_kernel).  The ring of
 * 2 x world panel slots and the mappings of the other ranks' rings belong to the PROCESS (one process per GPU), like
 * the NCCL communicator; a context attaches to them while it lives.
 *   lpb_peer_export: *state_out = 0: attached to a ring this process has mapped before -- nothing to do;
 *                    1: a new ring was allocated, handle64_out holds its cudaIpcMemHandle: all-gather the handles in
 *                       rank order and call lpb_peer_import with all `world` of them (64 bytes each);
 *                    2: another live context of this process holds the ring -- this one keeps ncclBroadcast.
 *   Every rank must reach the same verdict: unless ALL ranks exported and imported successfully, all of them call
 *   lpb_set_option(ctx, "peer_panels", -1) (give the ring up).  "peer_panels" = 0 / 1 switches the hand-off off / on
 *   for a context whose peers are mapped.  lpb_comm_finalize frees the ring. */
int lpb_peer_export(lpb_ctx* ctx, void* handle64_out, int* state_out);
int lpb_peer_import(lpb_ctx* ctx, const void* handles, int world);

/* Copy this context's (shard of the) slack-form problem back to the host: A_out m x n_local
 * (leading dimension lda_out >= n_local), b_out m, c_out n_local; any pointer may be NULL.
 * (Accessors Problem::A()/b()/c(), linear_program.rs:42-54, for device-generated shards.) */
int lpb_download_problem(lpb_ctx* ctx, double* A_out, int64_t lda_out, double* b_out, double* c_out);

/* ------------------------------------------------------------------ whole solve
 * Solver::solve + solve_normal_form (interior_point/mod.rs:161-169,199-240).
 * x_out: n doubles, x/tau in SLACK form (caller drops the last n_slack entries,
 * linear_program.rs:65-69); filled on LPB_OK and on LPB_ERR_ITERATION_LIMIT_EXCEEDED
 * (mod.rs:237-239).  fun = c.x_slack + c0 (linear_program.rs:61-63).  Sharded contexts write
 * only their own n_local entries.  x_out may be a host pointer only. */
int lpb_solve(lpb_ctx* ctx, const lpb_options* opts, double* x_out, double* fun, int64_t* iterations);

/* Per-iteration trace of the last lpb_solve (the `disp` columns of indicators.rs:25-33 plus tau,
 * kappa and the scalars of the corrector's Delta::compute, delta.rs:29-38): rows of LPB_TRACE_COLS
 * doubles {alpha, rho_p, rho_d, rho_A, rho_g, rho_mu, obj, bty, tau, kappa, c.p, b.q, c.u, b.v, d_tau, d_kappa}. */
#define LPB_TRACE_COLS 16
int64_t lpb_trace(lpb_ctx* ctx, double* rows, int64_t max_rows);

/* ------------------------------------------------------------------ phase calls
 * The same steps lpb_solve runs, exported so a host (the Rust shim, rust/src/lib.rs; the C++
 * mirror, lp_b200/host/ripped.hpp) can drive the loop itself.  Scalars tau/kappa live on the host. */
typedef struct lpb_residual_scalars {
  double nrm_rp;  /* ||b tau - A x||_2          residual.rs:23 */
  double nrm_rd;  /* ||c tau - A^T y - z||_2    residual.rs:24-26 */
  double cx;      /* c . x */
  double by;      /* b . y */
  double xz;      /* x . z */
} lpb_residual_scalars;

typedef struct lpb_direction_in {
  int32_t corrector;  /* 0: Rhat::predictor (rhat.rs:17-35), 1: Rhat::corrector (rhat.rs:37-75) */
  int32_t ip;
  double eta;
  double gamma;
  double mu;
  double alpha;       /* predictor step length (corrector only) */
} lpb_direction_in;

typedef struct lpb_direction_out {
  double cu, bv;      /* c.u, b.v  (delta.rs:30) */
  double cp, bq;      /* c.p, b.q  (delta.rs:32) */
  int32_t nan_pq;     /* newton_equations.rs:190-194 */
  int32_t reserved;
} lpb_direction_out;

/* FeasiblePoint::blind_start (feasible_point.rs:24-39): x = 1, y = 0, z = 1. */
int lpb_blind_start(lpb_ctx* ctx);
/* r_P, r_D (kept on device) and the scalars of feasible_point.rs:122-125 / residual.rs:13-44. */
int lpb_residuals(lpb_ctx* ctx, double tau, double kappa, lpb_residual_scalars* out);
/* EquationSolverType::build (newton_equations.rs:48-64): Dinv = x/z, M = A diag(Dinv) A^T,
 * Cholesky.  Non-positive / non-finite pivot -> LPB_ERR_NUMERICAL_PROBLEM (:63). */
int lpb_form_and_factor(lpb_ctx* ctx);
/* Rhat + solve_newton_equations (newton_equations.rs:176-225): (u,v) for the given rhat, and
 * (p,q) = sym_solve(c, b) on the predictor call (cached for the corrector: it only depends on M). */
int lpb_direction(lpb_ctx* ctx, const lpb_direction_in* in, double tau, double kappa,
                  lpb_direction_out* out);
/* delta.rs:33-37 (d_x, d_y, d_z from d_tau) fused with the vector part of the ratio test
 * (feasible_point.rs:61-62): alpha_xz[0] = min(1, min_{dx<0} x/-dx), [1] same for z. */
int lpb_assemble_delta(lpb_ctx* ctx, double d_tau, double alpha_xz[2]);
/* FeasiblePoint::do_step for x, y, z (feasible_point.rs:76-106), clamping x, z at 1 when ip. */
int lpb_do_step(lpb_ctx* ctx, double alpha, int ip);
/* x_out = x / tau (mod.rs:231) and fun = c . x_out + c0 (linear_program.rs:61-63). */
int lpb_extract_x(lpb_ctx* ctx, double tau, double* x_out, double* fun);

/* ------------------------------------------------------------------ batched mode
 * `batch` independent small LPs of identical slack-form dims (m x n), one CTA per problem, the
 * whole solve_normal_form loop on device.  A: batch*m*n, b: batch*m, c: batch*n; outputs
 * x_out: batch*n (x/tau, slack form), fun/iterations/status: batch. */
int lpb_solve_batched(int64_t batch, int64_t m, int64_t n, const double* A, const double* b,
                      const double* c, const lpb_options* opts, double* x_out, double* fun,
                      int64_t* iterations, int32_t* status, int mem, void* stream);
/* Same arguments and outputs as lpb_solve_batched, for 1 <= m <= 128.  The kernel follows from the shape: the
 * shared-memory kernel of lpb_solve_batched (K6) where it accepts (m, n) -- m <= 64 and A beside M within 227 KB
 * of shared memory, slack block not counted -- else K8, which reads A through L2 and keeps M and the vectors
 * (about 80 n + 8 m^2 bytes; (128, 768) fits) in shared memory.  Other shapes: LPB_ERR_UNSUPPORTED, checked
 * before any device is touched; lpb_last_error names the limit. */
int lpb_solve_many(int64_t batch, int64_t m, int64_t n, const double* A, const double* b,
                   const double* c, const lpb_options* opts, double* x_out, double* fun,
                   int64_t* iterations, int32_t* status, int mem, void* stream);
/* lpb_solve_many's shape limits for one LP of m x n, on the host: LPB_OK if lpb_solve_many (and
 * lpb_solve_many_ragged) can run the shape, LPB_ERR_UNSUPPORTED naming the limit (lpb_last_error) if not,
 * LPB_ERR_BAD_ARGUMENT for m <= 0 or n <= 0. */
int lpb_solve_many_check(int64_t m, int64_t n);
/* A list of `batch` independent slack-form LPs of different shapes, solved in one call.  m, n: host arrays of
 * `batch` dims.  A, b, c are packed in list order: LP i's A (row-major, m[i] x n[i]) starts at sum_{k<i} m[k] n[k],
 * its b at sum_{k<i} m[k], its c at sum_{k<i} n[k]; x_out is packed like c, fun / iterations / status hold `batch`
 * entries.  `mem` as for lpb_solve_batched.  Each LP gets its own slack structure and the kernel lpb_solve_many
 * picks for a batch of that LP alone, and its outputs are bit-identical to such a call: the order of the list and
 * the other LPs in it do not change them.  LPB_ERR_BAD_ARGUMENT for null pointers or non-positive dims,
 * LPB_ERR_UNSUPPORTED if any LP is outside lpb_solve_many's limits (lpb_last_error names the LP and the limit; the
 * whole call is refused); both checked before any device is touched. */
int lpb_solve_many_ragged(int64_t batch, const int64_t* m, const int64_t* n,
                          const double* A, const double* b, const double* c,
                          const lpb_options* opts, double* x_out, double* fun,
                          int64_t* iterations, int32_t* status, int mem, void* stream);
/* Free the device staging memory lpb_solve_batched / lpb_solve_many / lpb_solve_many_ragged keep between calls with
 * host inputs, and the page-locked host buffers of lpb_solve_many_ragged (per calling thread). */
int lpb_release_workspaces(void);

/* ------------------------------------------------------------------ kernel entry points
 * Device-pointer forms of the hot kernels (parity tests and roofline measurements). */
/* K1: lower(M) = A diag(d) A^T  (newton_equations.rs:54-57).  d == NULL means d = 1. */
int lpb_k_syrk_adat(lpb_ctx* ctx, int64_t m, int64_t n, const double* dA, int64_t lda,
                    const double* d_d, double* dM, int64_t ldm);
/* K2: in-place lower Cholesky of the m x m row-major matrix (M.cholesky(), :130 / potrf :88).
 * *info_host = 0 ok, j+1 = first bad pivot. */
int lpb_k_potrf(lpb_ctx* ctx, int64_t m, double* dM, int64_t ldm, int32_t* info_host);
/* K3: solve L L^T X = B in place, B column-major m x nrhs (nrhs 1 or 2) (solvec, :154 / :100).
 * If dL is the matrix the last lpb_k_potrf on this context factored, the fused fast path (stored
 * inverted diagonal blocks) is used; any other L goes through plain blocked substitution. */
int lpb_k_potrs(lpb_ctx* ctx, int64_t m, const double* dL, int64_t ldm, double* dB, int64_t nrhs);
/* K4: out = A w (gemv_n) / out = A^T v (gemv_t), raw products. */
int lpb_k_gemv_n(lpb_ctx* ctx, int64_t m, int64_t n, const double* dA, int64_t lda,
                 const double* d_w, double* d_out);
int lpb_k_gemv_t(lpb_ctx* ctx, int64_t m, int64_t n, const double* dA, int64_t lda,
                 const double* d_v, double* d_out);

/* ------------------------------------------------------------------ measurement
 * Device time per phase of the last lpb_solve (CUDA events on the context's stream). */
typedef struct lpb_profile {
  double total_ms;      /* whole loop */
  double syrk_ms;       /* K1 */
  double potrf_ms;      /* K2 */
  double solve_ms;      /* K3 */
  double sweep_ms;      /* K4 (GEMV sweeps over A incl. their epilogues) */
  double vector_ms;     /* K5 */
  double comm_ms;       /* K7 collectives */
  int64_t launches;     /* kernels launched by this library during the last solve */
  int64_t iterations;
  int64_t syrk_launches, potrf_launches;
  int64_t syrk_cols;    /* columns of A the SYRK contracts over: n minus the trailing singleton (slack) columns,
                           which are folded into the diagonal of M (executed flop = m (m + 1) syrk_cols) */
} lpb_profile;
int lpb_get_profile(lpb_ctx* ctx, lpb_profile* out);
/* FP64 tensor (DMMA) ISSUE peak of the device this context lives on, measured now: a register-only loop of
 * independent mma.sync.m8n8k4.f64 (32 accumulator fragments per warp, 8 warps per SM, every SM) run back to
 * back for about `seconds` (0.05 .. 2) on the context's stream.  bench.py reports it as roofline.peak_measured
 * beside the nominal 40 TFLOP/s (MEASURED_PEAKS.json carries no FP64 figure).  No reference counterpart. */
int lpb_measure_dmma_peak(lpb_ctx* ctx, double seconds, double* tflops_out);
/* Kernels launched by this library on this context since creation (all entry points). */
int64_t lpb_launch_count(lpb_ctx* ctx);
/* Tuning / debug knobs.  "syrk_impl": 0 = DMMA+TMA, 1 = plain DFMA reference kernels (parity tests
 * bisect with it); "solve_impl": 0 = single-launch pipelined solve (tagged hand-off, full block inverses),
 * 1 = one launch per 128-block step, 2 = plain substitution, 3 = the flag-based pipelined solve with blocked
 * substitution; "refine": iterative-refinement steps per sym_solve (default 0 = the reference's plain
 * factor-and-solve); "syrk_flush_blocks": K-blocks of 16 columns K1 sums in registers between two folds into M
 * (power of two >= 32, default 32); "syrk_chain": 1 = one register chain over the whole K extent (round-1 kernel);
 * "syrk_tail_split": 0 = never cut the tiles of a short last wave of K1 into K-parts (default 1);
 * "solve_grid_cap": > 0 caps the pipelined solve's grid (tests: several block rows per CTA);
 * "profile": 1 = record per-phase events; "structure": 0 = contract the SYRK over every column of A
 * (default 1: trailing singleton columns -- the slack block -- are folded into the diagonal of M).  Unknown key -> BAD_ARGUMENT. */
int lpb_set_option(lpb_ctx* ctx, const char* key, int64_t value);

/* Copy a named device buffer to the host (debugging / parity tests): "M" (m x ldm), n-vectors
 * "x" "z" "c" "rD" "dinv" "dx" "dz" "p" "u", m-vectors "b" "y" "rP" "dy", "t" / "W" (2 m).  Returns the
 * number of doubles the buffer holds (-1: unknown name) and copies min(count, that) of them. */
int64_t lpb_debug_read(lpb_ctx* ctx, const char* name, double* out, int64_t count);
/* Named debug counters of the context: "potrf_verify_runs" / "potrf_verify_mismatches" (option "potrf_verify" = 1
 * factors every M twice and compares the two factors bit for bit: a mismatch is a race), "refactorisations"
 * (option "regularize": factorisations repeated with a diagonal shift).  -1: unknown name. */
int64_t lpb_debug_counter(lpb_ctx* ctx, const char* name);

/* ---- opt-in presolve (host only; no reference counterpart: the crate's own TODO, CONTRIBUTING.md:8).
 * Works on the slack form (the output of lpb_build_slack_form): drops empty rows and rows that are multiples of an
 * earlier row (infeasible -> status LPB_ERR_INFEASIBLE if their right-hand sides disagree), then `scale_passes` rounds
 * of power-of-two geometric row / column equilibration.  Presolved problem: min (C c)'y st (R A C) y = R b, y >= 0,
 * x = C y.  Columns are never removed, so n and n_slack carry over. */
typedef struct lpb_presolve lpb_presolve;
int lpb_presolve_create(lpb_presolve** out, int64_t m, int64_t n, const double* A, int64_t lda, const double* b,
                        const double* c, int64_t n_slack, int scale_passes);
int lpb_presolve_info(const lpb_presolve* p, int64_t* m_out, int64_t* n_out, int64_t* n_slack_out,
                      int64_t* dropped_empty, int64_t* dropped_duplicate, int* status);
int lpb_presolve_get(const lpb_presolve* p, double* A_out, int64_t lda_out, double* b_out, double* c_out);
int lpb_presolve_restore_x(const lpb_presolve* p, const double* y, double* x);
int lpb_presolve_destroy(lpb_presolve* p);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* LPB200_H_ */
