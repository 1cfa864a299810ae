// lpb_api.cu -- the CUDA device context and the extern "C" boundary (include/lpb200.h).
//
// `CudaDev` implements the phase calls that lp_b200/csrc/ipm_driver.hpp drives; lpb_solve is that
// driver instantiated on it.  State layout in HBM (all FP64):
//   A   m x lda   row-major slack-form constraint matrix (lda = n rounded up to 16 doubles)
//   M   m x ldm   normal matrix, overwritten in place by its lower Cholesky factor
//   n-vectors: c x z rD dinv xs r1 p u dx dz xo       m-vectors: b y rP dy t[2] W[2] (W0 = v, W1 = q)
// Column-sharded contexts (world > 1) hold n_local columns of A and of every n-vector; m-vectors,
// M and all scalars are replicated, with NCCL all-reduces where SURVEY.md 8(e) says.
#include <nccl.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "ipm_driver.hpp"
#include "kernels.hpp"

namespace lpb {
int64_t gemv_t_partials_doubles(int64_t m, int64_t n);
int batched_launch(int64_t batch, int m, int n, const double* dA, const double* db, const double* dc,
                   const lpb_options& o, double* dx, double* dfun, int64_t* dit, int32_t* dst, cudaStream_t stream);
int solve_many_check_shape(int64_t m, int64_t n);
int solve_many_launch(int64_t batch, int m, int n, const double* dA, const double* db, const double* dc,
                      const lpb_options& o, double* dx, double* dfun, int64_t* dit, int32_t* dst, cudaStream_t stream);
int ragged_scan(int64_t lo, int64_t cnt, const LpDesc* ddesc, const double* dA, int* ns_dev, cudaStream_t stream);
int ragged_launch(int64_t lo, int64_t cnt, LpDesc* desc_host, const int* ns_host, int* order_host, LpDesc* desc_dev,
                  int* order_dev, const double* dA, const double* db, const double* dc, const lpb_options& o,
                  double* dx, double* dfun, int64_t* dit, int32_t* dst, cudaStream_t stream);
}

using namespace lpb;

enum Phase { PH_SYRK = 0, PH_POTRF, PH_SOLVE, PH_SWEEP, PH_VEC, PH_COMM, PH_COUNT };

struct PhaseRec {
  int phase;
  cudaEvent_t a, b;
};

struct lpb_ctx {
  LaunchCtx lc;
  bool own_stream = false;
  bool has_problem = false;
  int64_t m = 0, n = 0, n_global = 0, col0 = 0, lda = 0, ldm = 0;
  double c0 = 0.0;
  double *A = nullptr, *M = nullptr;
  double *b = nullptr, *y = nullptr, *rP = nullptr, *dy = nullptr, *t = nullptr, *W = nullptr, *R = nullptr;
  // Column structure (analyze_structure): columns [n_dense, n) are singleton / zero columns -- the slack block
  // [I; 0] of linear_program.rs:145-156 -- folded into the diagonal of M instead of being contracted over.
  int64_t n_dense = 0, n_singleton = 0;
  int use_structure = 1;
  int* sgl_col = nullptr;     // m: local column (>= n_dense) whose only non-zero sits in this row, or -1
  double* sgl_val = nullptr;  // m: that entry
  int* col_row = nullptr;     // n: for columns >= n_dense, the row of their only non-zero, or -1 (all-zero column)
  double* col_val = nullptr;  // n: ... and its value
  int refine = 0;  // iterative-refinement steps taken per sym_solve: 0 (default) = the plain factor-and-solve of the reference
  int refine_max = 0;  // > refine: take further steps (up to this many) while the d_tau scalars still move (off by default)
  int64_t refine_steps_taken = 0;
  int regularize = 0;        // 1 = retry a failed factorisation with a shifted diagonal (see form_and_factor)
  bool shifted_now = false;  // the factor of the current iteration belongs to a shifted M
  double *c = nullptr, *x = nullptr, *z = nullptr, *rD = nullptr, *dinv = nullptr, *xs = nullptr, *r1 = nullptr,
         *p = nullptr, *u = nullptr, *dx = nullptr, *dz = nullptr, *xo = nullptr;
  bool have_pq = false;
  double cp = 0.0, bq = 0.0;
  int nan_pq = 0;
  int syrk_impl = 0;
  bool profile = true;
  int rank = 0, world = 1;
  ncclComm_t comm = nullptr;
  int packed_allreduce = 1;             // sharded: all-reduce only the lower triangle of M (packed), not the square
  double* tri_buf = nullptr;            // its staging buffer (tri_packed_doubles(m))
  int potrf_verify = 0;                 // debug: factor every M twice and compare the two factors bit for bit
  double *vfy1 = nullptr, *vfy2 = nullptr;
  int64_t vfy_mismatch = 0, vfy_runs = 0;
  int64_t refactorisations = 0;         // option "regularize": factorisations repeated with a diagonal shift
  bool check_replicas = false;          // debug: compare checksums of replicated buffers across ranks
  unsigned long long* chk_dev = nullptr;  // 2 words: {checksum, ~checksum}
  unsigned long long* chk_host = nullptr; // pinned
  SolveOutput last;
  lpb_profile prof;
  std::vector<cudaEvent_t> ev_free;
  std::vector<PhaseRec> recs;
  std::vector<void*> allocs;
};

namespace {

#define LPB_NCCL(call)                                                                      \
  do {                                                                                      \
    ncclResult_t r__ = (call);                                                              \
    if (r__ != ncclSuccess) {                                                               \
      set_last_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, ncclGetErrorString(r__)); \
      return LPB_ERR_NCCL;                                                                  \
    }                                                                                       \
  } while (0)

int dev_alloc(lpb_ctx* c, double** p, int64_t count) {
  void* q = nullptr;
  if (count < 1) count = 1;
  LPB_CUDA(cudaMalloc(&q, sizeof(double) * (size_t)count));
  c->allocs.push_back(q);
  *p = static_cast<double*>(q);
  return LPB_OK;
}

struct PhaseTimer {
  lpb_ctx* c;
  PhaseRec rec;
  bool on;
  PhaseTimer(lpb_ctx* ctx, int phase) : c(ctx), on(ctx->profile) {
    if (!on) return;
    rec.phase = phase;
    rec.a = take();
    rec.b = take();
    if (rec.a && rec.b) cudaEventRecord(rec.a, c->lc.stream);
  }
  ~PhaseTimer() {
    if (!on || !rec.a || !rec.b) return;
    cudaEventRecord(rec.b, c->lc.stream);
    c->recs.push_back(rec);
  }
  cudaEvent_t take() {
    if (!c->ev_free.empty()) {
      cudaEvent_t e = c->ev_free.back();
      c->ev_free.pop_back();
      return e;
    }
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
    return e;
  }
};

void profile_reset(lpb_ctx* c) {
  for (auto& r : c->recs) {
    c->ev_free.push_back(r.a);
    c->ev_free.push_back(r.b);
  }
  c->recs.clear();
  std::memset(&c->prof, 0, sizeof(c->prof));
}

void profile_collect(lpb_ctx* c) {
  double ms[PH_COUNT] = {0};
  for (auto& r : c->recs) {
    float f = 0.f;
    if (cudaEventElapsedTime(&f, r.a, r.b) == cudaSuccess) ms[r.phase] += f;
    c->ev_free.push_back(r.a);
    c->ev_free.push_back(r.b);
  }
  c->recs.clear();
  c->prof.syrk_ms = ms[PH_SYRK];
  c->prof.potrf_ms = ms[PH_POTRF];
  c->prof.solve_ms = ms[PH_SOLVE];
  c->prof.sweep_ms = ms[PH_SWEEP];
  c->prof.vector_ms = ms[PH_VEC];
  c->prof.comm_ms = ms[PH_COMM];
}

// One NCCL communicator per process (one process per GPU): ncclCommInitRank costs seconds, contexts
// come and go with every solve.  Created by the first lpb_create_sharded that carries a unique id,
// shared by later contexts (nccl_unique_id == NULL), destroyed by lpb_comm_finalize.
struct ProcessComm {
  ncclComm_t comm = nullptr;
  int rank = -1, world = 0;
  int refs = 0;  // live contexts holding `comm`: it is neither rebuilt nor destroyed under them
};
ProcessComm g_comm;
std::mutex g_comm_mu;

// device staging arena of lpb_solve_batched / lpb_solve_many / lpb_solve_many_ragged for host inputs (per host
// thread, grow-only); the ragged call also keeps its descriptors, structure results and launch order there
thread_local void* g_batched_ws = nullptr;
thread_local cudaStream_t g_batched_copy_stream = nullptr;  // uploads of host inputs, see run_batched
thread_local cudaEvent_t g_batched_ev[4] = {nullptr, nullptr, nullptr, nullptr};
thread_local size_t g_batched_ws_cap = 0;
// page-locked host side of the ragged call's descriptors, structure results and launch order (grow-only)
thread_local void* g_ragged_host = nullptr;
thread_local size_t g_ragged_host_cap = 0;

int allreduce(lpb_ctx* c, double* buf, int64_t count, ncclRedOp_t op) {
  if (c->world <= 1) return LPB_OK;
  PhaseTimer tm(c, PH_COMM);
  LPB_NCCL(ncclAllReduce(buf, buf, (size_t)count, ncclDouble, op, c->comm, c->lc.stream));
  return LPB_OK;
}

// All ranks learn the worst status of any rank (one int all-reduce + sync): a rank-local failure (upload,
// allocation) then fails the call on EVERY rank instead of leaving the others blocked in the next collective.
int agree_status(lpb_ctx* c, int rc) {
  if (c->world <= 1 || !c->comm || !c->chk_dev) return rc;
  int* flag = reinterpret_cast<int*>(c->chk_dev);  // 16 bytes of device scratch owned by the context
  const int mine = rc == LPB_OK ? 0 : 1;
  if (cudaMemcpyAsync(flag, &mine, sizeof(int), cudaMemcpyHostToDevice, c->lc.stream) != cudaSuccess) return LPB_ERR_CUDA;
  if (ncclAllReduce(flag, flag, 1, ncclInt32, ncclMax, c->comm, c->lc.stream) != ncclSuccess) return LPB_ERR_NCCL;
  int any = 0;
  if (cudaMemcpyAsync(&any, flag, sizeof(int), cudaMemcpyDeviceToHost, c->lc.stream) != cudaSuccess ||
      cudaStreamSynchronize(c->lc.stream) != cudaSuccess)
    return LPB_ERR_CUDA;
  if (rc == LPB_OK && any) {
    set_last_error("another rank of the sharded problem failed");
    return LPB_ERR_NCCL;
  }
  return rc;
}

// Debug (option "check_replicas"): every rank must hold the same bits of a replicated buffer.  All
// ranks learn the verdict from the same all-reduce, so a divergence is reported on every rank at once
// instead of dead-locking the ranks that carry on.
int check_replicated(lpb_ctx* c, const char* what, const double* v, int64_t rows, int64_t cols, int64_t ld, int lower) {
  if (c->world <= 1 || !c->check_replicas) return LPB_OK;
  LPB_TRY(k_checksum(c->lc, v, rows, cols, ld, lower, c->chk_dev));
  LPB_CUDA(cudaMemcpyAsync(c->chk_dev + 1, c->chk_dev, sizeof(unsigned long long), cudaMemcpyDeviceToDevice,
                           c->lc.stream));
  LPB_NCCL(ncclAllReduce(c->chk_dev, c->chk_dev, 1, ncclUint64, ncclMin, c->comm, c->lc.stream));
  LPB_NCCL(ncclAllReduce(c->chk_dev + 1, c->chk_dev + 1, 1, ncclUint64, ncclMax, c->comm, c->lc.stream));
  LPB_CUDA(cudaMemcpyAsync(c->chk_host, c->chk_dev, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                           c->lc.stream));
  LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
  if (c->chk_host[0] != c->chk_host[1]) {
    set_last_error("replicas diverged: %s differs between ranks (iteration %lld)", what,
                   (long long)c->prof.syrk_launches);
    return LPB_ERR_NCCL;
  }
  return LPB_OK;
}

// Fold partials, all-reduce the first `n_sharded` values (they are sums / mins over this rank's
// columns), fetch all `nvals` to the host.
int finish_scalars(lpb_ctx* c, const RedSpec& spec, int n_sharded, ncclRedOp_t op) {
  LPB_TRY(reduce_finalize(c->lc, spec));
  if (n_sharded > 0) LPB_TRY(allreduce(c, c->lc.red_out, n_sharded, op));
  return fetch_scalars(c->lc, spec.nvals);
}

struct CudaDev {
  lpb_ctx* c;

  // t_k = A (dinv? dinv * w_k : w_k): the dense columns through the GEMV kernel, the trailing singleton columns
  // (the slack block) as one scaled add per row -- they are never read from A (lpb_ctx::n_dense).
  int sweep_n(const double* dinv, const double* w0, const double* w1, double* t0, double* t1, int nrhs) {
    if (c->n_dense > 0) {
      LPB_TRY(k_gemv_n(c->lc, c->m, c->n_dense, c->A, c->lda, dinv, w0, w1, t0, t1, nrhs));
    } else {
      LPB_CUDA(cudaMemsetAsync(t0, 0, sizeof(double) * (size_t)c->m, c->lc.stream));
      if (nrhs == 2) LPB_CUDA(cudaMemsetAsync(t1, 0, sizeof(double) * (size_t)c->m, c->lc.stream));
    }
    if (c->n_singleton > 0)
      LPB_TRY(k_slack_add(c->lc, c->m, c->sgl_col, c->sgl_val, dinv, w0, w1, t0, t1, nrhs));
    return LPB_OK;
  }
  // row-chunk partials of A^T v_k over the dense columns; `tail` tells the epilogue how to form the rest
  int sweep_t(const double* v0, const double* v1, int nrhs, int* nchunks, TailCols* tail) {
    *nchunks = 0;
    if (c->n_dense > 0) LPB_TRY(k_gemv_t_partials(c->lc, c->m, c->n_dense, c->A, c->lda, v0, v1, nrhs, nchunks));
    *tail = TailCols{c->n_dense, c->col_row, c->col_val, v0, v1};
    return LPB_OK;
  }

  int blind_start() {  // feasible_point.rs:24-39
    PhaseTimer tm(c, PH_VEC);
    LPB_TRY(k_fill(c->lc, c->x, c->n, 1.0));
    LPB_TRY(k_fill(c->lc, c->z, c->n, 1.0));
    LPB_TRY(k_fill(c->lc, c->y, c->m, 0.0));
    c->have_pq = false;
    return LPB_OK;
  }

  int residuals(double tau, double kappa, lpb_residual_scalars* o) {
    (void)kappa;
    RedSpec spec;
    spec.nvals = 5;
    int nb_n = 0, nb_m = 0, nchunks = 0;
    {
      PhaseTimer tm(c, PH_SWEEP);
      LPB_TRY(sweep_n(nullptr, c->x, nullptr, c->t, nullptr, 1));
    }
    LPB_TRY(allreduce(c, c->t, c->m, ncclSum));
    LPB_TRY(check_replicated(c, "A x after the all-reduce", c->t, 1, c->m, c->m, 0));
    LPB_TRY(check_replicated(c, "y", c->y, 1, c->m, c->m, 0));
    {
      PhaseTimer tm(c, PH_SWEEP);
      LPB_TRY(k_resid_p(c->lc, c->m, tau, c->b, c->t, c->y, c->rP, 3, &nb_m));
      TailCols tail;
      LPB_TRY(sweep_t(c->y, nullptr, 1, &nchunks, &tail));
      LPB_TRY(k_resid_d(c->lc, c->n, nchunks, tau, c->c, c->z, c->x, c->rD, 0, &nb_n, &tail));
    }
    spec.nblocks[0] = spec.nblocks[1] = spec.nblocks[2] = nb_n;
    spec.nblocks[3] = spec.nblocks[4] = nb_m;
    LPB_TRY(finish_scalars(c, spec, 3, ncclSum));
    const double* h = c->lc.red_host;
    o->nrm_rd = std::sqrt(h[0]);
    o->cx = h[1];
    o->xz = h[2];
    o->nrm_rp = std::sqrt(h[3]);
    o->by = h[4];
    return LPB_OK;
  }

  // M = A diag(x / z) A^T (lower triangle), all-reduced over the column shards   (newton_equations.rs:54-57)
  int form_normal_matrix() {
    {
      PhaseTimer tm(c, PH_SYRK);
      if (c->n_dense <= 0)  // a shard made of slack columns only
        LPB_CUDA(cudaMemsetAsync(c->M, 0, sizeof(double) * (size_t)(c->m * c->ldm), c->lc.stream));
      else if (c->syrk_impl == 1)
        LPB_TRY(k_syrk_simple(c->lc, c->m, c->n_dense, c->A, c->lda, c->dinv, c->M, c->ldm));
      else
        LPB_TRY(k_syrk_dmma(c->lc, c->m, c->n_dense, c->A, c->lda, c->dinv, c->M, c->ldm));
      if (c->n_singleton > 0) LPB_TRY(k_diag_add(c->lc, c->m, c->M, c->ldm, c->sgl_col, c->sgl_val, c->dinv));
      c->prof.syrk_launches++;
      c->prof.syrk_cols = c->n_dense;
    }
    if (c->world > 1 && c->packed_allreduce) {
      const int64_t cnt = tri_packed_doubles(c->m);
      if (!c->tri_buf) {  // normally allocated by lpb_create_sharded; option toggled on later
        LPB_TRY(dev_alloc(c, &c->tri_buf, cnt));
        LPB_CUDA(cudaMemsetAsync(c->tri_buf, 0, sizeof(double) * (size_t)cnt, c->lc.stream));  // padding stays finite
      }
      {
        PhaseTimer tm(c, PH_COMM);
        LPB_TRY(k_tri_pack(c->lc, c->M, c->ldm, c->m, c->tri_buf, true));
      }
      LPB_TRY(allreduce(c, c->tri_buf, cnt, ncclSum));
      {
        PhaseTimer tm(c, PH_COMM);
        LPB_TRY(k_tri_pack(c->lc, c->M, c->ldm, c->m, c->tri_buf, false));
      }
    } else {
      LPB_TRY(allreduce(c, c->M, c->m * c->ldm, ncclSum));
    }
    return check_replicated(c, "M after the all-reduce", c->M, c->m, c->m, c->ldm, 1);
  }

  // Cholesky of M in place; *info_out = 0 or first bad pivot + 1 (agreed across ranks)   (newton_equations.rs:129-132)
  int factor_normal_matrix(int* info_out) {
    const size_t mbytes = sizeof(double) * (size_t)(c->m * c->ldm);
    if (c->potrf_verify) {
      if (!c->vfy1) {
        LPB_TRY(dev_alloc(c, &c->vfy1, c->m * c->ldm));
        LPB_TRY(dev_alloc(c, &c->vfy2, c->m * c->ldm));
      }
      LPB_CUDA(cudaMemcpyAsync(c->vfy1, c->M, mbytes, cudaMemcpyDeviceToDevice, c->lc.stream));
    }
    {
      PhaseTimer tm(c, PH_POTRF);
      LPB_TRY(k_potrf(c->lc, c->m, c->M, c->ldm, c->syrk_impl));
      c->prof.potrf_launches++;
    }
    if (c->potrf_verify) {  // same input, second run: any bit that differs is a race
      LPB_CUDA(cudaMemcpyAsync(c->vfy2, c->M, mbytes, cudaMemcpyDeviceToDevice, c->lc.stream));
      LPB_CUDA(cudaMemcpyAsync(c->M, c->vfy1, mbytes, cudaMemcpyDeviceToDevice, c->lc.stream));
      const int saved = c->lc.sync_each_launch;
      if (c->potrf_verify == 2) c->lc.sync_each_launch = 1;
      LPB_TRY(k_potrf(c->lc, c->m, c->M, c->ldm, c->syrk_impl));
      c->lc.sync_each_launch = saved;
      unsigned long long* d3 = nullptr;
      LPB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d3), 3 * sizeof(unsigned long long)));
      LPB_TRY(k_diff(c->lc, c->M, c->vfy2, c->m, c->m, c->ldm, 1, d3));
      unsigned long long h3[3];
      LPB_CUDA(cudaMemcpyAsync(h3, d3, sizeof(h3), cudaMemcpyDeviceToHost, c->lc.stream));
      LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
      cudaFree(d3);
      c->vfy_runs++;
      if (h3[0]) {
        c->vfy_mismatch++;
        std::fprintf(stderr, "[potrf_verify] factorisation %lld: %llu entries differ between two runs on the same M; "
                     "first column %llu, first row %llu\n", (long long)c->vfy_runs, h3[0], h3[1], h3[2]);
      }
    }
    LPB_TRY(check_replicated(c, "the Cholesky factor", c->M, c->m, c->m, c->ldm, 1));
    if (c->world > 1) {  // every rank must take the same branch on a failed factorisation
      PhaseTimer tm(c, PH_COMM);
      LPB_NCCL(ncclAllReduce(c->lc.info_dev, c->lc.info_dev, 1, ncclInt32, ncclMax, c->comm, c->lc.stream));
    }
    LPB_CUDA(cudaMemcpyAsync(c->lc.info_host, c->lc.info_dev, sizeof(int), cudaMemcpyDeviceToHost, c->lc.stream));
    LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
    *info_out = *c->lc.info_host;
    return LPB_OK;
  }

  int form_and_factor() {  // newton_equations.rs:48-64
    {
      PhaseTimer tm(c, PH_VEC);
      LPB_TRY(k_dinv(c->lc, c->n, c->x, c->z, c->dinv));
    }
    LPB_TRY(form_normal_matrix());
    int info = 0;
    LPB_TRY(factor_normal_matrix(&info));
    c->have_pq = false;
    c->shifted_now = false;
    if (info == 0) return LPB_OK;
    // The reference gives up here (newton_equations.rs:63: any factorisation error -> NumericalProblem; its
    // Inverse / LeastSquares fallbacks only hang off a failed SOLVE, :201-209) and so does the default path.
    // Option "regularize" = 1 is the GPU analogue of that fallback chain for a failed FACTOR: M is formed again
    // and factored with a growing relative shift of its diagonal, M_ii (1 + delta); the regularised factor is then
    // only a preconditioner -- every sym_solve of this iteration runs >= 2 refinement steps against the exact
    // operator A D A^T (direction()), so the directions solve the unshifted normal equations.
    if (!c->regularize) return LPB_ERR_NUMERICAL_PROBLEM;
    double delta = 1e-13;
    for (int attempt = 0; attempt < 6 && info != 0; ++attempt, delta *= 100.0) {
      LPB_TRY(form_normal_matrix());
      {
        PhaseTimer tm(c, PH_VEC);
        LPB_TRY(k_diag_shift(c->lc, c->m, c->M, c->ldm, delta));
      }
      LPB_TRY(factor_normal_matrix(&info));
      c->refactorisations++;
    }
    if (info != 0) return LPB_ERR_NUMERICAL_PROBLEM;
    c->shifted_now = true;
    return LPB_OK;
  }

  int direction(const lpb_direction_in& in, double tau, double kappa, lpb_direction_out* o) {
    (void)tau;
    (void)kappa;
    const int with_pq = c->have_pq ? 0 : 1;
    const int nrhs = with_pq ? 2 : 1;
    const double gm = in.gamma * in.mu;
    const double a2 = in.alpha * in.alpha;
    const double s = (1.0 - in.alpha) * in.gamma * in.mu;
    const int mode = !in.corrector ? 0 : (in.ip ? 1 : 2);
    double* W0 = c->W;
    double* W1 = c->W + c->m;
    {
      PhaseTimer tm(c, PH_VEC);
      LPB_TRY(k_rhat(c->lc, c->n, mode, in.eta, gm, a2, s, c->x, c->z, c->rD, c->dx, c->dz, c->xs, c->r1));
    }
    {
      PhaseTimer tm(c, PH_SWEEP);
      LPB_TRY(sweep_n(c->dinv, c->r1, c->c, c->t, c->t + c->m, nrhs));
    }
    LPB_TRY(allreduce(c, c->t, c->m * nrhs, ncclSum));
    LPB_TRY(check_replicated(c, "A (Dinv r1) after the all-reduce", c->t, 1, c->m * nrhs, c->m * nrhs, 0));
    {
      PhaseTimer tm(c, PH_VEC);
      LPB_TRY(k_sym_fwd_rhs(c->lc, c->m, in.eta, c->rP, c->b, c->t, c->t + c->m, W0, W1, with_pq));
    }
    {
      PhaseTimer tm(c, PH_SOLVE);
      LPB_TRY(k_potrs(c->lc, c->m, c->M, c->ldm, c->W, nrhs, c->syrk_impl == 0));
    }
    LPB_TRY(check_replicated(c, "the solve output (v, q)", c->W, 1, c->m * nrhs, c->m * nrhs, 0));
    RedSpec spec;
    spec.nvals = 6;
    int nchunks = 0, nb_n = 0, nb_m = 0;
    {
      PhaseTimer tm(c, PH_SWEEP);
      TailCols tail;
      LPB_TRY(sweep_t(W0, W1, nrhs, &nchunks, &tail));
      LPB_TRY(k_sym_back(c->lc, c->n, nchunks, with_pq, c->dinv, c->r1, c->c, c->u, c->p, 0, &nb_n, &tail));
    }
    // OPTIONAL iterative refinement against the OPERATOR A Dinv A^T (not the stored M): the residual of
    //   M v = r2 + A Dinv r1   is   r2 - A u   with u = Dinv (A^T v - r1),   i.e.  rP*eta - A u  and  b - A p,
    // one more sweep each way and one more solve per step.  The reference has no such step and neither has the
    // default path (`refine` = 0).  History: with K1 summing each entry of M in ONE register chain (round 1, and what
    // a single cuBLAS DGEMM does) S = -c.p + b.q -- the denominator of d_tau next to kappa / tau, delta.rs:32;
    // mathematically p' Dinv^-1 p >= 0, numerically a difference of two numbers ~ the objective -- lost all its digits
    // late in the iteration and a refinement step was needed to follow the oracle's trajectory at C3.  The cause was
    // the summation order of M, not the factor or the solves (tools/diag_bisect_host.py); K1 now blocks the sum over
    // K (dmma_gemm.cu) and the unrefined solve tracks the oracle to 2e-8 in x (DESIGN.md section 5).
    // Steps: `refine` are always taken; up to `refine_max` while the scalars the host needs, S and T = -c.u + b.v,
    // still move by more than 1e-4 relative from one step to the next.  The regularised refactorisation
    // (`regularize`) forces two steps, because its factor belongs to a shifted M.  All ranks of a sharded solve see
    // the same all-reduced scalars and take the same decision.
    auto fetch = [&](double out[6]) -> int {
      {
        PhaseTimer tm(c, PH_SWEEP);
        LPB_TRY(k_dots_m(c->lc, c->m, c->b, W0, W1, with_pq, 3, &nb_m));
      }
      spec.nblocks[0] = spec.nblocks[1] = spec.nblocks[2] = nb_n;
      spec.nblocks[3] = spec.nblocks[4] = spec.nblocks[5] = nb_m;
      LPB_TRY(finish_scalars(c, spec, 3, ncclSum));
      for (int k = 0; k < 6; ++k) out[k] = c->lc.red_host[k];
      return LPB_OK;
    };
    const int steps_min = c->shifted_now ? std::max(c->refine, 2) : c->refine;
    const int steps_max = steps_min > 0 ? std::max(steps_min, c->refine_max) : 0;
    double cur[6] = {0, 0, 0, 0, 0, 0}, prev[6];
    bool have_cur = false;
    for (int step = 0; step < steps_max; ++step) {
      if (step >= steps_min) {  // an optional step: only if the last one still moved the scalars
        const double Sc = -cur[1] + cur[4], Sp = -prev[1] + prev[4];
        const double Tc = -cur[0] + cur[3], Tp = -prev[0] + prev[3];
        const bool s_ok = !with_pq || std::fabs(Sc - Sp) <= 1e-4 * std::fabs(Sc);
        const bool t_ok = std::fabs(Tc - Tp) <= 1e-4 * std::fabs(Tc) + 1e-13 * (std::fabs(cur[0]) + std::fabs(cur[3]));
        if (s_ok && t_ok) break;
      }
      if (step + 1 >= steps_min && steps_max > steps_min && !have_cur) {  // the value the next comparison starts from
        LPB_TRY(fetch(cur));
        have_cur = true;
      }
      double* R0 = c->R;
      double* R1 = c->R + c->m;
      {
        PhaseTimer tm(c, PH_SWEEP);
        LPB_TRY(sweep_n(nullptr, c->u, c->p, c->t, c->t + c->m, nrhs));
      }
      LPB_TRY(allreduce(c, c->t, c->m * nrhs, ncclSum));
      {
        PhaseTimer tm(c, PH_VEC);
        LPB_TRY(k_refine_rhs(c->lc, c->m, in.eta, c->rP, c->b, c->t, c->t + c->m, R0, R1, with_pq));
      }
      {
        PhaseTimer tm(c, PH_SOLVE);
        LPB_TRY(k_potrs(c->lc, c->m, c->M, c->ldm, c->R, nrhs, c->syrk_impl == 0));
      }
      {
        PhaseTimer tm(c, PH_VEC);
        LPB_TRY(k_add_inplace(c->lc, c->m * nrhs, c->R, c->W));
      }
      {
        PhaseTimer tm(c, PH_SWEEP);
        TailCols tail;
        LPB_TRY(sweep_t(W0, W1, nrhs, &nchunks, &tail));
        LPB_TRY(k_sym_back(c->lc, c->n, nchunks, with_pq, c->dinv, c->r1, c->c, c->u, c->p, 0, &nb_n, &tail));
      }
      c->refine_steps_taken++;
      if (have_cur) {
        for (int k = 0; k < 6; ++k) prev[k] = cur[k];
        LPB_TRY(fetch(cur));
      }
    }
    if (!have_cur) LPB_TRY(fetch(cur));
    const double* h = cur;
    if (with_pq) {
      c->cp = h[1];
      c->bq = h[4];
      c->nan_pq = (h[2] > 0.0 || h[5] > 0.0) ? 1 : 0;
      c->have_pq = true;
    }
    o->cu = h[0];
    o->bv = h[3];
    o->cp = c->cp;
    o->bq = c->bq;
    o->nan_pq = c->nan_pq;
    o->reserved = 0;
    return LPB_OK;
  }

  int assemble_delta(double d_tau, double axz[2]) {
    RedSpec spec;
    spec.nvals = 2;
    int nb = 0;
    {
      PhaseTimer tm(c, PH_VEC);
      LPB_TRY(k_assemble_delta_n(c->lc, c->n, d_tau, c->u, c->p, c->xs, c->x, c->z, c->dx, c->dz, 0, &nb));
      LPB_TRY(k_assemble_delta_m(c->lc, c->m, d_tau, c->W, c->W + c->m, c->dy));
    }
    spec.nblocks[0] = spec.nblocks[1] = nb;
    spec.op[0] = spec.op[1] = kRedMin;
    LPB_TRY(finish_scalars(c, spec, 2, ncclMin));
    axz[0] = c->lc.red_host[0];
    axz[1] = c->lc.red_host[1];
    return LPB_OK;
  }

  int do_step(double alpha, int ip) {
    PhaseTimer tm(c, PH_VEC);
    LPB_TRY(k_step(c->lc, c->n, alpha, ip, c->x, c->dx));
    LPB_TRY(k_step(c->lc, c->n, alpha, ip, c->z, c->dz));
    LPB_TRY(k_step(c->lc, c->m, alpha, 0, c->y, c->dy));
    return LPB_OK;
  }

  int extract_x(double tau, double* x_out, double* fun) {
    RedSpec spec;
    spec.nvals = 1;
    int nb = 0;
    LPB_TRY(k_extract_x(c->lc, c->n, tau, c->x, c->c, c->xo, 0, &nb));
    spec.nblocks[0] = nb;
    LPB_TRY(finish_scalars(c, spec, 1, ncclSum));
    if (x_out)
      LPB_CUDA(cudaMemcpyAsync(x_out, c->xo, sizeof(double) * c->n, cudaMemcpyDeviceToHost, c->lc.stream));
    LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
    if (fun) *fun = c->lc.red_host[0] + c->c0;  // linear_program.rs:61-63
    return LPB_OK;
  }
};

int check_device() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    set_last_error("no CUDA device visible; liblpb200 has no CPU fallback");
    return LPB_ERR_NO_DEVICE;
  }
  return LPB_OK;
}

int ctx_base_init(lpb_ctx* c, void* stream) {
  if (stream) {
    c->lc.stream = static_cast<cudaStream_t>(stream);
  } else {
    LPB_CUDA(cudaStreamCreateWithFlags(&c->lc.stream, cudaStreamNonBlocking));
    c->own_stream = true;
  }
  LPB_TRY(dev_alloc(c, &c->lc.red_partials, (int64_t)kMaxRedVals * kMaxRedBlocks));
  LPB_TRY(dev_alloc(c, &c->lc.red_out, kMaxRedVals + 1));
  LPB_CUDA(cudaMemsetAsync(c->lc.red_out, 0, sizeof(double) * (kMaxRedVals + 1), c->lc.stream));
  c->lc.fault_dev = reinterpret_cast<unsigned long long*>(c->lc.red_out + kMaxRedVals);
  LPB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&c->lc.red_host), sizeof(double) * (kMaxRedVals + 1)));
  LPB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&c->lc.info_host), sizeof(int)));
  void* q = nullptr;
  LPB_CUDA(cudaMalloc(&q, sizeof(int)));
  c->allocs.push_back(q);
  c->lc.info_dev = static_cast<int*>(q);
  LPB_CUDA(cudaMalloc(&q, 2 * sizeof(unsigned long long)));
  c->allocs.push_back(q);
  c->chk_dev = static_cast<unsigned long long*>(q);
  LPB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&c->chk_host), 2 * sizeof(unsigned long long)));
  std::memset(&c->prof, 0, sizeof(c->prof));
  return LPB_OK;
}

int ctx_alloc_vectors(lpb_ctx* c, int64_t m, int64_t n, bool with_matrices) {
  c->m = m;
  c->n = n;
  c->lda = round_up(n, 16);
  c->ldm = round_up(m, 16);
  c->lc.gemv_partials_cap = gemv_t_partials_doubles(m, n);
  LPB_TRY(dev_alloc(c, &c->lc.gemv_partials, c->lc.gemv_partials_cap));
  if (!with_matrices) return LPB_OK;
  LPB_TRY(dev_alloc(c, &c->A, m * c->lda));
  LPB_TRY(dev_alloc(c, &c->M, m * c->ldm));
  double** mv[] = {&c->b, &c->y, &c->rP, &c->dy};
  for (auto p : mv) LPB_TRY(dev_alloc(c, p, m));
  LPB_TRY(dev_alloc(c, &c->t, 2 * m));
  LPB_TRY(dev_alloc(c, &c->W, 2 * m));
  LPB_TRY(dev_alloc(c, &c->R, 2 * m));
  LPB_TRY(dev_alloc(c, &c->sgl_val, m));
  LPB_TRY(dev_alloc(c, &c->col_val, n));
  {
    void* q = nullptr;
    LPB_CUDA(cudaMalloc(&q, sizeof(int) * (size_t)(m + n)));
    c->allocs.push_back(q);
    c->sgl_col = static_cast<int*>(q);
    c->col_row = c->sgl_col + m;
  }
  double** nv[] = {&c->c, &c->x, &c->z, &c->rD, &c->dinv, &c->xs, &c->r1, &c->p, &c->u, &c->dx, &c->dz, &c->xo};
  for (auto p : nv) LPB_TRY(dev_alloc(c, p, round_up(n, 2)));
  LPB_CUDA(cudaMemsetAsync(c->A, 0, sizeof(double) * (size_t)(m * c->lda), c->lc.stream));
  LPB_CUDA(cudaMemsetAsync(c->M, 0, sizeof(double) * (size_t)(m * c->ldm), c->lc.stream));
  LPB_CUDA(cudaMemsetAsync(c->dx, 0, sizeof(double) * (size_t)round_up(n, 2), c->lc.stream));
  LPB_CUDA(cudaMemsetAsync(c->dz, 0, sizeof(double) * (size_t)round_up(n, 2), c->lc.stream));
  return LPB_OK;
}

// Find the trailing run of singleton / zero columns of the resident A (one pass over A on the device, the
// bookkeeping on the host) and fold it out of the SYRK: see lpb_ctx::n_dense.  The run must map its
// columns to DISTINCT rows (always true for a slack block), so the diagonal update needs no atomics and
// stays deterministic; otherwise, or when the run is shorter than one K-block, A is treated as dense.
int analyze_structure(lpb_ctx* c) {
  c->n_dense = c->n;
  c->n_singleton = 0;
  if (!c->use_structure || !c->A || c->n < 16) return LPB_OK;
  const int64_t n = c->n, m = c->m;
  int* d_int = nullptr;
  double* d_val = nullptr;
  LPB_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_int), sizeof(int) * (size_t)(2 * n)));
  if (cudaMalloc(reinterpret_cast<void**>(&d_val), sizeof(double) * (size_t)n) != cudaSuccess) {
    cudaFree(d_int);
    set_last_error("analyze_structure: out of device memory");
    return LPB_ERR_CUDA;
  }
  std::vector<int> h_int((size_t)(2 * n));
  std::vector<double> h_val((size_t)n);
  int rc = k_col_structure(c->lc, c->A, m, n, c->lda, d_int, d_int + n, d_val);
  if (rc == LPB_OK &&
      (cudaMemcpyAsync(h_int.data(), d_int, sizeof(int) * (size_t)(2 * n), cudaMemcpyDeviceToHost, c->lc.stream) !=
           cudaSuccess ||
       cudaMemcpyAsync(h_val.data(), d_val, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, c->lc.stream) !=
           cudaSuccess ||
       cudaStreamSynchronize(c->lc.stream) != cudaSuccess)) {
    set_last_error("analyze_structure: copy failed");
    rc = LPB_ERR_CUDA;
  }
  cudaFree(d_int);
  cudaFree(d_val);
  LPB_TRY(rc);
  const int* nnz = h_int.data();
  const int* row = h_int.data() + n;
  std::vector<int> col_of_row((size_t)m, -1);
  std::vector<double> sq((size_t)m, 0.0);
  int64_t nd = n, nsgl = 0;
  while (nd > 0) {
    const int64_t j = nd - 1;
    if (nnz[j] > 1) break;
    if (nnz[j] == 1) {
      const int r = row[j];
      if (r < 0 || r >= m || col_of_row[r] >= 0) break;
      col_of_row[r] = (int)j;
      sq[r] = h_val[j];  // the entry itself; squared on the device where M needs it
      ++nsgl;
    }
    --nd;
  }
  if (n - nd < 16) return LPB_OK;  // not worth a separate pass
  for (int64_t j = nd; j < n; ++j)  // column-indexed view of the same run, for the A^T v epilogues
    if (nnz[j] != 1) h_int[(size_t)(n + j)] = -1;
  LPB_CUDA(cudaMemcpyAsync(c->sgl_col, col_of_row.data(), sizeof(int) * (size_t)m, cudaMemcpyHostToDevice, c->lc.stream));
  LPB_CUDA(cudaMemcpyAsync(c->sgl_val, sq.data(), sizeof(double) * (size_t)m, cudaMemcpyHostToDevice, c->lc.stream));
  LPB_CUDA(cudaMemcpyAsync(c->col_row, row, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, c->lc.stream));
  LPB_CUDA(cudaMemcpyAsync(c->col_val, h_val.data(), sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, c->lc.stream));
  LPB_CUDA(cudaStreamSynchronize(c->lc.stream));  // the host vectors go out of scope
  c->n_dense = nd;
  c->n_singleton = nsgl;
  return LPB_OK;
}

int upload_problem(lpb_ctx* c, const double* A, int64_t lda, const double* b, const double* cc, double c0, int mem) {
  if (!A || !b || !cc || lda < c->n) {
    set_last_error("set_problem: null pointer or lda < n");
    return LPB_ERR_BAD_ARGUMENT;
  }
  const cudaMemcpyKind kind = mem == LPB_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  if (lda == c->lda && lda == c->n)  // contiguous on both sides: one linear copy at full PCIe / HBM rate
    LPB_CUDA(cudaMemcpyAsync(c->A, A, sizeof(double) * (size_t)(c->m * c->lda), kind, c->lc.stream));
  else
    LPB_CUDA(cudaMemcpy2DAsync(c->A, sizeof(double) * c->lda, A, sizeof(double) * lda, sizeof(double) * c->n, c->m,
                               kind, c->lc.stream));
  LPB_CUDA(cudaMemcpyAsync(c->b, b, sizeof(double) * c->m, kind, c->lc.stream));
  LPB_CUDA(cudaMemcpyAsync(c->c, cc, sizeof(double) * c->n, kind, c->lc.stream));
  if (std::getenv("LPB_TIME_CREATE")) {
    const auto t0 = std::chrono::steady_clock::now();
    LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    std::fprintf(stderr, "[upload] copies drained in %.1f ms after issue (%.1f GB/s)\n", ms,
                 8.0 * c->m * c->n / (ms * 1e-3) / 1e9);
  }
  LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
  c->c0 = c0;
  c->has_problem = true;
  c->have_pq = false;
  return analyze_structure(c);
}

void ctx_free(lpb_ctx* c) {
  if (!c) return;
  if (c->lc.stream) cudaStreamSynchronize(c->lc.stream);
  for (auto& r : c->recs) {
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  for (auto e : c->ev_free) cudaEventDestroy(e);
  for (void* p : c->allocs) cudaFree(p);
  if (c->lc.chol_ws) cudaFree(c->lc.chol_ws);
  if (c->lc.syrk_ws) cudaFree(c->lc.syrk_ws);
  if (c->lc.panel_buf) cudaFree(c->lc.panel_buf);
  k_peer_release(c->lc);
  for (int i = 0; i < 2; ++i)
    if (c->lc.panel_slot[i]) cudaFree(c->lc.panel_slot[i]);
  for (int e = 0; e < 4; ++e)
    if (c->lc.ev_dist[e]) cudaEventDestroy(c->lc.ev_dist[e]);
  if (c->lc.side_stream) {
    cudaStreamSynchronize(c->lc.side_stream);
    for (int e = 0; e < 2; ++e) {
      if (c->lc.ev_col[e]) cudaEventDestroy(c->lc.ev_col[e]);
      if (c->lc.ev_pan[e]) cudaEventDestroy(c->lc.ev_pan[e]);
    }
    cudaStreamDestroy(c->lc.side_stream);
  }
  if (c->lc.red_host) cudaFreeHost(c->lc.red_host);
  if (c->lc.info_host) cudaFreeHost(c->lc.info_host);
  if (c->chk_host) cudaFreeHost(c->chk_host);
  if (c->own_stream && c->lc.stream) cudaStreamDestroy(c->lc.stream);
  if (c->comm) {
    std::lock_guard<std::mutex> g(g_comm_mu);
    if (c->comm == g_comm.comm && g_comm.refs > 0) --g_comm.refs;
  }
  delete c;
}

int need_problem(lpb_ctx* c) {
  if (!c || !c->has_problem) {
    set_last_error("context has no problem attached");
    return LPB_ERR_BAD_ARGUMENT;
  }
  return LPB_OK;
}

size_t carve_up(size_t v) { return (v + 255) & ~(size_t)255; }

// Consecutive 256-byte aligned pieces of the staging arena.
struct Carver {
  char* p = nullptr;
  char* operator()(size_t bytes) {
    char* r = p;
    p += carve_up(bytes);
    return r;
  }
};

// The per-thread staging arena, grown to at least `need` bytes (its contents are not kept).
int batched_arena(size_t need, Carver* out) {
  if (g_batched_ws_cap < need) {
    if (g_batched_ws) cudaFree(g_batched_ws);
    g_batched_ws = nullptr;
    g_batched_ws_cap = 0;
    LPB_CUDA(cudaMalloc(&g_batched_ws, need));
    g_batched_ws_cap = need;
  }
  out->p = static_cast<char*>(g_batched_ws);
  return LPB_OK;
}

// The per-thread copy stream of host-input uploads and the four chunk events
int batched_copy_stream() {
  if (!g_batched_copy_stream) LPB_CUDA(cudaStreamCreateWithFlags(&g_batched_copy_stream, cudaStreamNonBlocking));
  for (int q = 0; q < 4; ++q)
    if (!g_batched_ev[q]) LPB_CUDA(cudaEventCreateWithFlags(&g_batched_ev[q], cudaEventDisableTiming));
  return LPB_OK;
}

using BatchedLaunch = int (*)(int64_t, int, int, const double*, const double*, const double*, const lpb_options&, double*,
                              double*, int64_t*, int32_t*, cudaStream_t);

// Runs `launch` (K6 alone, or solve_many's choice) over the batch: directly on device arrays, or with host arrays staged
// through the per-thread arena.
int run_batched(BatchedLaunch launch, int64_t batch, int64_t m, int64_t n, const double* A, const double* b, const double* c,
                const lpb_options& o, double* x_out, double* fun, int64_t* iterations, int32_t* status, int mem,
                cudaStream_t st) {
  if (mem == LPB_MEM_DEVICE) {
    LPB_TRY(launch(batch, (int)m, (int)n, A, b, c, o, x_out, fun, iterations, status, st));
    LPB_CUDA(cudaStreamSynchronize(st));
    return LPB_OK;
  }
  // Host arrays: stage through ONE cached device arena per host thread (grow-only; lpb_release_workspaces
  // frees it), so a call costs the three uploads, the kernel and the four downloads -- no cudaMalloc / cudaFree.
  const size_t sA = sizeof(double) * (size_t)(batch * m * n), sb = sizeof(double) * (size_t)(batch * m),
               sc = sizeof(double) * (size_t)(batch * n), s8 = sizeof(double) * (size_t)batch,
               s4 = sizeof(int32_t) * (size_t)batch;
  Carver carve;
  LPB_TRY(batched_arena(carve_up(sA) + carve_up(sb) + 2 * carve_up(sc) + 2 * carve_up(s8) + carve_up(s4), &carve));
  double* dA = reinterpret_cast<double*>(carve(sA));
  double* db = reinterpret_cast<double*>(carve(sb));
  double* dc = reinterpret_cast<double*>(carve(sc));
  double* dx = reinterpret_cast<double*>(carve(sc));
  double* df = reinterpret_cast<double*>(carve(s8));
  int64_t* dit = reinterpret_cast<int64_t*>(carve(s8));
  int32_t* dst = reinterpret_cast<int32_t*>(carve(s4));
  // The batch goes through in chunks: all uploads are queued on a copy stream up front, chunk i's kernel waits for its
  // own upload only, so the upload of chunk i + 1 (PCIe) runs under the kernel of chunk i and the downloads of chunk
  // i - 1.  At C4 the upload (558 MB, ~10 ms from pinned memory) and the kernel (~11 ms) used to add up.
  const int64_t nchunk = batch >= 1024 ? 4 : 1;
  LPB_TRY(batched_copy_stream());
  LPB_CUDA(cudaEventRecord(g_batched_ev[0], st));  // the copy stream starts behind whatever `st` holds already
  LPB_CUDA(cudaStreamWaitEvent(g_batched_copy_stream, g_batched_ev[0], 0));
  auto lo = [&](int64_t q) { return batch * q / nchunk; };
  for (int64_t q = 0; q < nchunk; ++q) {
    const int64_t b0 = lo(q), nb = lo(q + 1) - b0;
    LPB_CUDA(cudaMemcpyAsync(dA + b0 * m * n, A + b0 * m * n, sizeof(double) * (size_t)(nb * m * n), cudaMemcpyHostToDevice,
                             g_batched_copy_stream));
    LPB_CUDA(cudaMemcpyAsync(db + b0 * m, b + b0 * m, sizeof(double) * (size_t)(nb * m), cudaMemcpyHostToDevice,
                             g_batched_copy_stream));
    LPB_CUDA(cudaMemcpyAsync(dc + b0 * n, c + b0 * n, sizeof(double) * (size_t)(nb * n), cudaMemcpyHostToDevice,
                             g_batched_copy_stream));
    LPB_CUDA(cudaEventRecord(g_batched_ev[q], g_batched_copy_stream));
  }
  for (int64_t q = 0; q < nchunk; ++q) {
    const int64_t b0 = lo(q), nb = lo(q + 1) - b0;
    LPB_CUDA(cudaStreamWaitEvent(st, g_batched_ev[q], 0));
    LPB_TRY(launch(nb, (int)m, (int)n, dA + b0 * m * n, db + b0 * m, dc + b0 * n, o, dx + b0 * n, df + b0, dit + b0,
                   dst + b0, st));
    LPB_CUDA(cudaMemcpyAsync(x_out + b0 * n, dx + b0 * n, sizeof(double) * (size_t)(nb * n), cudaMemcpyDeviceToHost, st));
    LPB_CUDA(cudaMemcpyAsync(fun + b0, df + b0, sizeof(double) * (size_t)nb, cudaMemcpyDeviceToHost, st));
    LPB_CUDA(cudaMemcpyAsync(iterations + b0, dit + b0, sizeof(int64_t) * (size_t)nb, cudaMemcpyDeviceToHost, st));
    LPB_CUDA(cudaMemcpyAsync(status + b0, dst + b0, sizeof(int32_t) * (size_t)nb, cudaMemcpyDeviceToHost, st));
  }
  LPB_CUDA(cudaStreamSynchronize(st));
  return LPB_OK;
}

int batched_args(const char* who, int64_t batch, int64_t m, int64_t n, const double* A, const double* b, const double* c,
                 const lpb_options* opts, double* x_out, double* fun, int64_t* iterations, int32_t* status,
                 lpb_options* o) {
  if (batch <= 0 || m <= 0 || n <= 0 || !A || !b || !c || !x_out || !fun || !iterations || !status) {
    set_last_error("%s: null pointer or non-positive size", who);
    return LPB_ERR_BAD_ARGUMENT;
  }
  if (opts)
    *o = *opts;
  else
    options_default(o);
  return lpb_options_validate(o);
}

// A ragged list (lpb_solve_many_ragged) on device arrays, or with host arrays staged through the per-thread arena as
// in run_batched.  Per chunk: its upload, then its structure scan and the download of the scan's results, on the copy
// stream; the host waits for those results (while the previous chunk's kernels run), plans the chunk and queues its
// launches and downloads on `st`.  Device inputs are one chunk, scanned on `st`: one synchronisation before the plan.
int run_ragged(int64_t batch, const int64_t* m, const int64_t* n, const double* A, const double* b, const double* c,
               const lpb_options& o, double* x_out, double* fun, int64_t* iterations, int32_t* status, int mem,
               cudaStream_t st) {
  const bool host = mem != LPB_MEM_DEVICE;
  const size_t sd = sizeof(LpDesc) * (size_t)batch, si = sizeof(int) * (size_t)batch;
  if (g_ragged_host_cap < sd + 2 * si) {
    if (g_ragged_host) cudaFreeHost(g_ragged_host);
    g_ragged_host = nullptr;
    g_ragged_host_cap = 0;
    LPB_CUDA(cudaMallocHost(&g_ragged_host, sd + 2 * si));
    g_ragged_host_cap = sd + 2 * si;
  }
  LpDesc* hdesc = static_cast<LpDesc*>(g_ragged_host);
  int* hns = reinterpret_cast<int*>(hdesc + batch);
  int* hord = hns + batch;
  int64_t nA = 0, nb = 0, nc = 0;  // packed lengths
  for (int64_t i = 0; i < batch; ++i) {
    hdesc[i] = LpDesc{(int)m[i], (int)n[i], 0, 0, nA, nb, nc};
    nA += m[i] * n[i];
    nb += m[i];
    nc += n[i];
  }
  const size_t sA = sizeof(double) * (size_t)nA, sb = sizeof(double) * (size_t)nb, sc = sizeof(double) * (size_t)nc,
               s8 = sizeof(double) * (size_t)batch, s4 = sizeof(int32_t) * (size_t)batch;
  size_t need = carve_up(sd) + 2 * carve_up(si);
  if (host) need += carve_up(sA) + carve_up(sb) + 2 * carve_up(sc) + 2 * carve_up(s8) + carve_up(s4);
  Carver carve;
  LPB_TRY(batched_arena(need, &carve));
  LpDesc* ddesc = reinterpret_cast<LpDesc*>(carve(sd));
  int* dns = reinterpret_cast<int*>(carve(si));
  int* dord = reinterpret_cast<int*>(carve(si));
  const double* dA = host ? reinterpret_cast<double*>(carve(sA)) : A;
  const double* db = host ? reinterpret_cast<double*>(carve(sb)) : b;
  const double* dc = host ? reinterpret_cast<double*>(carve(sc)) : c;
  double* dx = host ? reinterpret_cast<double*>(carve(sc)) : x_out;
  double* df = host ? reinterpret_cast<double*>(carve(s8)) : fun;
  int64_t* dit = host ? reinterpret_cast<int64_t*>(carve(s8)) : iterations;
  int32_t* dst = host ? reinterpret_cast<int32_t*>(carve(s4)) : status;
  LPB_TRY(batched_copy_stream());
  cudaStream_t cs = st;
  if (host) {
    cs = g_batched_copy_stream;
    LPB_CUDA(cudaEventRecord(g_batched_ev[0], st));  // the copy stream starts behind whatever `st` holds already
    LPB_CUDA(cudaStreamWaitEvent(cs, g_batched_ev[0], 0));
  }
  // chunks by LP count; [a_off, b_off, c_off) of LP `lo(q)` .. the end of the packed arrays for q = nchunk
  const int64_t nchunk = host && batch >= 1024 ? 4 : 1;
  auto lo = [&](int64_t q) { return batch * q / nchunk; };
  auto off = [&](int64_t i, int which) -> int64_t {
    if (i == batch) return which == 0 ? nA : which == 1 ? nb : nc;
    return which == 0 ? hdesc[i].a_off : which == 1 ? hdesc[i].b_off : hdesc[i].c_off;
  };
  LPB_CUDA(cudaMemcpyAsync(ddesc, hdesc, sd, cudaMemcpyHostToDevice, cs));
  for (int64_t q = 0; q < nchunk; ++q) {
    const int64_t l0 = lo(q), l1 = lo(q + 1);
    if (host) {
      const double* src[3] = {A, b, c};
      const double* dst3[3] = {dA, db, dc};
      for (int w = 0; w < 3; ++w)
        LPB_CUDA(cudaMemcpyAsync(const_cast<double*>(dst3[w]) + off(l0, w), src[w] + off(l0, w),
                                 sizeof(double) * (size_t)(off(l1, w) - off(l0, w)), cudaMemcpyHostToDevice, cs));
    }
    LPB_TRY(ragged_scan(l0, l1 - l0, ddesc, dA, dns, cs));
    LPB_CUDA(cudaMemcpyAsync(hns + l0, dns + l0, sizeof(int) * (size_t)(l1 - l0), cudaMemcpyDeviceToHost, cs));
    LPB_CUDA(cudaEventRecord(g_batched_ev[q], cs));
  }
  for (int64_t q = 0; q < nchunk; ++q) {
    const int64_t l0 = lo(q), l1 = lo(q + 1);
    LPB_CUDA(cudaEventSynchronize(g_batched_ev[q]));
    if (host) LPB_CUDA(cudaStreamWaitEvent(st, g_batched_ev[q], 0));
    LPB_TRY(ragged_launch(l0, l1 - l0, hdesc, hns, hord, ddesc, dord, dA, db, dc, o, dx, df, dit, dst, st));
    if (!host) continue;
    const int64_t x0 = off(l0, 2), x1 = off(l1, 2);
    LPB_CUDA(cudaMemcpyAsync(x_out + x0, dx + x0, sizeof(double) * (size_t)(x1 - x0), cudaMemcpyDeviceToHost, st));
    LPB_CUDA(cudaMemcpyAsync(fun + l0, df + l0, sizeof(double) * (size_t)(l1 - l0), cudaMemcpyDeviceToHost, st));
    LPB_CUDA(cudaMemcpyAsync(iterations + l0, dit + l0, sizeof(int64_t) * (size_t)(l1 - l0), cudaMemcpyDeviceToHost, st));
    LPB_CUDA(cudaMemcpyAsync(status + l0, dst + l0, sizeof(int32_t) * (size_t)(l1 - l0), cudaMemcpyDeviceToHost, st));
  }
  LPB_CUDA(cudaStreamSynchronize(st));
  return LPB_OK;
}
}  // namespace

// ====================================================================== extern "C"
extern "C" {

void lpb_options_default(lpb_options* o) {
  if (o) options_default(o);
}

int lpb_options_validate(const lpb_options* o) {
  const int rc = options_validate(o);
  if (rc == LPB_ERR_UNSUPPORTED)
    set_last_error("solver_type %d: only EquationSolverType::Cholesky runs on the GPU path", o->solver_type);
  return rc;
}

const char* lpb_strerror(int code) {
  switch (code) {
    case LPB_OK: return "ok";
    case LPB_ERR_UNCONSTRAINED:
      return "The problem is unconstrained, meaning the solution is the all-zeros vector if `c` is nonnegative, or "
             "unbounded otherwise.";
    case LPB_ERR_NUMERICAL_PROBLEM:
      return "The solver encountered numerical problems it could not recover from. Likely causes are linearly "
             "dependent constraints or variables whose scale differs by multiple orders of magnitude.";
    case LPB_ERR_INVALID_PARAMETER: return "A parameter was set to an invalid value";
    case LPB_ERR_INCOMPATIBLE_INPUT_DIMENSIONS: return "The dimensions of your cost- and constraint arrays do not align.";
    case LPB_ERR_INFEASIBLE: return "The solver finished successfully, it appears that the problem is infeasible.";
    case LPB_ERR_UNBOUNDED: return "The solver finished successfully, it appears that your problem is unbounded.";
    case LPB_ERR_ITERATION_LIMIT_EXCEEDED:
      return "The solver failed to converge within the maximum number of iterations.";
    case LPB_ERR_CUDA: return "CUDA error";
    case LPB_ERR_NCCL: return "NCCL error";
    case LPB_ERR_NO_DEVICE: return "no CUDA device (there is no CPU fallback)";
    case LPB_ERR_BAD_ARGUMENT: return "bad argument";
    case LPB_ERR_UNSUPPORTED: return "unsupported on the B200 path";
    default: return "unknown lpb status";
  }
}

const char* lpb_last_error(void) { return get_last_error(); }
int lpb_abi_version(void) { return LPB_ABI_VERSION; }

int lpb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

// ---------------------------------------------------------------- problem model (host only)
int lpb_slack_dims(int64_t n_c, int64_t rows_ub, int64_t cols_ub, int64_t len_b_ub, int64_t rows_eq, int64_t cols_eq,
                   int64_t len_b_eq, int64_t* m_out, int64_t* n_out, int64_t* n_slack_out) {
  if (rows_ub < 0 || rows_eq < 0 || n_c < 0) return LPB_ERR_BAD_ARGUMENT;
  if (rows_ub + rows_eq == 0) return LPB_ERR_UNCONSTRAINED;  // linear_program.rs:134-136
  if (cols_ub != cols_eq || cols_eq != n_c || rows_ub != len_b_ub || rows_eq != len_b_eq)
    return LPB_ERR_INCOMPATIBLE_INPUT_DIMENSIONS;            // :137-143
  if (m_out) *m_out = rows_ub + rows_eq;
  if (n_out) *n_out = n_c + rows_ub;
  if (n_slack_out) *n_slack_out = rows_ub;                   // :161
  return LPB_OK;
}

int lpb_build_slack_form(const double* c, int64_t n_c, const double* A_ub, int64_t rows_ub, int64_t cols_ub,
                         int64_t ld_ub, const double* b_ub, int64_t len_b_ub, const double* A_eq, int64_t rows_eq,
                         int64_t cols_eq, int64_t ld_eq, const double* b_eq, int64_t len_b_eq, double* A_out,
                         int64_t ld_out, double* b_out, double* c_out) {
  int64_t m, n, ns;
  LPB_TRY(lpb_slack_dims(n_c, rows_ub, cols_ub, len_b_ub, rows_eq, cols_eq, len_b_eq, &m, &n, &ns));
  if (!c || !A_out || !b_out || !c_out || ld_out < n || (rows_ub && (!A_ub || !b_ub || ld_ub < n_c)) ||
      (rows_eq && (!A_eq || !b_eq || ld_eq < n_c))) {
    set_last_error("build_slack_form: null pointer or leading dimension too small");
    return LPB_ERR_BAD_ARGUMENT;
  }
  for (int64_t i = 0; i < m; ++i) {  // A = [[A_ub, I], [A_eq, 0]]   linear_program.rs:145-156
    double* row = A_out + i * ld_out;
    const double* src = i < rows_ub ? A_ub + i * ld_ub : A_eq + (i - rows_ub) * ld_eq;
    std::memcpy(row, src, sizeof(double) * (size_t)n_c);
    for (int64_t j = 0; j < ns; ++j) row[n_c + j] = 0.0;
    if (i < rows_ub) row[n_c + i] = 1.0;
    b_out[i] = i < rows_ub ? b_ub[i] : b_eq[i - rows_ub];  // :157
  }
  std::memcpy(c_out, c, sizeof(double) * (size_t)n_c);     // :159
  for (int64_t j = 0; j < ns; ++j) c_out[n_c + j] = 0.0;
  return LPB_OK;
}

int lpb_host_alloc(void** p, uint64_t bytes) {
  if (!p) return LPB_ERR_BAD_ARGUMENT;
  LPB_TRY(check_device());
  LPB_CUDA(cudaMallocHost(p, bytes ? bytes : 1));
  return LPB_OK;
}

int lpb_host_free(void* p) {
  if (p) LPB_CUDA(cudaFreeHost(p));
  return LPB_OK;
}

// ---------------------------------------------------------------- contexts
int lpb_create_bare(lpb_ctx** out, int64_t m_max, int64_t n_max, void* stream) {
  if (!out || m_max <= 0 || n_max <= 0) return LPB_ERR_BAD_ARGUMENT;
  LPB_TRY(check_device());
  lpb_ctx* c = new (std::nothrow) lpb_ctx();
  if (!c) return LPB_ERR_BAD_ARGUMENT;
  int rc = ctx_base_init(c, stream);
  if (rc == LPB_OK) rc = ctx_alloc_vectors(c, m_max, n_max, false);
  if (rc != LPB_OK) {
    ctx_free(c);
    return rc;
  }
  c->n_global = n_max;
  *out = c;
  return LPB_OK;
}

int lpb_create(lpb_ctx** out, int64_t m, int64_t n, const double* A, int64_t lda, const double* b, const double* cc,
               double c0, int mem, void* stream) {
  if (!out || m <= 0 || n <= 0) {
    set_last_error("create: m and n must be positive");
    return LPB_ERR_BAD_ARGUMENT;
  }
  LPB_TRY(check_device());
  lpb_ctx* c = new (std::nothrow) lpb_ctx();
  if (!c) return LPB_ERR_BAD_ARGUMENT;
  const bool timing = std::getenv("LPB_TIME_CREATE") != nullptr;  // stage times of the e2e path, to stderr
  auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  int rc = ctx_base_init(c, stream);
  if (rc == LPB_OK) rc = ctx_alloc_vectors(c, m, n, true);
  if (timing && rc == LPB_OK) cudaStreamSynchronize(c->lc.stream);
  const double t1 = now();
  if (rc == LPB_OK) rc = upload_problem(c, A, lda, b, cc, c0, mem);
  const double t2 = now();
  if (timing)
    std::fprintf(stderr, "[lpb_create %lldx%lld] alloc+memset %.1f ms, upload+structure %.1f ms (%.1f GB/s incl. the "
                 "structure scan)\n", (long long)m, (long long)n, t1 - t0, t2 - t1,
                 8.0 * m * n / ((t2 - t1) * 1e-3) / 1e9);
  if (rc != LPB_OK) {
    ctx_free(c);
    return rc;
  }
  c->n_global = n;
  *out = c;
  return LPB_OK;
}

int lpb_set_problem(lpb_ctx* c, const double* A, int64_t lda, const double* b, const double* cc, double c0, int mem) {
  if (!c || !c->A) return LPB_ERR_BAD_ARGUMENT;
  return upload_problem(c, A, lda, b, cc, c0, mem);
}

int lpb_destroy(lpb_ctx* c) {
  ctx_free(c);
  return LPB_OK;
}

int lpb_comm_finalize(void) {
  std::lock_guard<std::mutex> g(g_comm_mu);
  if (g_comm.refs > 0) {
    set_last_error("comm_finalize: %d live context(s) still use the process communicator", g_comm.refs);
    return LPB_ERR_BAD_ARGUMENT;
  }
  if (g_comm.comm) ncclCommDestroy(g_comm.comm);
  g_comm = ProcessComm();
  k_peer_free_process();  // the panel ring and the mappings of the other ranks' rings go with the communicator
  return LPB_OK;
}

int lpb_peer_export(lpb_ctx* c, void* handle64_out, int* state_out) {
  if (!c || !handle64_out || !state_out) return LPB_ERR_BAD_ARGUMENT;
  return k_peer_export(c->lc, c->m, static_cast<unsigned char*>(handle64_out), state_out);
}

int lpb_peer_import(lpb_ctx* c, const void* handles, int world) {
  if (!c || !handles) return LPB_ERR_BAD_ARGUMENT;
  return k_peer_import(c->lc, static_cast<const unsigned char*>(handles), world);
}

int lpb_comm_ready(int rank, int world) { return g_comm.comm && g_comm.rank == rank && g_comm.world == world ? 1 : 0; }

int lpb_nccl_unique_id(void* id128) {
  if (!id128) return LPB_ERR_BAD_ARGUMENT;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  LPB_NCCL(ncclGetUniqueId(&id));
  std::memcpy(id128, &id, sizeof(id));
  return LPB_OK;
}

int lpb_create_sharded(lpb_ctx** out, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, const double* A_local,
                       int64_t lda, const double* b, const double* c_local, double c0, int mem, int rank, int world,
                       const void* nccl_unique_id, void* stream) {
  if (!out || m <= 0 || n_local <= 0 || n_global < n_local || col0 < 0 || col0 + n_local > n_global || world < 1 ||
      rank < 0 || rank >= world) {
    set_last_error("create_sharded: inconsistent shard description");
    return LPB_ERR_BAD_ARGUMENT;
  }
  if (world > 1 && !nccl_unique_id && !(g_comm.comm && g_comm.world == world && g_comm.rank == rank)) {
    set_last_error("create_sharded: no ncclUniqueId given and no process communicator for rank %d of %d yet", rank,
                   world);
    return LPB_ERR_BAD_ARGUMENT;
  }
  LPB_TRY(check_device());
  lpb_ctx* c = new (std::nothrow) lpb_ctx();
  if (!c) return LPB_ERR_BAD_ARGUMENT;
  int rc = ctx_base_init(c, stream);
  // The communicator comes FIRST: every later rank-local failure (allocation, upload) is then agreed on across
  // the ranks (agree_status) instead of leaving the others blocked in ncclCommInitRank or in the first all-reduce.
  if (world > 1) {
    std::lock_guard<std::mutex> g(g_comm_mu);
    int rc_comm = rc;
    if (nccl_unique_id) {  // (re)build the process communicator -- every rank enters, whatever its local status
      if (g_comm.refs > 0) {
        set_last_error("create_sharded: a new ncclUniqueId was given while %d live context(s) still use the process "
                       "communicator", g_comm.refs);
        rc_comm = LPB_ERR_BAD_ARGUMENT;
      } else {
        if (g_comm.comm) ncclCommDestroy(g_comm.comm);
        g_comm = ProcessComm();
        ncclUniqueId id;
        std::memcpy(&id, nccl_unique_id, sizeof(id));
        ncclResult_t r = ncclCommInitRank(&g_comm.comm, world, id, rank);
        if (r != ncclSuccess) {
          set_last_error("ncclCommInitRank -> %s", ncclGetErrorString(r));
          g_comm = ProcessComm();
          rc_comm = LPB_ERR_NCCL;
        } else {
          g_comm.rank = rank;
          g_comm.world = world;
        }
      }
    }
    if (g_comm.comm && g_comm.world == world && g_comm.rank == rank) {
      c->comm = g_comm.comm;
      c->lc.nccl_comm = g_comm.comm;
      c->lc.rank = rank;
      c->lc.world = world;
      c->world = world;
      c->rank = rank;
      ++g_comm.refs;
    } else if (rc_comm == LPB_OK) {
      rc_comm = LPB_ERR_NCCL;
    }
    if (rc == LPB_OK) rc = rc_comm;
  }
  if (rc == LPB_OK) rc = ctx_alloc_vectors(c, m, n_local, true);
  if (rc == LPB_OK && world > 1) {  // buffers of the sharded factorisation: allocated here, not in the middle of a solve
    const int64_t cnt = tri_packed_doubles(m);
    rc = dev_alloc(c, &c->tri_buf, cnt);
    if (rc == LPB_OK && cudaMemsetAsync(c->tri_buf, 0, sizeof(double) * (size_t)cnt, c->lc.stream) != cudaSuccess)
      rc = LPB_ERR_CUDA;  // padding of the packed triangle stays finite
    if (rc == LPB_OK) rc = k_potrf_dist_reserve(c->lc, m);
  }
  if (rc == LPB_OK && A_local) rc = upload_problem(c, A_local, lda, b, c_local, c0, mem);
  rc = agree_status(c, rc);
  if (rc != LPB_OK) {
    ctx_free(c);
    return rc;
  }
  c->n_global = n_global;
  c->col0 = col0;
  c->rank = rank;
  c->world = world;
  *out = c;
  return LPB_OK;
}

// Device-side instance of the SURVEY 8(d) generator for column shards (config C5: A never exists on
// the host).  User columns [0, n0), n0 = n_global - m/2, are i.i.d. N(0,1) keyed by (seed, row, column);
// slack columns are [I; 0].  b = A0 x0 (+ s0 on the inequality rows) needs the one all-reduce;
// c = A0^T y0 + z0 is local to each shard.  Strictly primal- and dual-feasible by construction.
int lpb_create_sharded_synthetic(lpb_ctx** out, int64_t m, int64_t n_global, int64_t col0, int64_t n_local,
                                 uint64_t seed, int rank, int world, const void* nccl_unique_id, void* stream) {
  if ((m & 1) || n_global <= m / 2) {
    set_last_error("create_sharded_synthetic: needs even m and n_global > m/2");
    return LPB_ERR_BAD_ARGUMENT;
  }
  lpb_ctx* c = nullptr;
  LPB_TRY(lpb_create_sharded(&c, m, n_global, col0, n_local, nullptr, 0, nullptr, nullptr, 0.0, LPB_MEM_DEVICE, rank,
                             world, nccl_unique_id, stream));
  const int64_t mh = m / 2, n0 = n_global - mh;
  const int64_t n_user = std::max<int64_t>(0, std::min(n0, col0 + n_local) - col0);  // user columns in this shard
  int rc = LPB_OK;
  auto run = [&]() -> int {
    LPB_TRY(k_fill_normal(c->lc, c->A, m, n_user, c->lda, 0, col0, seed));
    LPB_TRY(k_slack_identity(c->lc, c->A, m, n_local, c->lda, col0, n0));
    // x0 (user columns of this shard) -> xs ; y0 -> y ; z0 -> rD ; s0 -> rP (scratch use of iterate buffers)
    LPB_TRY(k_fill(c->lc, c->xs, n_local, 0.0));
    LPB_TRY(k_fill_vec(c->lc, c->xs, n_user, col0, seed + 1, 0, 0.5, 1.5, 0));
    LPB_TRY(k_fill_vec(c->lc, c->y, m, 0, seed + 2, 2, 0.0, 0.0, mh));
    LPB_TRY(k_fill(c->lc, c->rD, n_local, 0.0));
    LPB_TRY(k_fill_vec(c->lc, c->rD, n_user, col0, seed + 3, 0, 0.5, 1.5, 0));
    LPB_TRY(k_fill_vec(c->lc, c->rP, mh, 0, seed + 4, 0, 0.5, 1.5, 0));
    // b = sum_k A_k x0_k + [s0; 0]   (slack columns contribute nothing: x0 is zero there)
    LPB_TRY(k_gemv_n(c->lc, m, n_local, c->A, c->lda, nullptr, c->xs, nullptr, c->t, nullptr, 1));
    LPB_TRY(allreduce(c, c->t, m, ncclSum));
    LPB_TRY(k_add_vec(c->lc, c->b, c->t, c->rP, m, mh));
    // c = A^T y0 + z0 on user columns, 0 on slack columns
    int nchunks = 0;
    LPB_TRY(k_gemv_t_partials(c->lc, m, n_local, c->A, c->lda, c->y, nullptr, 1, &nchunks));
    LPB_TRY(k_gemv_t_raw(c->lc, n_local, nchunks, 1, c->u, nullptr));
    LPB_TRY(k_add_vec(c->lc, c->c, c->u, c->rD, n_local, n_local));
    if (n_user < n_local) LPB_TRY(k_fill(c->lc, c->c + n_user, n_local - n_user, 0.0));
    LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
    return LPB_OK;
  };
  rc = agree_status(c, run());
  if (rc != LPB_OK) {
    ctx_free(c);
    return rc;
  }
  c->c0 = 0.0;
  c->has_problem = true;
  c->have_pq = false;
  rc = analyze_structure(c);
  if (rc != LPB_OK) {
    ctx_free(c);
    return rc;
  }
  *out = c;
  return LPB_OK;
}

// Copy this context's (shard of the) problem back to host memory: A_out m x n_local (leading
// dimension lda_out), b_out m, c_out n_local.  Any pointer may be NULL.  Parity tests use it to hand
// the device-generated synthetic shards to the CPU oracle.
int lpb_download_problem(lpb_ctx* c, double* A_out, int64_t lda_out, double* b_out, double* c_out) {
  LPB_TRY(need_problem(c));
  if (A_out && lda_out < c->n) {
    set_last_error("download_problem: lda_out < n_local");
    return LPB_ERR_BAD_ARGUMENT;
  }
  if (A_out)
    LPB_CUDA(cudaMemcpy2DAsync(A_out, sizeof(double) * lda_out, c->A, sizeof(double) * c->lda, sizeof(double) * c->n,
                               c->m, cudaMemcpyDeviceToHost, c->lc.stream));
  if (b_out) LPB_CUDA(cudaMemcpyAsync(b_out, c->b, sizeof(double) * c->m, cudaMemcpyDeviceToHost, c->lc.stream));
  if (c_out) LPB_CUDA(cudaMemcpyAsync(c_out, c->c, sizeof(double) * c->n, cudaMemcpyDeviceToHost, c->lc.stream));
  LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
  return LPB_OK;
}

// Copy a named device buffer of the context to the host (debugging / parity tests): "M" (m x ldm,
// the normal matrix or its factor), the n-vectors x z c rD dinv dx dz p u and the m-vectors b y rP dy.
// Returns the number of doubles the buffer holds; copies min(count, that) of them.
int64_t lpb_debug_read(lpb_ctx* c, const char* name, double* out, int64_t count) {
  if (!c || !name || !c->A) return -1;
  const std::string k(name);
  struct Ent { const char* n; const double* p; int64_t len; };
  const Ent tab[] = {{"M", c->M, c->m * c->ldm}, {"x", c->x, c->n}, {"z", c->z, c->n}, {"c", c->c, c->n},
                     {"rD", c->rD, c->n}, {"dinv", c->dinv, c->n}, {"dx", c->dx, c->n}, {"dz", c->dz, c->n},
                     {"p", c->p, c->n}, {"u", c->u, c->n}, {"b", c->b, c->m}, {"y", c->y, c->m},
                     {"rP", c->rP, c->m}, {"dy", c->dy, c->m}, {"t", c->t, 2 * c->m}, {"W", c->W, 2 * c->m}};
  for (const Ent& e : tab) {
    if (k != e.n) continue;
    const int64_t cnt = std::min(count, e.len);
    if (out && cnt > 0) {
      if (cudaMemcpyAsync(out, e.p, sizeof(double) * (size_t)cnt, cudaMemcpyDeviceToHost, c->lc.stream) != cudaSuccess ||
          cudaStreamSynchronize(c->lc.stream) != cudaSuccess) {
        set_last_error("debug_read: copy failed");
        return -1;
      }
    }
    return e.len;
  }
  set_last_error("debug_read: unknown buffer '%s'", name);
  return -1;
}

int64_t lpb_debug_counter(lpb_ctx* c, const char* name) {
  if (!c || !name) return -1;
  const std::string k(name);
  if (k == "potrf_verify_runs") return c->vfy_runs;
  if (k == "potrf_verify_mismatches") return c->vfy_mismatch;
  if (k == "refactorisations") return c->refactorisations;
  if (k == "refine_steps") return c->refine_steps_taken;
  return -1;
}

// ---------------------------------------------------------------- phases
int lpb_blind_start(lpb_ctx* c) {
  LPB_TRY(need_problem(c));
  CudaDev d{c};
  return d.blind_start();
}
int lpb_residuals(lpb_ctx* c, double tau, double kappa, lpb_residual_scalars* out) {
  LPB_TRY(need_problem(c));
  if (!out) return LPB_ERR_BAD_ARGUMENT;
  CudaDev d{c};
  return d.residuals(tau, kappa, out);
}
int lpb_form_and_factor(lpb_ctx* c) {
  LPB_TRY(need_problem(c));
  CudaDev d{c};
  return d.form_and_factor();
}
int lpb_direction(lpb_ctx* c, const lpb_direction_in* in, double tau, double kappa, lpb_direction_out* out) {
  LPB_TRY(need_problem(c));
  if (!in || !out) return LPB_ERR_BAD_ARGUMENT;
  CudaDev d{c};
  return d.direction(*in, tau, kappa, out);
}
int lpb_assemble_delta(lpb_ctx* c, double d_tau, double alpha_xz[2]) {
  LPB_TRY(need_problem(c));
  if (!alpha_xz) return LPB_ERR_BAD_ARGUMENT;
  CudaDev d{c};
  return d.assemble_delta(d_tau, alpha_xz);
}
int lpb_do_step(lpb_ctx* c, double alpha, int ip) {
  LPB_TRY(need_problem(c));
  CudaDev d{c};
  return d.do_step(alpha, ip);
}
int lpb_extract_x(lpb_ctx* c, double tau, double* x_out, double* fun) {
  LPB_TRY(need_problem(c));
  CudaDev d{c};
  return d.extract_x(tau, x_out, fun);
}

// ---------------------------------------------------------------- whole solve
int lpb_solve(lpb_ctx* c, const lpb_options* opts, double* x_out, double* fun, int64_t* iterations) {
  LPB_TRY(need_problem(c));
  lpb_options o;
  if (opts)
    o = *opts;
  else
    options_default(&o);
  LPB_TRY(lpb_options_validate(&o));
  profile_reset(c);
  const int64_t launches0 = c->lc.launches;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (c->profile) {
    LPB_CUDA(cudaEventCreate(&e0));
    LPB_CUDA(cudaEventCreate(&e1));
    LPB_CUDA(cudaEventRecord(e0, c->lc.stream));
  }
  CudaDev dev{c};
  int rc = solve_normal_form(dev, o, c->n_global, c->c0, &c->last);
  if (iterations) *iterations = c->last.iterations;
  if (rc == LPB_OK || rc == LPB_ERR_ITERATION_LIMIT_EXCEEDED) {
    const int rc2 = dev.extract_x(c->last.tau, x_out, fun);
    if (rc2 != LPB_OK) rc = rc2;
  }
  if (c->profile) {
    cudaEventRecord(e1, c->lc.stream);
    cudaEventSynchronize(e1);
    float f = 0.f;
    cudaEventElapsedTime(&f, e0, e1);
    profile_collect(c);
    c->prof.total_ms = f;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
  }
  c->prof.launches = c->lc.launches - launches0;
  c->prof.iterations = c->last.iterations;
  return rc;
}

int64_t lpb_trace(lpb_ctx* c, double* rows, int64_t max_rows) {
  if (!c || !rows) return 0;
  int64_t k = 0;
  for (; k < (int64_t)c->last.trace.size() && k < max_rows; ++k)
    std::memcpy(rows + k * LPB_TRACE_COLS, c->last.trace[k].v, sizeof(double) * LPB_TRACE_COLS);
  return k;
}

// ---------------------------------------------------------------- kernel entry points
int lpb_k_syrk_adat(lpb_ctx* c, int64_t m, int64_t n, const double* dA, int64_t lda, const double* d_d, double* dM,
                    int64_t ldm) {
  if (!c || !dA || !dM) return LPB_ERR_BAD_ARGUMENT;
  int rc = c->syrk_impl == 1 ? k_syrk_simple(c->lc, m, n, dA, lda, d_d, dM, ldm)
                             : k_syrk_dmma(c->lc, m, n, dA, lda, d_d, dM, ldm);
  if (rc != LPB_OK) return rc;
  LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
  return LPB_OK;
}

int lpb_k_potrf(lpb_ctx* c, int64_t m, double* dM, int64_t ldm, int32_t* info_host) {
  if (!c || !dM) return LPB_ERR_BAD_ARGUMENT;
  LPB_TRY(k_potrf(c->lc, m, dM, ldm, c->syrk_impl));
  LPB_CUDA(cudaMemcpyAsync(c->lc.info_host, c->lc.info_dev, sizeof(int), cudaMemcpyDeviceToHost, c->lc.stream));
  LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
  if (info_host) *info_host = *c->lc.info_host;
  return LPB_OK;
}

int lpb_k_potrs(lpb_ctx* c, int64_t m, const double* dL, int64_t ldm, double* dB, int64_t nrhs) {
  if (!c || !dL || !dB) return LPB_ERR_BAD_ARGUMENT;
  LPB_TRY(k_potrs(c->lc, m, dL, ldm, dB, (int)nrhs, c->syrk_impl == 0));
  return fetch_scalars(c->lc, 0);  // stream sync + the fault word of the pipelined solve
}

int lpb_k_gemv_n(lpb_ctx* c, int64_t m, int64_t n, const double* dA, int64_t lda, const double* d_w, double* d_out) {
  if (!c || !dA || !d_w || !d_out) return LPB_ERR_BAD_ARGUMENT;
  LPB_TRY(k_gemv_n(c->lc, m, n, dA, lda, nullptr, d_w, nullptr, d_out, nullptr, 1));
  LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
  return LPB_OK;
}

int lpb_k_gemv_t(lpb_ctx* c, int64_t m, int64_t n, const double* dA, int64_t lda, const double* d_v, double* d_out) {
  if (!c || !dA || !d_v || !d_out) return LPB_ERR_BAD_ARGUMENT;
  if (gemv_t_partials_doubles(m, n) > c->lc.gemv_partials_cap) {
    set_last_error("gemv_t: context work buffers were sized for a smaller problem");
    return LPB_ERR_BAD_ARGUMENT;
  }
  int nchunks = 0;
  LPB_TRY(k_gemv_t_partials(c->lc, m, n, dA, lda, d_v, nullptr, 1, &nchunks));
  LPB_TRY(k_gemv_t_raw(c->lc, n, nchunks, 1, d_out, nullptr));
  LPB_CUDA(cudaStreamSynchronize(c->lc.stream));
  return LPB_OK;
}

int lpb_solve_batched(int64_t batch, int64_t m, int64_t n, const double* A, const double* b, const double* c,
                      const lpb_options* opts, double* x_out, double* fun, int64_t* iterations, int32_t* status,
                      int mem, void* stream) {
  lpb_options o;
  LPB_TRY(batched_args("solve_batched", batch, m, n, A, b, c, opts, x_out, fun, iterations, status, &o));
  LPB_TRY(check_device());
  return run_batched(batched_launch, batch, m, n, A, b, c, o, x_out, fun, iterations, status, mem,
                     static_cast<cudaStream_t>(stream));
}

int lpb_solve_many(int64_t batch, int64_t m, int64_t n, const double* A, const double* b, const double* c,
                   const lpb_options* opts, double* x_out, double* fun, int64_t* iterations, int32_t* status, int mem,
                   void* stream) {
  lpb_options o;
  LPB_TRY(batched_args("solve_many", batch, m, n, A, b, c, opts, x_out, fun, iterations, status, &o));
  LPB_TRY(solve_many_check_shape(m, n));  // shape limits first: they hold or fail without a device
  LPB_TRY(check_device());
  return run_batched(solve_many_launch, batch, m, n, A, b, c, o, x_out, fun, iterations, status, mem,
                     static_cast<cudaStream_t>(stream));
}

int lpb_solve_many_check(int64_t m, int64_t n) {
  if (m <= 0 || n <= 0) {
    set_last_error("solve_many: non-positive size (m = %lld, n = %lld)", (long long)m, (long long)n);
    return LPB_ERR_BAD_ARGUMENT;
  }
  return solve_many_check_shape(m, n);
}

int lpb_solve_many_ragged(int64_t batch, const int64_t* m, const int64_t* n, const double* A, const double* b,
                          const double* c, const lpb_options* opts, double* x_out, double* fun, int64_t* iterations,
                          int32_t* status, int mem, void* stream) {
  if (batch <= 0 || !m || !n || !A || !b || !c || !x_out || !fun || !iterations || !status) {
    set_last_error("solve_many_ragged: null pointer or non-positive size");
    return LPB_ERR_BAD_ARGUMENT;
  }
  if (batch > INT32_MAX) {  // one CTA per LP, indexed by int
    set_last_error("solve_many_ragged: at most %d LPs per call (got %lld)", INT32_MAX, (long long)batch);
    return LPB_ERR_UNSUPPORTED;
  }
  for (int64_t i = 0; i < batch; ++i) {
    if (m[i] <= 0 || n[i] <= 0) {
      set_last_error("solve_many_ragged: LP %lld has m = %lld, n = %lld", (long long)i, (long long)m[i], (long long)n[i]);
      return LPB_ERR_BAD_ARGUMENT;
    }
  }
  for (int64_t i = 0; i < batch; ++i) {  // shape limits first: they hold or fail without a device
    if (solve_many_check_shape(m[i], n[i]) != LPB_OK) {
      const std::string why = get_last_error();
      set_last_error("solve_many_ragged: LP %lld: %s", (long long)i, why.c_str());
      return LPB_ERR_UNSUPPORTED;
    }
  }
  lpb_options o;
  if (opts)
    o = *opts;
  else
    options_default(&o);
  LPB_TRY(lpb_options_validate(&o));
  LPB_TRY(check_device());
  return run_ragged(batch, m, n, A, b, c, o, x_out, fun, iterations, status, mem, static_cast<cudaStream_t>(stream));
}

int lpb_release_workspaces(void) {
  if (g_batched_ws) cudaFree(g_batched_ws);
  g_batched_ws = nullptr;
  g_batched_ws_cap = 0;
  if (g_ragged_host) cudaFreeHost(g_ragged_host);
  g_ragged_host = nullptr;
  g_ragged_host_cap = 0;
  if (g_batched_copy_stream) cudaStreamDestroy(g_batched_copy_stream);
  g_batched_copy_stream = nullptr;
  for (int q = 0; q < 4; ++q) {
    if (g_batched_ev[q]) cudaEventDestroy(g_batched_ev[q]);
    g_batched_ev[q] = nullptr;
  }
  return LPB_OK;
}

// ---------------------------------------------------------------- measurement
int lpb_get_profile(lpb_ctx* c, lpb_profile* out) {
  if (!c || !out) return LPB_ERR_BAD_ARGUMENT;
  *out = c->prof;
  return LPB_OK;
}

int64_t lpb_launch_count(lpb_ctx* c) { return c ? c->lc.launches : 0; }

int lpb_measure_dmma_peak(lpb_ctx* c, double seconds, double* tflops_out) {
  if (!c || !tflops_out) return LPB_ERR_BAD_ARGUMENT;
  return k_dmma_peak(c->lc, seconds, tflops_out);
}

int lpb_set_option(lpb_ctx* c, const char* key, int64_t value) {
  if (!c || !key) return LPB_ERR_BAD_ARGUMENT;
  const std::string k(key);
  if (k == "syrk_impl") {
    if (value != 0 && value != 1) return LPB_ERR_BAD_ARGUMENT;
    c->syrk_impl = (int)value;
    return LPB_OK;
  }
  if (k == "solve_impl") {
    if (value < 0 || value > 3) return LPB_ERR_BAD_ARGUMENT;
    c->lc.solve_impl = (int)value;
    return LPB_OK;
  }
  if (k == "trsm_impl" || k == "update_impl") {
    if (value < 0 || value > 6) return LPB_ERR_BAD_ARGUMENT;
    (k == "trsm_impl" ? c->lc.trsm_impl : c->lc.update_impl) = (int)value;
    return LPB_OK;
  }
  if (k == "syrk_tail_split") {  // K1: 0 = every work item is a whole tile (a short last wave then costs a full tile-time)
    c->lc.syrk_tail_split = value != 0;
    return LPB_OK;
  }
  if (k == "syrk_chain") {  // 1: K1 without blocked accumulation (the round-1 summation order)
    c->lc.syrk_chain = value != 0;
    return LPB_OK;
  }
  if (k == "peer_panels") {  // 0: ncclBroadcast for the first rows of every panel; 1: peer memory (only if mapped);
                             // -1: every rank agreed to give the ring up (a failed export / import somewhere)
    if (value > 0 && !c->lc.peer_mapped) return LPB_ERR_BAD_ARGUMENT;
    if (value < 0)
      k_peer_abandon(c->lc);
    else
      c->lc.peer_ready = value != 0;
    return LPB_OK;
  }
  if (k == "syrk_flush_blocks") {  // K1: K-blocks between two flushes of the accumulators into C (power of two >= 32)
    if (value < 32 || value > (1 << 20) || (value & (value - 1))) return LPB_ERR_BAD_ARGUMENT;
    c->lc.syrk_flush_blocks = (int)value;
    return LPB_OK;
  }
  if (k == "potf2_impl") {  // 1: textbook panel factorisation without inverses (forces the substitution TRSM / solves)
    if (value < 0 || value > 1) return LPB_ERR_BAD_ARGUMENT;
    c->lc.potf2_impl = (int)value;
    if (value == 1) c->lc.trsm_impl = 1;
    return LPB_OK;
  }
  if (k == "solve_grid_cap") {
    if (value < 0) return LPB_ERR_BAD_ARGUMENT;
    c->lc.solve_grid_cap = (int)value;
    return LPB_OK;
  }
  if (k == "refine") {
    if (value < 0 || value > 4) return LPB_ERR_BAD_ARGUMENT;
    c->refine = (int)value;
    return LPB_OK;
  }
  if (k == "refine_max") {
    if (value < 0 || value > 8) return LPB_ERR_BAD_ARGUMENT;
    c->refine_max = (int)value;
    return LPB_OK;
  }
  if (k == "regularize") {  // 0 (default, the reference's behaviour): a failed factorisation is NumericalProblem
    c->regularize = value != 0;
    return LPB_OK;
  }
  if (k == "structure") {  // 0: contract over every column of A (no slack-column shortcut)
    c->use_structure = value != 0;
    return c->has_problem ? analyze_structure(c) : LPB_OK;
  }
  if (k == "potrf_lookahead") {  // 0: strictly sequential panels (single-GPU factorisation)
    c->lc.potrf_lookahead = value != 0;
    return LPB_OK;
  }
  if (k == "packed_allreduce") {
    c->packed_allreduce = value != 0;
    return LPB_OK;
  }
  if (k == "potrf_dist") {  // sharded contexts: 0 = replicated factorisation on every rank, 1 = one broadcast per
    if (value < 0 || value > 2) return LPB_ERR_BAD_ARGUMENT;  // panel, 2 = two broadcasts + side-stream potf2 (default)
    c->lc.potrf_dist = (int)value;
    return LPB_OK;
  }
  if (k == "potrf_verify") {
    c->potrf_verify = (int)value;
    return LPB_OK;
  }
  if (k == "sync_each_launch") {
    c->lc.sync_each_launch = (int)value;
    return LPB_OK;
  }
  if (k == "check_replicas") {
    c->check_replicas = value != 0;
    return LPB_OK;
  }
  if (k == "profile") {
    c->profile = value != 0;
    return LPB_OK;
  }
  set_last_error("unknown option '%s'", key);
  return LPB_ERR_BAD_ARGUMENT;
}

}  // extern "C"
