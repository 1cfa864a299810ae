// kernels.hpp -- host-side launchers of the sm_100a kernels (internal C++ interface).
#pragma once
#include "common.cuh"

namespace lpb {

// ---------------------------------------------------------------- reductions (vec_kernels.cu)
struct RedSpec {
  int nvals = 0;
  int nblocks[kMaxRedVals] = {0};
  int op[kMaxRedVals] = {0};
};
// Fold block partials (lc.red_partials) into lc.red_out[0..nvals).
int reduce_finalize(LaunchCtx& lc, const RedSpec& spec);
// D2H of lc.red_out[0..nvals) into lc.red_host + stream sync.
int fetch_scalars(LaunchCtx& lc, int nvals);

// ---------------------------------------------------------------- K5 vector kernels (vec_kernels.cu)
int k_fill(LaunchCtx& lc, double* p, int64_t n, double v);
int k_copy(LaunchCtx& lc, double* dst, const double* src, int64_t n);
int k_dinv(LaunchCtx& lc, int64_t n, const double* x, const double* z, double* dinv);

// rhat.rs:32 / :54-55 / :64 and the r1 = d_hat - xs/x of newton_equations.rs:188.
//   mode 0 predictor: xs = (x*-1)*z + gm
//   mode 1 corrector, ip: xs = (x*-1)*z - (dx*dz)*a2 + s
//   mode 2 corrector:     xs = (x*-1)*z + gm - dx*dz
int k_rhat(LaunchCtx& lc, int64_t n, int mode, double eta, double gm, double a2, double s, const double* x,
           const double* z, const double* rD, const double* dx, const double* dz, double* xs, double* r1);

// delta.rs:33,37 + ratio test feasible_point.rs:61-62; block partial mins -> red_partials rows
// (val_base, val_base+1).  Returns number of blocks used in *nblocks.
int k_assemble_delta_n(LaunchCtx& lc, int64_t n, double d_tau, const double* u, const double* p, const double* xs,
                       const double* x, const double* z, double* dx, double* dz, int val_base, int* nblocks);
// d_y = v + q d_tau (delta.rs:34)
int k_assemble_delta_m(LaunchCtx& lc, int64_t m, double d_tau, const double* v, const double* q, double* dy);
// feasible_point.rs:77-95
int k_step(LaunchCtx& lc, int64_t n, double alpha, int clamp, double* x, const double* dx);
// x_out = x / tau ; partial c.x_out -> red row val
int k_extract_x(LaunchCtx& lc, int64_t n, double tau, const double* x, const double* c, double* xo, int val,
                int* nblocks);

// m-side epilogues of the A.w sweeps
// rP = b*tau - t ; partials: sum rP^2 -> val_base, b.y -> val_base+1
int k_resid_p(LaunchCtx& lc, int64_t m, double tau, const double* b, const double* t, const double* y, double* rP,
              int val_base, int* nblocks);
// rhs0 = rP*eta + t0 ; (with_pq) rhs1 = b + t1          (newton_equations.rs:220)
int k_sym_fwd_rhs(LaunchCtx& lc, int64_t m, double eta, const double* rP, const double* b, const double* t0,
                  const double* t1, double* rhs0, double* rhs1, int with_pq);
// refinement residuals rho0 = rP*eta - A u ; (with_pq) rho1 = b - A p ;  and y += x
int k_refine_rhs(LaunchCtx& lc, int64_t m, double eta, const double* rP, const double* b, const double* au,
                 const double* ap, double* rho0, double* rho1, int with_pq);
int k_add_inplace(LaunchCtx& lc, int64_t count, const double* x, double* y);
// partials: b.v -> val_base ; (with_pq) b.q -> val_base+1, #NaN(q) -> val_base+2
int k_dots_m(LaunchCtx& lc, int64_t m, const double* b, const double* v, const double* q, int with_pq, int val_base,
             int* nblocks);

// ---------------------------------------------------------------- K4 sweeps over A (vec_kernels.cu)
// t_k = A (dinv? dinv∘w_k : w_k), k < nrhs (1 or 2).  Raw products (no epilogue).
int k_gemv_n(LaunchCtx& lc, int64_t m, int64_t n, const double* A, int64_t lda, const double* dinv, const double* w0,
             const double* w1, double* t0, double* t1, int nrhs);
// Row-chunk partials of A^T v_k into lc.gemv_partials; returns chunk count.
int k_gemv_t_partials(LaunchCtx& lc, int64_t m, int64_t n, const double* A, int64_t lda, const double* v0,
                      const double* v1, int nrhs, int* nchunks);
// Trailing singleton / zero columns of A (lpb_ctx::n_dense): the partials cover columns [0, nd) only (pitch
// round_up(nd, 2)); for j >= nd, (A^T v_k)[j] = col_val[j] * v_k[col_row[j]] (0 if col_row[j] < 0).
struct TailCols {
  int64_t nd;
  const int* col_row;
  const double* col_val;
  const double* v0;
  const double* v1;
};
// n-side epilogues consuming the partials (tail == nullptr: every column comes from the partials):
//  raw: out = sum_chunks
int k_gemv_t_raw(LaunchCtx& lc, int64_t n, int nchunks, int nrhs, double* out0, double* out1);
//  residual: rD = c*tau - s - z ; partials sum rD^2 -> val_base, c.x -> +1, x.z -> +2
int k_resid_d(LaunchCtx& lc, int64_t n, int nchunks, double tau, const double* c, const double* z, const double* x,
              double* rD, int val_base, int* nblocks, const TailCols* tail = nullptr);
//  sym_solve back (newton_equations.rs:223): u = dinv*(s0 - r1) ; (with_pq) p = dinv*(s1 - c)
//  partials c.u -> val_base ; (with_pq) c.p -> +1, #NaN(p) -> +2
int k_sym_back(LaunchCtx& lc, int64_t n, int nchunks, int with_pq, const double* dinv, const double* r1,
               const double* c, double* u, double* p, int val_base, int* nblocks, const TailCols* tail = nullptr);

// ---------------------------------------------------------------- K1 / K2 trailing update (dmma_gemm.cu)
// C(lower tiles) = A diag(d) A^T over k in [0, n)           (accumulate == 0, d may be null)
// C(lower tiles) -= P P^T with P = Mat[row0.., k0..k0+kb)    (accumulate == 1)
int k_syrk_dmma(LaunchCtx& lc, int64_t m, int64_t n, const double* A, int64_t lda, const double* d, double* Cmat,
                int64_t ldc);
int k_trailing_update_dmma(LaunchCtx& lc, int64_t m, double* Mat, int64_t ldm, int64_t k0, int64_t kb);
// C -= P P^T restricted to a tile list (look-ahead column / the block columns one rank owns): see dmma_gemm.cu
// single_col: 0 = a triangle / the owned columns, 1 = the whole block column tile0, 2 = only its diagonal tile,
// 3 = the column without its diagonal tile.  packed != null: the panel is read from a packed buffer of
// `packed_rows` rows of 128 doubles (k_potrf_dist2) instead of from Mat.  Launches on lc.side_stream when
// lc.launch_on_side is set.
int k_trailing_update_part(LaunchCtx& lc, int64_t m, double* Mat, int64_t ldm, int64_t k0, int64_t kb, int tile0,
                           int single_col, int own_mod, int own_rem, const double* packed = nullptr,
                           int64_t packed_rows = 0);
// panel TRSM as a DMMA GEMM with the inverted 128 x 128 diagonal block (dense, ld 128)
int k_trsm_dmma(LaunchCtx& lc, int64_t m, double* Mat, int64_t ldm, int64_t k0, const double* Linv);
// DMMA issue peak: register-only loop of independent DMMAs on every SM for ~seconds; TFLOP/s out
int k_dmma_peak(LaunchCtx& lc, double seconds, double* tflops);
// plain DFMA reference kernels (tests / bisecting only)
int k_syrk_simple(LaunchCtx& lc, int64_t m, int64_t n, const double* A, int64_t lda, const double* d, double* Cmat,
                  int64_t ldc);
int k_trailing_update_simple(LaunchCtx& lc, int64_t m, double* Mat, int64_t ldm, int64_t k0, int64_t kb);

// ---------------------------------------------------------------- K2 / K3 (cholesky.cu)
// In-place blocked right-looking lower Cholesky; info (device int) = 0 or first bad pivot + 1.
int k_potrf(LaunchCtx& lc, int64_t m, double* Mat, int64_t ldm, int syrk_impl);
// Allocate the panel buffers of the distributed factorisation for order m up front (column-sharded contexts).
int k_potrf_dist_reserve(LaunchCtx& lc, int64_t m);
// Peer-memory panel hand-off of the distributed factorisation: allocate this rank's ring and export its IPC handle
// (64 bytes); map the other ranks' rings (handles = world x 64 bytes, in rank order); unmap / free.
int k_peer_export(LaunchCtx& lc, int64_t m, unsigned char* handle_out, int* state_out);
int k_peer_import(LaunchCtx& lc, const unsigned char* handles, int world);
void k_peer_release(LaunchCtx& lc);       // detach this context (the ring stays with the process)
void k_peer_abandon(LaunchCtx& lc);       // every rank agreed to give the ring up
void k_peer_free_process();               // free the process ring if no context holds it
// Solve L L^T X = B in place; B column-major m x nrhs.  use_linv: use the inverted diagonal blocks the
// last k_potrf on this context left behind (L must be that factor); otherwise plain substitution.
int k_potrs(LaunchCtx& lc, int64_t m, const double* L, int64_t ldm, double* B, int nrhs, bool use_linv);

// ---------------------------------------------------------------- synthetic shard fill (vec_kernels.cu)
int k_fill_normal(LaunchCtx& lc, double* A, int64_t rows, int64_t cols, int64_t lda, int64_t row0, int64_t col0,
                  uint64_t seed);
int k_fill_vec(LaunchCtx& lc, double* v, int64_t count, int64_t idx0, uint64_t seed, int kind, double lo, double hi,
               int64_t neg_below);
int k_slack_identity(LaunchCtx& lc, double* A, int64_t rows, int64_t cols, int64_t lda, int64_t col0, int64_t n0);
int k_add_vec(LaunchCtx& lc, double* out, const double* a, const double* b, int64_t count, int64_t count_b);
// per-column structure of A: nnz count, last non-zero row (-1 if none), value (valid iff nnz == 1)
int k_col_structure(LaunchCtx& lc, const double* A, int64_t m, int64_t n, int64_t lda, int* nnz, int* row, double* val);
// M[r][r] += val[r]^2 * dinv[col[r]] where col[r] >= 0 (singleton columns folded into the diagonal)
int k_diag_add(LaunchCtx& lc, int64_t m, double* M, int64_t ldm, const int* col, const double* val, const double* dinv);
// M[r][r] *= (1 + delta) (+ delta if the entry is not positive): the diagonal shift of the regularised retry
int k_diag_shift(LaunchCtx& lc, int64_t m, double* M, int64_t ldm, double delta);
// t_k[r] += val[r] * (dinv ? dinv[j] : 1) * w_k[j], j = col[r] >= 0: the singleton columns' share of A (dinv * w_k)
int k_slack_add(LaunchCtx& lc, int64_t m, const int* col, const double* val, const double* dinv, const double* w0,
                const double* w1, double* t0, double* t1, int nrhs);
// lower triangle of M <-> packed buffer of tri_packed_doubles(m) doubles (block row i: 128 x 128 (i + 1), contiguous)
int64_t tri_packed_doubles(int64_t m);
int k_tri_pack(LaunchCtx& lc, double* M, int64_t ldm, int64_t m, double* buf, bool pack);
// order-independent bit checksum of a matrix block (replica-agreement checks of the sharded path)
int k_diff(LaunchCtx& lc, const double* a, const double* b, int64_t rows, int64_t cols, int64_t ld, int lower_only,
           unsigned long long* out_dev3);
int k_checksum(LaunchCtx& lc, const double* v, int64_t rows, int64_t cols, int64_t ld, int lower_only,
               unsigned long long* out_dev);

// ---------------------------------------------------------------- batched mode, ragged lists (batched.cu)
// One LP of a list of LPs of different shapes (lpb_solve_many_ragged): its dims, the number ns of trailing columns
// that are the implicit identity block (0 until the structure scan has run), and where its A (m x n, row-major), b
// and c start in the packed arrays.  x_out is packed like c.
struct LpDesc {
  int m, n, ns, pad;
  int64_t a_off, b_off, c_off;
};

}  // namespace lpb
