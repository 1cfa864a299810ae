// batched.cu -- K6 / K8: many small independent LPs, one CTA per problem, the whole
// solve_normal_form loop (interior_point/mod.rs:199-240) on the device.
//
// K6 (m <= 64) keeps A (m x n), M / L (m x m) and every iterate vector in shared memory; K8 (m <= 128) keeps A in
// global memory and reads it through L2 (batched_streamed_kernel).  Both run the
// SAME driver template as the single-problem path (ipm_driver.hpp: solve_normal_form_rec), here
// instantiated on `SmemDev`, whose phase calls are block-cooperative device functions.  All threads
// of the CTA execute the scalar logic redundantly on block-broadcast reduction results, so control
// flow is uniform and the statuses / iteration counts follow the reference exactly like the
// large-problem path does.  Problems are independent: sharding a batch over GPUs needs no collective.
#include "ipm_driver.hpp"
#include "kernels.hpp"
#include "panel_factor.cuh"

#include <algorithm>
#include <type_traits>
#include <vector>

namespace lpb {
namespace {

constexpr int kBT = 256;       // threads per CTA
constexpr int kMaxM = 64;      // register-tiled SYRK covers 64 x 64
constexpr int kSB = 16;        // sub-block of the in-CTA blocked Cholesky
constexpr int kXP = kSB + 1;   // pitch of the 16 x 16 inverted diagonal sub-blocks
constexpr int kBT8 = 512;      // K8 (batched_streamed_kernel): 16 warps of 8 rows each for up to kMaxM8 rows
constexpr int kMaxM8 = 128;

__device__ __forceinline__ double bw_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double bw_min(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block all-reduce of NV values over NW warps; every thread returns with the folded results (fixed order).
template <int NW, int NV>
__device__ __forceinline__ void block_allreduce(double (&v)[NV], const bool is_min, double* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const double r = is_min ? bw_min(v[k]) : bw_sum(v[k]);
    if (lane == 0) red[k * NW + warp] = r;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    double r = red[k * NW];
#pragma unroll
    for (int w = 1; w < NW; ++w) r = is_min ? fmin(r, red[k * NW + w]) : r + red[k * NW + w];
    v[k] = r;
  }
  __syncthreads();
}

// The device side of the driver for one LP per CTA: MAXM rows at most, NT threads, A in shared memory (K6) or read
// through L2 from global memory (A_GLOBAL, K8).  Everything else -- M / L, the inverted diagonal sub-blocks, every
// vector -- lives in shared memory in both.
template <int MAXM, int NT, bool A_GLOBAL>
struct SmemDev {
  static constexpr int kMaxM = MAXM;
  static constexpr int kBT = NT;
  static constexpr int kBWarps = NT / 32;
  static constexpr bool kAGlobal = A_GLOBAL;
  static_assert(kMaxM / kBWarps == 8, "rows_dot's transposing butterfly folds 8 rows per warp");
  int m, n, lda, ldm;
  int nd, ns;  // A holds the nd = n - ns leading columns; the ns trailing ones are the implicit identity block e_0 .. e_{ns-1}
  int mp, nsb;           // m rounded up to a multiple of 16 (rows >= m of M are identity padding), mp / 16
  double *Xinv, *cbuf;   // nsb x 16 x kXP inverted diagonal sub-blocks of L; scratch of factor_sub16 (panel_factor.cuh)
  int* flag;             // bad-pivot flag of the factorisation (shared)
  const double* A;       // K6: shared, pitch batched_lda(nd); K8: this LP's rows in global memory, pitch n
  double *M, *b, *c, *x, *y, *z, *rP, *rD, *dinv, *xs, *r1, *p, *q, *u, *v, *dx, *dy, *dz, *t0, *t1, *sx, *red;
  int have_pq, nan_pq;
  double cp, bq;

  // A is read-only for the whole solve: from global memory through the non-coherent (read-only) path
  __device__ __forceinline__ static double load_a(const double* p) {
    if constexpr (A_GLOBAL)
      return __ldg(p);
    else
      return *p;
  }

  // t_k[i] = sum_j A[i][j] * (w_k[j] * (scale ? dinv[j] : 1)).  A warp owns the rows warp, warp + 8, ... (8 of them at
  // m = 64) and sums them TOGETHER: 8 accumulators per lane over its columns, then a transposing butterfly -- at offset
  // 16 / 8 / 4 each lane keeps half of its rows and adds the partner's partial sums of those, after which lane l holds
  // row (l >> 2) summed over the lanes with its bits 4..2, and two more exchanges finish it: 9 shuffled doubles per
  // warp and right-hand side instead of 8 rows x 5 (one full warp reduction per row was a chain of 40 dependent
  // shuffles; the three sweeps of an iteration were ~20 % of the kernel's samples, profiles/ncu_batched_C4_r02.txt).
  template <int NRHS, bool SCALE>
  __device__ __forceinline__ void rows_dot(const double* w0, const double* w1, double* o0, double* o1) const {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned full = 0xffffffffu;
    constexpr int R = kMaxM / kBWarps;  // 8 rows per warp
    double s0[R], s1[R];
    std::conditional_t<A_GLOBAL, int, const double*> ar[R];  // K8: 32-bit row offsets (pointers spill there)
#pragma unroll
    for (int r = 0; r < R; ++r) {
      s0[r] = s1[r] = 0.0;
      const int row = warp + kBWarps * r;
      if constexpr (A_GLOBAL)
        ar[r] = (row < m ? row : 0) * lda;
      else
        ar[r] = A + (row < m ? row : 0) * lda;  // rows >= m: a valid row, result dropped
    }
    for (int j = lane; j < nd; j += 32) {
      const double d = SCALE ? dinv[j] : 1.0;
      const double x0 = SCALE ? d * w0[j] : w0[j];
      const double x1 = NRHS == 2 ? (SCALE ? d * w1[j] : w1[j]) : 0.0;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        double a;
        if constexpr (A_GLOBAL)
          a = __ldg(A + j + ar[r]);
        else
          a = ar[r][j];
        s0[r] += a * x0;
        if (NRHS == 2) s1[r] += a * x1;
      }
    }
    auto fold = [&](double (&s)[R]) {
#pragma unroll
      for (int half = R / 2, off = 16; half >= 1; half >>= 1, off >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int r = 0; r < half; ++r) {
          const double send = up ? s[r] : s[r + half];
          const double keep = up ? s[r + half] : s[r];
          s[r] = keep + __shfl_xor_sync(full, send, off);
        }
      }
      s[0] += __shfl_xor_sync(full, s[0], 2);
      s[0] += __shfl_xor_sync(full, s[0], 1);
    };
    fold(s0);
    if (NRHS == 2) fold(s1);
    const int row = warp + kBWarps * (lane >> 2);
    if ((lane & 3) == 0 && row < m) {
      if (row < ns) {  // the implicit slack column nd + row is e_row
        const int j = nd + row;
        const double d = SCALE ? dinv[j] : 1.0;
        s0[0] += SCALE ? d * w0[j] : w0[j];
        if (NRHS == 2) s1[0] += SCALE ? d * w1[j] : w1[j];
      }
      o0[row] = s0[0];
      if (NRHS == 2) o1[row] = s1[0];
    }
  }

  // s_k[j] = sum_i A[i][j] v_k[i]; thread per column, four interleaved partial sums (one chain of m dependent FMAs at
  // ~20 cycles each was the cost of this pass, not its loads)
  template <int NRHS>
  __device__ __forceinline__ void col_dot(int j, const double* v0, const double* v1, double* s0, double* s1) const {
    if (j >= nd) {  // implicit slack column e_{j - nd}
      *s0 = v0[j - nd];
      if (NRHS == 2) *s1 = v1[j - nd];
      return;
    }
    double a0[4] = {0.0, 0.0, 0.0, 0.0}, a1[4] = {0.0, 0.0, 0.0, 0.0};
    const double* col = A + j;
    int i = 0;
    for (; i + 3 < m; i += 4) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const double a = load_a(col + (i + e) * lda);
        a0[e] += a * v0[i + e];
        if (NRHS == 2) a1[e] += a * v1[i + e];
      }
    }
    for (; i < m; ++i) {
      const double a = load_a(col + i * lda);
      a0[0] += a * v0[i];
      if (NRHS == 2) a1[0] += a * v1[i];
    }
    *s0 = (a0[0] + a0[1]) + (a0[2] + a0[3]);
    if (NRHS == 2) *s1 = (a1[0] + a1[1]) + (a1[2] + a1[3]);
  }

  __device__ int blind_start() {  // feasible_point.rs:24-39
    for (int j = threadIdx.x; j < n; j += kBT) {
      x[j] = 1.0;
      z[j] = 1.0;
    }
    for (int i = threadIdx.x; i < m; i += kBT) y[i] = 0.0;
    have_pq = 0;
    __syncthreads();
    return LPB_OK;
  }

  __device__ int residuals(double tau, double kappa, lpb_residual_scalars* o) {
    (void)kappa;
    rows_dot<1, false>(x, nullptr, t0, nullptr);
    double r[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int j = threadIdx.x; j < n; j += kBT) {
      double s, unused;
      col_dot<1>(j, y, nullptr, &s, &unused);
      const double cj = c[j], zj = z[j], xj = x[j];
      const double rd = cj * tau - s - zj;  // feasible_point.rs:123
      rD[j] = rd;
      r[0] += rd * rd;
      r[1] += cj * xj;
      r[2] += xj * zj;
    }
    __syncthreads();  // t0 complete
    for (int i = threadIdx.x; i < m; i += kBT) {
      const double bi = b[i];
      const double rp = bi * tau - t0[i];  // feasible_point.rs:122
      rP[i] = rp;
      r[3] += rp * rp;
      r[4] += bi * y[i];
    }
    block_allreduce<kBWarps>(r, false, red);
    o->nrm_rd = sqrt(r[0]);
    o->cx = r[1];
    o->xz = r[2];
    o->nrm_rp = sqrt(r[3]);
    o->by = r[4];
    return LPB_OK;
  }

  __device__ int form_and_factor() {  // newton_equations.rs:48-64
    for (int j = threadIdx.x; j < n; j += kBT) dinv[j] = x[j] / z[j];
    __syncthreads();
    {  // lower(M) = A diag(dinv) A^T on the FP64 tensor path (mma.m8n8k4.f64), 8 x 8 tiles of the lower triangle dealt
       // round-robin to the warps.  The DFMA version it replaces (4 x 4 register tile per thread, the full square)
       // was bound by shared-memory bandwidth: 8 loads per 16 FMAs and thread, 22 % of the kernel's samples
       // (profiles/ncu_batched_C4_r02.txt); a fragment load feeds 8 x as many FMAs, and the upper triangle -- never
       // read -- is no longer formed.  A warp keeps up to kTilesPerWarp accumulator pairs in flight so that the
       // DMMAs of one K-step are independent.  The pitch of A (batched_lda: = 4 mod 16) makes the fragment loads --
       // lane (g, t) reads A[row0 + g][k0 + t] -- bank-conflict free.  Rows >= m of the last tile row read whatever
       // follows A in shared memory (possibly NaN patterns): they only reach entries that are not stored.
      const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
      const int g = lane >> 2, t = lane & 3;
      const int nt = (m + 7) >> 3, ntiles = nt * (nt + 1) / 2;
      constexpr int kTilesPerWarp = (kMaxM / 8) * (kMaxM / 8 + 1) / 2 / kBWarps + 1;  // K6: 36 / 8 -> 5, K8: 136 / 16 -> 9
      // K6: fragment pointers into shared memory; K8: 32-bit offsets of the tile rows from A (64-bit pointers spill there)
      using Frag = std::conditional_t<A_GLOBAL, int, const double*>;
      Frag ap[kTilesPerWarp], bp[kTilesPerWarp];
      int trow[kTilesPerWarp], tcol[kTilesPerWarp];
      double c0[kTilesPerWarp], c1[kTilesPerWarp];
#pragma unroll
      for (int q = 0; q < kTilesPerWarp; ++q) {
        int tile = warp + q * kBWarps;
        const bool live = tile < ntiles;
        if (!live) tile = 0;
        int bi = 0;
        while ((bi + 1) * (bi + 2) / 2 <= tile) ++bi;
        const int bj = tile - bi * (bi + 1) / 2;
        if constexpr (A_GLOBAL) {  // rows >= m are clamped to a row of this LP: reading past it could leave the allocation
          ap[q] = min(bi * 8 + g, m - 1) * lda;
          bp[q] = min(bj * 8 + g, m - 1) * lda;
        } else {
          ap[q] = A + (bi * 8 + g) * lda + t;
          bp[q] = A + (bj * 8 + g) * lda + t;
        }
        trow[q] = live ? bi * 8 + g : m;  // m: nothing is stored
        tcol[q] = bj * 8 + 2 * t;
        c0[q] = c1[q] = 0.0;
      }
      // No per-lane select may feed the mma: ptxas if-converts `kin ? mma(a, b) : mma(0, 0)` into two DMMAs predicated
      // per LANE, each behind a predicated WARPSYNC.ALL -- a deadlock as soon as n is not a multiple of 4 (found the
      // hard way).  Instead the padding columns nd .. lda-1 of A are zero (written at load) and the index of dinv is
      // clamped, so the K tail contributes exact zeros.
      // K8 reads A where the caller put it, so its columns past nd are not zeros: there the column index is clamped
      // as well and the weight is multiplied by live = 0 (integer min / max, no predicate), which makes the K tail
      // exact zeros for finite A.
      for (int k0 = 0; k0 < nd; k0 += 4) {
        double dk;
        const double* ak;  // ap[q] / bp[q] are relative to it
        if constexpr (A_GLOBAL) {
          const int kc = min(k0 + t, nd - 1);
          dk = dinv[kc] * (double)min(max(nd - (k0 + t), 0), 1);
          ak = A + kc;
        } else {
          dk = dinv[min(k0 + t, nd - 1)];
          ak = nullptr;
        }
#pragma unroll
        for (int q = 0; q < kTilesPerWarp; ++q) {
          double a, bv;
          if constexpr (A_GLOBAL) {
            a = __ldg(ak + ap[q]);
            bv = __ldg(ak + bp[q]) * dk;
          } else {
            a = ap[q][k0];
            bv = bp[q][k0] * dk;
          }
          asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                       : "+d"(c0[q]), "+d"(c1[q])
                       : "d"(a), "d"(bv));
        }
      }
#pragma unroll
      for (int q = 0; q < kTilesPerWarp; ++q) {
        if (trow[q] < m) {
          // the implicit slack column nd + r contributes dinv[nd + r] to M[r][r] and nothing else
          if (trow[q] < ns && trow[q] == tcol[q]) c0[q] += dinv[nd + trow[q]];
          if (trow[q] < ns && trow[q] == tcol[q] + 1) c1[q] += dinv[nd + trow[q]];
          if (tcol[q] < m) M[trow[q] * ldm + tcol[q]] = c0[q];
          if (tcol[q] + 1 < m) M[trow[q] * ldm + tcol[q] + 1] = c1[q];
        }
      }
    }
    __syncthreads();
    // In-place lower Cholesky, blocked by 16 columns like potf2_inv_kernel (cholesky.cu): per block ONE warp
    // factors the 16 x 16 diagonal sub-block and inverts it in the same 16 pivot steps (lanes 0..15: rows of
    // the sub-block; lanes 16..31: forward substitutions L x = e_c for the columns of the inverse), then the
    // CTA applies the inverse to the rows below and the rank-16 update to the remaining sub-blocks: 3 CTA
    // barriers per 16 columns instead of 2 per column.  Pivot <= 0 or non-finite -> NumericalProblem
    // (newton_equations.rs:63), decided uniformly from a shared flag.
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) *flag = 0;
    for (int kb = 0; kb < nsb; ++kb) {
      const int c0 = kb * kSB;
      double* Xd = Xinv + kb * kSB * kXP;
      if (warp == 0) {
        // panel_factor.cuh: the same rolled, branch-free pivot loop as the panel kernel of K2 (hardware rsqrt seed +
        // one cubic step instead of the library rsqrt, no per-pivot test: a bad pivot poisons its lane)
        if (factor_sub16<kXP, false>(M + (c0 + (lane & 15)) * ldm + c0, Xd, cbuf, nullptr, lane) && lane == 0) *flag = 1;
      }
      __syncthreads();
      {  // rows below: P[r][c] = sum_l M[r][c0+l] X[c][l]  (4 columns per thread, the 4 threads of a row in one warp)
        const int r = c0 + kSB + (tid >> 2), q4 = tid & 3;
        const bool act = r < mp;
        double out[4] = {0.0, 0.0, 0.0, 0.0};
        if (act) {
          double row[kSB];
#pragma unroll
          for (int l = 0; l < kSB; ++l) row[l] = M[r * ldm + c0 + l];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const double* xr = Xd + (4 * q4 + e) * kXP;
            double acc = 0.0;
#pragma unroll
            for (int l = 0; l < kSB; ++l) acc += row[l] * xr[l];
            out[e] = acc;
          }
        }
        __syncwarp();
        if (act) {
#pragma unroll
          for (int e = 0; e < 4; ++e) M[r * ldm + c0 + 4 * q4 + e] = out[e];
        }
      }
      __syncthreads();
      {  // rank-16 update of the remaining 16 x 16 sub-blocks (lower triangle), one per warp per round
        const int nrem = nsb - 1 - kb;
        const int T = nrem * (nrem + 1) / 2;
        const int ii = lane & 15, jh = lane >> 4;
        for (int t = warp; t < T; t += kBWarps) {
          int bi = 0;
          while ((bi + 1) * (bi + 2) / 2 <= t) ++bi;
          const int bj = t - bi * (bi + 1) / 2;
          const int ri = (kb + 1 + bi) * kSB + ii;
          const int cj = (kb + 1 + bj) * kSB + 8 * jh;
          double pr[kSB];
#pragma unroll
          for (int l = 0; l < kSB; ++l) pr[l] = M[ri * ldm + c0 + l];
          double acc[8];
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) {
            const double* pj = M + (cj + jj) * ldm + c0;
            double a8 = 0.0;
#pragma unroll
            for (int l = 0; l < kSB; ++l) a8 += pr[l] * pj[l];
            acc[jj] = a8;
          }
#pragma unroll
          for (int jj = 0; jj < 8; ++jj)
            if (cj + jj <= ri) M[ri * ldm + cj + jj] -= acc[jj];
        }
      }
      __syncthreads();
    }
    have_pq = 0;
    if (*flag) return LPB_ERR_NUMERICAL_PROBLEM;  // uniform: every thread reads the same shared word
    return LPB_OK;
  }

  // solve L L^T w = rhs in place for NRHS vectors (r0, r1v; mp entries each): blocked substitution over the
  // 16-row blocks with the inverted diagonal sub-blocks inside them -- 2 CTA barriers per block and direction.
  // Thread t < mp owns row t of the first right-hand side, thread mp + t row t of the second.
  template <int NRHS>
  __device__ __forceinline__ void chol_solve(double* r0, double* r1v) {
    const int tid = threadIdx.x;
    const int which = tid >= mp ? 1 : 0;
    const int row = tid - which * mp;
    const bool act = which < NRHS && row < mp;
    double* cv = which ? r1v : r0;
    double* wv = sx + which * kMaxM;
    if (act && row >= m) cv[row] = 0.0;  // identity padding rows carry a zero right-hand side
    __syncthreads();
    for (int s = 0; s < nsb; ++s) {      // forward: L w = c
      const int c0 = s * kSB;
      if (act && row >= c0 && row < c0 + kSB) {
        const double* xr = Xinv + (s * kSB + (row - c0)) * kXP;
        double acc = 0.0;
#pragma unroll
        for (int l = 0; l < kSB; ++l) acc += xr[l] * cv[c0 + l];  // X is zero above its diagonal
        wv[row] = acc;
      }
      __syncthreads();
      if (act && row >= c0) {
        if (row < c0 + kSB) {
          cv[row] = wv[row];
        } else {
          const double* lr = M + row * ldm + c0;
          double acc = 0.0;
#pragma unroll
          for (int l = 0; l < kSB; ++l) acc += lr[l] * wv[c0 + l];
          cv[row] -= acc;
        }
      }
      __syncthreads();
    }
    for (int s = nsb - 1; s >= 0; --s) {  // backward: L^T x = w
      const int c0 = s * kSB;
      if (act && row >= c0 && row < c0 + kSB) {
        const int i = row - c0;
        double acc = 0.0;
#pragma unroll
        for (int l = 0; l < kSB; ++l) acc += Xinv[(s * kSB + l) * kXP + i] * cv[c0 + l];  // x_i = sum_l X[l][i] c_l
        wv[row] = acc;
      }
      __syncthreads();
      if (act && row < c0 + kSB) {
        if (row >= c0) {
          cv[row] = wv[row];
        } else {
          double acc = 0.0;
#pragma unroll
          for (int l = 0; l < kSB; ++l) acc += M[(c0 + l) * ldm + row] * wv[c0 + l];
          cv[row] -= acc;
        }
      }
      __syncthreads();
    }
  }

  __device__ int direction(const lpb_direction_in& in, double tau, double kappa, lpb_direction_out* o) {
    (void)tau;
    (void)kappa;
    const int with_pq = have_pq ? 0 : 1;
    const double gm = in.gamma * in.mu;
    const double a2 = in.alpha * in.alpha;
    const double s = (1.0 - in.alpha) * in.gamma * in.mu;
    for (int j = threadIdx.x; j < n; j += kBT) {
      const double xj = x[j];
      const double mxz = (xj * -1.0) * z[j];
      double val;
      if (!in.corrector)
        val = mxz + gm;                          // rhat.rs:32
      else if (in.ip)
        val = mxz - (dx[j] * dz[j]) * a2 + s;    // rhat.rs:54-55
      else
        val = mxz + gm - (dx[j] * dz[j]);        // rhat.rs:64
      xs[j] = val;
      r1[j] = rD[j] * in.eta - val / xj;         // newton_equations.rs:188
    }
    __syncthreads();
    if (with_pq)
      rows_dot<2, true>(r1, c, t0, t1);
    else
      rows_dot<1, true>(r1, nullptr, t0, nullptr);
    __syncthreads();
    for (int i = threadIdx.x; i < m; i += kBT) {
      v[i] = rP[i] * in.eta + t0[i];             // newton_equations.rs:220
      if (with_pq) q[i] = b[i] + t1[i];
    }
    __syncthreads();
    if (with_pq)
      chol_solve<2>(v, q);
    else
      chol_solve<1>(v, nullptr);
    double r[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int j = threadIdx.x; j < n; j += kBT) {
      double s0, s1 = 0.0;
      if (with_pq)
        col_dot<2>(j, v, q, &s0, &s1);
      else
        col_dot<1>(j, v, nullptr, &s0, &s1);
      const double dj = dinv[j], cj = c[j];
      const double uj = dj * (s0 - r1[j]);       // newton_equations.rs:223
      u[j] = uj;
      r[0] += cj * uj;
      if (with_pq) {
        const double pj = dj * (s1 - cj);
        p[j] = pj;
        r[1] += cj * pj;
        r[2] += (pj != pj) ? 1.0 : 0.0;
      }
    }
    for (int i = threadIdx.x; i < m; i += kBT) {
      const double bi = b[i];
      r[3] += bi * v[i];
      if (with_pq) {
        const double qi = q[i];
        r[4] += bi * qi;
        r[5] += (qi != qi) ? 1.0 : 0.0;
      }
    }
    block_allreduce<kBWarps>(r, false, red);
    if (with_pq) {
      cp = r[1];
      bq = r[4];
      nan_pq = (r[2] > 0.0 || r[5] > 0.0) ? 1 : 0;
      have_pq = 1;
    }
    o->cu = r[0];
    o->bv = r[3];
    o->cp = cp;
    o->bq = bq;
    o->nan_pq = nan_pq;
    o->reserved = 0;
    return LPB_OK;
  }

  __device__ int assemble_delta(double d_tau, double axz[2]) {
    double r[2] = {1.0, 1.0};
    for (int j = threadIdx.x; j < n; j += kBT) {
      const double xj = x[j], zj = z[j];
      const double dxj = u[j] + p[j] * d_tau;        // delta.rs:33
      const double dzj = (xs[j] - zj * dxj) / xj;    // delta.rs:37
      dx[j] = dxj;
      dz[j] = dzj;
      if (dxj < 0.0) r[0] = fmin(r[0], xj / -dxj);   // feasible_point.rs:61
      if (dzj < 0.0) r[1] = fmin(r[1], zj / -dzj);   // :62
    }
    for (int i = threadIdx.x; i < m; i += kBT) dy[i] = v[i] + q[i] * d_tau;  // delta.rs:34
    block_allreduce<kBWarps>(r, true, red);
    axz[0] = r[0];
    axz[1] = r[1];
    return LPB_OK;
  }

  __device__ int do_step(double alpha, int ip) {  // feasible_point.rs:76-106
    for (int j = threadIdx.x; j < n; j += kBT) {
      double xv = x[j] + dx[j] * alpha, zv = z[j] + dz[j] * alpha;
      if (ip) {
        xv = fmax(xv, 1.0);
        zv = fmax(zv, 1.0);
      }
      x[j] = xv;
      z[j] = zv;
    }
    for (int i = threadIdx.x; i < m; i += kBT) y[i] = y[i] + dy[i] * alpha;
    __syncthreads();
    return LPB_OK;
  }
};

using K6Dev = SmemDev<kMaxM, kBT, false>;
using K8Dev = SmemDev<kMaxM8, kBT8, true>;

__host__ __device__ inline int batched_mp(int m) { return (m + kSB - 1) / kSB * kSB; }
// pitch of A in shared memory: = 4 (mod 16) doubles, so that the 8 x 4 DMMA fragment loads of the in-CTA SYRK (row g,
// column t of a tile: 8 (g) + 2 (t) words apart) fall into 32 different banks per half-warp
__host__ __device__ inline int batched_lda(int n) { return (n + 15) / 16 * 16 + 4; }
// everything but A (the only term of K6's footprint that K8 does not have)
template <class Dev>
__host__ __device__ inline size_t batched_vec_smem_doubles(int m, int n) {
  const size_t mp = (size_t)batched_mp(m);
  return mp * (mp + 1) + 10 * (size_t)n + 5 * (size_t)m + 2 * mp + 2 * Dev::kMaxM + 8 * Dev::kBWarps +
         (mp / kSB) * kSB * kXP + panel_factor_scratch(kXP) + 2;
}
__host__ __device__ inline size_t batched_smem_doubles(int m, int n, int ns) {
  return (size_t)m * batched_lda(n - ns) + batched_vec_smem_doubles<K6Dev>(m, n);
}

// Layout of everything behind A in the dynamic shared memory (the same for K6 and K8).
template <class Dev>
__device__ __forceinline__ void carve_smem(Dev& d, double* ptr) {
  auto take = [&](size_t cnt) {
    double* r = ptr;
    ptr += cnt;
    return r;
  };
  d.M = take((size_t)d.mp * d.ldm);
  d.c = take(d.n); d.x = take(d.n); d.z = take(d.n); d.rD = take(d.n); d.dinv = take(d.n); d.xs = take(d.n);
  d.r1 = take(d.n); d.p = take(d.n); d.dx = take(d.n); d.dz = take(d.n);
  d.u = d.r1;        // u[j] = dinv[j] * (s - r1[j]) overwrites r1[j] in place (r1 is dead afterwards)
  d.b = take(d.m); d.y = take(d.m); d.rP = take(d.m); d.q = take(d.mp); d.v = take(d.mp); d.dy = take(d.m);
  d.t0 = take(d.m);
  d.t1 = d.dy;       // t1 is consumed (q = b + t1) before d_y is written
  d.sx = take(2 * Dev::kMaxM);
  d.red = take(8 * Dev::kBWarps);
  d.Xinv = take((size_t)d.nsb * kSB * kXP);
  d.cbuf = take(panel_factor_scratch(kXP));
  d.flag = reinterpret_cast<int*>(take(2));
  d.have_pq = 0;
  d.nan_pq = 0;
  d.cp = d.bq = 0.0;
}

template <class Dev>
__device__ __forceinline__ void init_dims(Dev& d, int m, int n, int ns) {
  d.m = m;
  d.n = n;
  d.ns = ns;
  d.nd = n - ns;
  d.lda = Dev::kAGlobal ? n : batched_lda(d.nd);
  d.mp = batched_mp(m);
  d.nsb = d.mp / kSB;
  d.ldm = d.mp + 1;
}

// Loads the rest of one LP (A is in place) from gb + b_off and gc + c_off, runs the driver and writes x to
// x_out + c_off and fun / iterations / status to output slot `slot`.
template <class Dev>
__device__ __forceinline__ void solve_one(Dev& d, const double* __restrict__ gb, int64_t b_off,
                                          const double* __restrict__ gc, int64_t c_off, const lpb_options& opts,
                                          double* __restrict__ x_out, int64_t slot,
                                          double* __restrict__ fun_out, int64_t* __restrict__ it_out,
                                          int32_t* __restrict__ st_out) {
  constexpr int kT = Dev::kBT;
  const int m = d.m, n = d.n;
  for (int idx = threadIdx.x; idx < d.mp * d.mp; idx += kT) {  // identity padding of M beyond m (kept by the factorisation)
    const int r = idx / d.mp, cc = idx - r * d.mp;
    if (r >= m || cc >= m) d.M[r * d.ldm + cc] = (r == cc) ? 1.0 : 0.0;
  }
  for (int i = threadIdx.x; i < m; i += kT) d.b[i] = gb[b_off + i];
  for (int j = threadIdx.x; j < n; j += kT) {
    d.c[j] = gc[c_off + j];
    d.dx[j] = 0.0;
    d.dz[j] = 0.0;
  }
  __syncthreads();

  SolveScalars sc;
  NullRecorder rec;
  const int rc = solve_normal_form_rec(d, opts, (int64_t)n, 0.0, &sc, rec);

  double f[1] = {0.0};
  if (rc == LPB_OK || rc == LPB_ERR_ITERATION_LIMIT_EXCEEDED) {
    for (int j = threadIdx.x; j < n; j += kT) {
      const double t = d.x[j] / sc.tau;  // mod.rs:231
      x_out[c_off + j] = t;
      f[0] += d.c[j] * t;                // linear_program.rs:62
    }
  }
  block_allreduce<Dev::kBWarps>(f, false, d.red);
  if (threadIdx.x == 0) {
    fun_out[slot] = f[0];
    it_out[slot] = sc.iterations;
    st_out[slot] = rc;
  }
  __syncthreads();
}

// One LP of m x n with ns implicit slack columns on one CTA (its A at A, the rest located as for solve_one): K6
// copies the nd = n - ns stored columns of A into shared memory, K8 reads A where it is.  The body of both the uniform
// and the ragged kernels.
template <class Dev>
__device__ __forceinline__ void run_lp(double* sm, int m, int n, int ns, const double* A,
                                       const double* __restrict__ gb, int64_t b_off, const double* __restrict__ gc,
                                       int64_t c_off, const lpb_options& opts, double* __restrict__ x_out, int64_t slot,
                                       double* __restrict__ fun_out, int64_t* __restrict__ it_out,
                                       int32_t* __restrict__ st_out) {
  Dev d;
  init_dims(d, m, n, ns);
  if constexpr (Dev::kAGlobal) {
    d.A = A;
    carve_smem(d, sm);
  } else {
    double* sA = sm;
    d.A = sA;
    carve_smem(d, sm + (size_t)m * d.lda);
    for (int idx = threadIdx.x; idx < m * d.nd; idx += Dev::kBT) {
      const int i = idx / d.nd, j = idx - i * d.nd;
      sA[i * d.lda + j] = A[i * n + j];
    }
    for (int idx = threadIdx.x; idx < m * (d.lda - d.nd); idx += Dev::kBT) {  // zero padding columns: the K tail of the DMMA SYRK
      const int i = idx / (d.lda - d.nd), j = d.nd + idx - i * (d.lda - d.nd);
      sA[i * d.lda + j] = 0.0;
    }
  }
  solve_one(d, gb, b_off, gc, c_off, opts, x_out, slot, fun_out, it_out, st_out);
}

// Two CTAs per SM (128 registers, <= 113 KB of shared memory each) whenever the batch has the slack structure: one LP's
// serial sections -- the factoring warp above all, 22 % of the time with seven warps waiting -- are then covered by
// the other LP's parallel ones.  `ns` (from batched_structure_kernel, the same for every LP of the batch) is the
// number of trailing columns that are e_0 .. e_{ns-1} in EVERY problem; they are not stored.
__global__ void __launch_bounds__(kBT, 2)
batched_ipm_kernel(int64_t batch, int m, int n, int ns, const double* __restrict__ gA, const double* __restrict__ gb,
                   const double* __restrict__ gc, lpb_options opts, double* __restrict__ x_out,
                   double* __restrict__ fun_out, int64_t* __restrict__ it_out, int32_t* __restrict__ st_out) {
  extern __shared__ double sm[];
  for (int64_t lp = blockIdx.x; lp < batch; lp += gridDim.x)
    run_lp<K6Dev>(sm, m, n, ns, gA + lp * (int64_t)m * n, gb, lp * m, gc, lp * n, opts, x_out, lp, fun_out, it_out, st_out);
}

// K8: LPs of up to 128 rows.  A (m x n, 128 x 256 = 256 KB) no longer fits beside M, so it stays in global memory and
// every pass over it -- the SYRK, the row sweeps, the column sweeps -- reads it through L2 (148 resident LPs of
// 128 x 128 dense columns are ~19 MB); the shared memory holds M / L and the vectors.  One CTA of 16 warps per SM:
// rows_dot's 8 rows per warp then cover 128 rows, and chol_solve's thread-per-row layout covers both right-hand sides.
__global__ void __launch_bounds__(kBT8, 1)
batched_streamed_kernel(int64_t batch, int m, int n, int ns, const double* __restrict__ gA,
                        const double* __restrict__ gb, const double* __restrict__ gc, lpb_options opts,
                        double* __restrict__ x_out, double* __restrict__ fun_out, int64_t* __restrict__ it_out,
                        int32_t* __restrict__ st_out) {
  extern __shared__ double sm[];
  for (int64_t lp = blockIdx.x; lp < batch; lp += gridDim.x)
    run_lp<K8Dev>(sm, m, n, ns, gA + lp * (int64_t)m * n, gb, lp * m, gc, lp * n, opts, x_out, lp, fun_out, it_out, st_out);
}

// Ragged launch (lpb_solve_many_ragged): a list of LPs of different shapes, one CTA per LP.  CTA k solves LP order[k]:
// the host decides which LPs start first (the costliest), and the block scheduler hands each freed SM the next LP of
// the list.  LP lp's dims and offsets come from desc[lp] (x_out uses c's offset); every CTA runs the same arithmetic as
// the uniform kernel on a batch of that LP alone.
template <class Dev>
__device__ __forceinline__ void run_ragged(double* sm, const LpDesc* __restrict__ desc, const int* __restrict__ order,
                                           const double* __restrict__ gA, const double* __restrict__ gb,
                                           const double* __restrict__ gc, const lpb_options& opts,
                                           double* __restrict__ x_out, double* __restrict__ fun_out,
                                           int64_t* __restrict__ it_out, int32_t* __restrict__ st_out) {
  const int lp = order[blockIdx.x];
  const LpDesc e = desc[lp];
  run_lp<Dev>(sm, e.m, e.n, e.ns, gA + e.a_off, gb, e.b_off, gc, e.c_off, opts, x_out, lp, fun_out, it_out, st_out);
}

__global__ void __launch_bounds__(kBT, 2)
ragged_ipm_kernel(const LpDesc* __restrict__ desc, const int* __restrict__ order, const double* __restrict__ gA,
                  const double* __restrict__ gb, const double* __restrict__ gc, lpb_options opts,
                  double* __restrict__ x_out, double* __restrict__ fun_out, int64_t* __restrict__ it_out,
                  int32_t* __restrict__ st_out) {
  extern __shared__ double sm[];
  run_ragged<K6Dev>(sm, desc, order, gA, gb, gc, opts, x_out, fun_out, it_out, st_out);
}

__global__ void __launch_bounds__(kBT8, 1)
ragged_streamed_kernel(const LpDesc* __restrict__ desc, const int* __restrict__ order, const double* __restrict__ gA,
                       const double* __restrict__ gb, const double* __restrict__ gc, lpb_options opts,
                       double* __restrict__ x_out, double* __restrict__ fun_out, int64_t* __restrict__ it_out,
                       int32_t* __restrict__ st_out) {
  extern __shared__ double sm[];
  run_ragged<K8Dev>(sm, desc, order, gA, gb, gc, opts, x_out, fun_out, it_out, st_out);
}

// Length of the run of trailing columns of one LP (m x n, row-major at A) that are exactly e_0 .. e_{s-1} (the slack
// block ProblemBuilder::build appends, linear_program.rs:145-156): columns from the right while column n - s + r is
// the unit vector e_r for a consistent s.  One CTA; the result is in `best` for every thread on return.
__device__ __forceinline__ void slack_run(const double* __restrict__ A, int m, int n, int smax, int (&urow)[kMaxM8],
                                          int& best) {  // smax = min(m, n)
  if (threadIdx.x == 0) best = 0;
  for (int t = threadIdx.x; t < smax; t += blockDim.x) {  // adjacent threads read adjacent columns of a row: coalesced
    const int j = n - smax + t;
    int r = -1;
    for (int i = 0; i < m; ++i) {
      const double v = A[(int64_t)i * n + j];
      if (v != 0.0) r = (v == 1.0 && r == -1) ? i : -2;
    }
    urow[t] = r >= 0 ? r : -1;  // urow[t]: column n - smax + t is the unit vector e_{urow[t]} (entry exactly 1), else -1
  }
  __syncthreads();
  for (int s = 1 + threadIdx.x; s <= smax; s += blockDim.x) {  // candidate: the last s columns are e_0 .. e_{s-1}
    bool good = true;
    for (int r = 0; r < s; ++r) good = good && urow[smax - s + r] == r;
    if (good) atomicMax(&best, s);
  }
  __syncthreads();
}

// Largest ns such that in EVERY problem of the batch the last ns columns are exactly e_0 .. e_{ns-1}.  Detected from
// the data, never assumed: one CTA per problem finds its own run (slack_run), the batch takes the minimum.  A batch
// without the structure gets 0 and the kernel stores all of A.
__global__ void __launch_bounds__(256)
batched_structure_kernel(int64_t batch, int m, int n, const double* __restrict__ gA, int* __restrict__ ns_out) {
  __shared__ int urow[kMaxM8];
  __shared__ int best;
  const int smax = m < n ? m : n;
  for (int64_t lp = blockIdx.x; lp < batch; lp += gridDim.x) {
    slack_run(gA + lp * (int64_t)m * n, m, n, smax, urow, best);
    if (threadIdx.x == 0) atomicMin(ns_out, best);
    __syncthreads();
  }
}

// The ragged counterpart: every LP of [lo, lo + cnt) keeps its own run, ns_out[lp] (unclamped: the host clamps).
__global__ void __launch_bounds__(256)
ragged_structure_kernel(int64_t lo, int64_t cnt, const LpDesc* __restrict__ desc, const double* __restrict__ gA,
                        int* __restrict__ ns_out) {
  __shared__ int urow[kMaxM8];
  __shared__ int best;
  for (int64_t lp = lo + blockIdx.x; lp < lo + cnt; lp += gridDim.x) {
    const LpDesc e = desc[lp];
    slack_run(gA + e.a_off, e.m, e.n, e.m < e.n ? e.m : e.n, urow, best);
    if (threadIdx.x == 0) ns_out[lp] = best;
    __syncthreads();
  }
}

}  // namespace

namespace {
constexpr size_t kSmemCap = 227 * 1024;

// Structure scan (batched_structure_kernel): dit (int64 per problem, written by the solve afterwards) lends its first
// word for the result.
int scan_slack_structure(int64_t batch, int m, int n, const double* dA, int64_t* dit, cudaStream_t stream, int* ns_out) {
  int* ns_dev = reinterpret_cast<int*>(dit);
  int ns = m < n ? m : n;
  LPB_CUDA(cudaMemcpyAsync(ns_dev, &ns, sizeof(int), cudaMemcpyHostToDevice, stream));
  const int64_t sgrid = batch < (int64_t)kNumSMs * 8 ? batch : (int64_t)kNumSMs * 8;
  batched_structure_kernel<<<(unsigned)sgrid, 256, 0, stream>>>(batch, m, n, dA, ns_dev);
  LPB_CUDA(cudaGetLastError());
  LPB_CUDA(cudaMemcpyAsync(&ns, ns_dev, sizeof(int), cudaMemcpyDeviceToHost, stream));
  LPB_CUDA(cudaStreamSynchronize(stream));
  if (ns < 0 || ns > m || ns >= n) ns = 0;
  *ns_out = ns;
  return LPB_OK;
}

int launch_k6(int64_t batch, int m, int n, int ns, const double* dA, const double* db, const double* dc,
              const lpb_options& o, double* dx, double* dfun, int64_t* dit, int32_t* dst, cudaStream_t stream) {
  const size_t smem = batched_smem_doubles(m, n, ns) * sizeof(double);
  LPB_CUDA(cudaFuncSetAttribute(batched_ipm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t grid = batch < (int64_t)kNumSMs * 64 ? batch : (int64_t)kNumSMs * 64;
  batched_ipm_kernel<<<(unsigned)grid, kBT, smem, stream>>>(batch, m, n, ns, dA, db, dc, o, dx, dfun, dit, dst);
  LPB_CUDA(cudaGetLastError());
  return LPB_OK;
}
}  // namespace

int batched_launch(int64_t batch, int m, int n, const double* dA, const double* db, const double* dc,
                   const lpb_options& o, double* dx, double* dfun, int64_t* dit, int32_t* dst, cudaStream_t stream) {
  if (m > kMaxM) {
    set_last_error("solve_batched: needs m <= %d", kMaxM);
    return LPB_ERR_UNSUPPORTED;
  }
  int ns = 0;
  LPB_TRY(scan_slack_structure(batch, m, n, dA, dit, stream, &ns));
  const size_t smem = batched_smem_doubles(m, n, ns) * sizeof(double);
  if (smem > kSmemCap) {
    set_last_error("solve_batched: %zu bytes of shared memory > 227 KB", smem);
    return LPB_ERR_UNSUPPORTED;
  }
  return launch_k6(batch, m, n, ns, dA, db, dc, o, dx, dfun, dit, dst, stream);
}

// K8's footprint does not depend on the slack structure, and K6 fits wherever K8 does not only if K8 fits too: the
// shape alone decides whether solve_many can run it, before any device is touched.
int solve_many_check_shape(int64_t m, int64_t n) {
  if (m > kMaxM8) {
    set_last_error("solve_many: needs m <= %d (got m = %lld)", kMaxM8, (long long)m);
    return LPB_ERR_UNSUPPORTED;
  }
  // n beyond 2^20 is far past the limit; the clamp keeps the count in int
  const size_t smem = batched_vec_smem_doubles<K8Dev>((int)m, (int)(n < (1 << 20) ? n : (1 << 20))) * sizeof(double);
  if (smem > kSmemCap) {
    set_last_error("solve_many: m = %lld, n = %lld needs %zu bytes of shared memory > 227 KB (232448 bytes)",
                   (long long)m, (long long)n, smem);
    return LPB_ERR_UNSUPPORTED;
  }
  return LPB_OK;
}

// K6 where it accepts (m, n, ns) -- m <= 64 and A fits beside M -- else K8.  Which of the two is faster where both
// run has not been measured: this only picks a kernel that can run the shape.
int solve_many_launch(int64_t batch, int m, int n, const double* dA, const double* db, const double* dc,
                      const lpb_options& o, double* dx, double* dfun, int64_t* dit, int32_t* dst, cudaStream_t stream) {
  LPB_TRY(solve_many_check_shape(m, n));
  int ns = 0;
  LPB_TRY(scan_slack_structure(batch, m, n, dA, dit, stream, &ns));
  if (m <= kMaxM && batched_smem_doubles(m, n, ns) * sizeof(double) <= kSmemCap)
    return launch_k6(batch, m, n, ns, dA, db, dc, o, dx, dfun, dit, dst, stream);
  const size_t smem = batched_vec_smem_doubles<K8Dev>(m, n) * sizeof(double);
  LPB_CUDA(cudaFuncSetAttribute(batched_streamed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t grid = batch < (int64_t)kNumSMs * 64 ? batch : (int64_t)kNumSMs * 64;
  batched_streamed_kernel<<<(unsigned)grid, kBT8, smem, stream>>>(batch, m, n, ns, dA, db, dc, o, dx, dfun, dit, dst);
  LPB_CUDA(cudaGetLastError());
  return LPB_OK;
}

// ---------------------------------------------------------------- ragged lists (lpb_solve_many_ragged)
// Structure scan of LPs [lo, lo + cnt) of a ragged list: ns_dev[lp] = the run of trailing unit columns of LP lp.
int ragged_scan(int64_t lo, int64_t cnt, const LpDesc* ddesc, const double* dA, int* ns_dev, cudaStream_t stream) {
  const int64_t sgrid = cnt < (int64_t)kNumSMs * 8 ? cnt : (int64_t)kNumSMs * 8;
  ragged_structure_kernel<<<(unsigned)sgrid, 256, 0, stream>>>(lo, cnt, ddesc, dA, ns_dev);
  LPB_CUDA(cudaGetLastError());
  return LPB_OK;
}

namespace {
// Largest dynamic shared memory (bytes) at which ragged_ipm_kernel still runs two CTAs per SM.
int ragged_two_per_sm_bytes(size_t* out) {
  int lo = 0, hi = (int)(kSmemCap / sizeof(double));  // in doubles: lo is known to fit twice, hi + 1 not known
  while (lo < hi) {
    const int mid = (lo + hi + 1) / 2;
    int blocks = 0;
    LPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, ragged_ipm_kernel, kBT, (size_t)mid * sizeof(double)));
    if (blocks >= 2)
      lo = mid;
    else
      hi = mid - 1;
  }
  *out = (size_t)lo * sizeof(double);
  return LPB_OK;
}
}  // namespace

// Plans and launches LPs [lo, lo + cnt) of a ragged list, whose raw structure-scan results are in ns_host.  Each LP
// gets its own clamped ns (written to desc_host) and the kernel solve_many_launch would pick for a batch of that LP
// alone: K6 where m <= 64 and A fits beside M, else K8.  Up to three launches on `stream`: K8, then the K6 LPs too
// large for two CTAs per SM, then those that fit two per SM; each with the largest footprint of its group and one CTA
// per LP, the LPs in descending order of m^2 (n - ns) + m^3 (ties by index), so that the longest solves start first
// and the short ones fill the tail.  desc_host / order_host [lo, lo + cnt) must be page-locked: they are uploaded to
// desc_dev / order_dev on `stream`.
int ragged_launch(int64_t lo, int64_t cnt, LpDesc* desc_host, const int* ns_host, int* order_host, LpDesc* desc_dev,
                  int* order_dev, const double* dA, const double* db, const double* dc, const lpb_options& o,
                  double* dx, double* dfun, int64_t* dit, int32_t* dst, cudaStream_t stream) {
  LPB_CUDA(cudaFuncSetAttribute(ragged_ipm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemCap));
  LPB_CUDA(cudaFuncSetAttribute(ragged_streamed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemCap));
  size_t two_bytes = 0;
  LPB_TRY(ragged_two_per_sm_bytes(&two_bytes));
  enum { kK8 = 0, kK6One = 1, kK6Two = 2 };
  std::vector<int> grp[3];
  std::vector<double> cost((size_t)cnt);
  size_t smem[3] = {0, 0, 0};
  for (int64_t k = 0; k < cnt; ++k) {
    LpDesc& e = desc_host[lo + k];
    int ns = ns_host[lo + k];
    if (ns < 0 || ns > e.m || ns >= e.n) ns = 0;  // as scan_slack_structure
    e.ns = ns;
    int g;
    size_t bytes;
    const size_t k6 = batched_smem_doubles(e.m, e.n, ns) * sizeof(double);
    if (e.m <= kMaxM && k6 <= kSmemCap) {
      g = k6 <= two_bytes ? kK6Two : kK6One;
      bytes = k6;
    } else {
      g = kK8;
      bytes = batched_vec_smem_doubles<K8Dev>(e.m, e.n) * sizeof(double);
    }
    grp[g].push_back((int)(lo + k));
    smem[g] = std::max(smem[g], bytes);
    const double m = e.m;
    cost[(size_t)k] = m * m * (double)(e.n - ns) + m * m * m;
  }
  int* ord = order_host + lo;
  for (int g = 0; g < 3; ++g) {
    std::sort(grp[g].begin(), grp[g].end(), [&](int a, int b) {
      const double ca = cost[(size_t)(a - lo)], cb = cost[(size_t)(b - lo)];
      return ca > cb || (ca == cb && a < b);
    });
    ord = std::copy(grp[g].begin(), grp[g].end(), ord);
  }
  LPB_CUDA(cudaMemcpyAsync(desc_dev + lo, desc_host + lo, sizeof(LpDesc) * (size_t)cnt, cudaMemcpyHostToDevice, stream));
  LPB_CUDA(cudaMemcpyAsync(order_dev + lo, order_host + lo, sizeof(int) * (size_t)cnt, cudaMemcpyHostToDevice, stream));
  int64_t at = lo;
  for (int g = 0; g < 3; ++g) {
    const unsigned grid = (unsigned)grp[g].size();
    if (grid == 0) continue;
    if (g == kK8)
      ragged_streamed_kernel<<<grid, kBT8, smem[g], stream>>>(desc_dev, order_dev + at, dA, db, dc, o, dx, dfun, dit, dst);
    else
      ragged_ipm_kernel<<<grid, kBT, smem[g], stream>>>(desc_dev, order_dev + at, dA, db, dc, o, dx, dfun, dit, dst);
    LPB_CUDA(cudaGetLastError());
    at += grid;
  }
  return LPB_OK;
}

}  // namespace lpb
