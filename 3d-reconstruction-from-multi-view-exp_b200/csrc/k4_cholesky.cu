// K4 (factor/solve part): blocked right-looking Cholesky of the reduced camera system and the
// back substitution, replacing reference lib/bundle_adjustment.py:146 (`np.linalg.solve`, LAPACK
// dgesv).  The system is symmetric positive definite, so LU with pivoting is not needed; the
// survey measured <= 3e-14 relative effect on every per-iteration cost.
//
// Layout: S is n_pad x n_pad row-major (lower triangle used); row `rhs_row` = n carries the
// right-hand side and is swept along as one more row, so after the factorisation it holds
// y = L^-1 b.  Only L^T x = y is left for chol_backsolve_kernel.
//
// Two regimes by size, n_rows = n + 1 counting the right-hand-side row:
//   n_rows < 2048  the whole factorisation in ONE persistent cooperative launch (chol_fused_kernel:
//                  one step per 64-column panel, a grid barrier between the steps);
//   larger         two-level blocking: per 64-column panel the two launches below, and per 256-wide
//                  outer block one rank-256 update on the FP64 tensor cores (launch_chol_wide_update,
//                  divided over the ranks of a sharded run).
// Back substitution: one CTA (n < 1024), one 8-CTA cluster over distributed shared memory
// (n < 2048), the whole grid (larger).
//
// Large systems, per 64-column panel two launches:
//   chol_panel_kernel   every block eliminates the tall panel [diagonal block; its 64 rows] in
//                       shared memory (re-factoring the diagonal block per block is cheaper than
//                       a third launch, and the rows below need no separate triangular solve).
//                       Block 0 carries the rows of the identity instead, which yields
//                       W = L_D^-T for the back substitution (no serial solve there either).
//                       Writes L rows in place and a k-major copy Lt for the update.
//   chol_update_kernel  trailing update S -= L_panel L_panel^T on 64x64 tiles.
#include <cooperative_groups.h>

#include "ba_common.cuh"

namespace cg = cooperative_groups;

namespace ba {

constexpr int NB = kCholNB;

// Reciprocal to full double precision (<= ~1 ulp) with a short dependency chain: the hardware
// seed (MUFU.RCP64H, ~2^-20) and two Newton steps.  FP64 latency dominates the pivot chain below.
__device__ __forceinline__ double rcp_newton(double d) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
  r = fma(r, fma(-d, r, 1.0), r);
  r = fma(r, fma(-d, r, 1.0), r);
  return r;
}

// First non-positive pivot of a panel, encoded so that atomicMin picks the lowest column: a pivot
// that is exactly zero (or NaN) means a singular system -- the reference's LU raises
// LinAlgError("Singular matrix") there (:146; e.g. a camera without observations has an all-zero
// row) -- while a negative one is a system that damping can still repair: the step is rejected.
// Only the first failing panel of a factorisation reports (later pivots are contaminated).
constexpr int kNoBadPivot = 1 << 20;
__device__ __forceinline__ int bad_pivot_code(int col, double d) {
  return 2 * col + ((d == 0.0 || d != d) ? 1 : 0);
}
__device__ __forceinline__ void report_bad_pivot(ba_lm_state* ctl, int code) {
  if (code == kNoBadPivot || ctl->chol_fail) return;
  ctl->chol_fail = 1;
  if ((code & 1) && ctl->status == BA_OK) ctl->status = BA_ERR_SINGULAR;
}

constexpr int kPanelThreads = 8 * NB;  // 4 threads per row of the tall panel (16 columns each)
constexpr int kPanelCols = 16;          // columns per thread

__global__ void __launch_bounds__(kPanelThreads)
chol_panel_kernel(double* __restrict__ S, int ld, int n_rows, int k0, int nb,
                  double* __restrict__ Lt, double* __restrict__ W, ba_lm_state* ctl, int use_ctl) {
  if (use_ctl && ctl->done) return;
  extern __shared__ double psm[];
  // tall panel T[128][65]: rows 0..63 the diagonal block, rows 64..127 this block's rows
  double(*T)[NB + 1] = reinterpret_cast<double(*)[NB + 1]>(psm);
  double* col = psm + 2 * NB * (NB + 1);  // [2][128] published pivot column (double buffered)
  double* piv = col + 4 * NB;             // [64] pivots d_k
  __shared__ int s_fail;
  const int tid = threadIdx.x;
  // block 0 carries the rows of the identity (-> W = L_D^-T), block b >= 1 the 64 rows from rbase
  const int rbase = k0 + nb + ((int)blockIdx.x - 1) * NB;
  if (tid == 0) s_fail = kNoBadPivot;
  {
    // coalesced loads, all issued before the first use (L2 latency paid once)
    double vd[8], va[8];
    const int c = tid & 63;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int r = (tid >> 6) + 8 * u;
      vd[u] = (r == c) ? 1.0 : 0.0;
      if (r < nb && c <= r) vd[u] = S[(size_t)(k0 + r) * ld + k0 + c];
      va[u] = (blockIdx.x == 0 && r == c) ? 1.0 : 0.0;
      if (blockIdx.x != 0 && rbase + r < n_rows && c < nb) va[u] = S[(size_t)(rbase + r) * ld + k0 + c];
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int r = (tid >> 6) + 8 * u;
      T[r][c] = vd[u];
      T[NB + r][c] = va[u];
    }
  }
  __syncthreads();
  // Right-looking elimination with unscaled columns (A = Lu D^-1 Lu^T):
  //   a[r][c] -= a[r][k] a[c][k] / d_k   for c > k  (diagonal block: c <= r matters).
  // The rows below the diagonal block ride along, so there is no separate triangular solve.
  // Thread (r, cg) keeps columns 16 cg .. 16 cg + 15 of row r in registers; warps are uniform in
  // cg.  Per column: the owners publish column k of all 128 rows, one barrier, then every thread
  // still holding live columns does <= 16 FMAs with broadcast loads of the pivot row.  The whole
  // column step is one dependent chain (publish -> barrier -> reciprocal -> scale -> FMA ->
  // publish), so the 4-way split of a row is what shortens the panel: 16 instead of 64 FMAs behind
  // every barrier, 16 warps instead of 4 to hide the FP64 and shared-memory latencies.
  const int r = tid & (2 * NB - 1);  // row of the tall panel
  const int cg = tid >> 7;           // column group
  double a[kPanelCols];
#pragma unroll
  for (int j = 0; j < kPanelCols; ++j) a[j] = T[r][kPanelCols * cg + j];
  for (int g = 0; g < NB / kPanelCols; ++g) {
#pragma unroll
    for (int kk = 0; kk < kPanelCols; ++kk) {
      const int k = kPanelCols * g + kk;
      double* ck = col + (kk & 1) * (2 * NB);
      if (cg == g) ck[r] = a[kk];
      __syncthreads();
      if (cg >= g) {  // warp-uniform; groups < g hold finished columns only
        const double d = ck[k];
        if (r == k && cg == g) piv[k] = d;
        const double la = ck[r] * rcp_newton(d);
        const double2* pr = reinterpret_cast<const double2*>(ck + kPanelCols * cg);
        if (cg > g) {
#pragma unroll
          for (int jp = 0; jp < kPanelCols / 2; ++jp) {
            const double2 cv = pr[jp];
            a[2 * jp] = fma(-la, cv.x, a[2 * jp]);
            a[2 * jp + 1] = fma(-la, cv.y, a[2 * jp + 1]);
          }
        } else {
          // No per-row predicates: rows r <= k and the upper triangle of the diagonal block
          // accumulate values nobody reads.
#pragma unroll
          for (int jp = 0; jp < kPanelCols / 2; ++jp) {
            if (2 * jp + 1 > kk) {
              const double2 cv = pr[jp];
              if (2 * jp > kk) a[2 * jp] = fma(-la, cv.x, a[2 * jp]);
              a[2 * jp + 1] = fma(-la, cv.y, a[2 * jp + 1]);
            }
          }
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < kPanelCols; ++j) T[r][kPanelCols * cg + j] = a[j];
  __syncthreads();
  if (tid < NB) {
    const double d = piv[tid];
    if (tid < nb && !(d > 0.0)) atomicMin(&s_fail, bad_pivot_code(tid, d));
    piv[tid] = rsqrt(d);  // = 1 / L[tid][tid]
  }
  __syncthreads();
  for (int q = tid; q < 2 * NB * NB; q += kPanelThreads)  // L[r][c] = Lu[r][c] / sqrt(d_c)
    T[q >> 6][q & 63] *= piv[q & 63];
  __syncthreads();
  if (blockIdx.x == 0) {
    if (tid == 0) report_bad_pivot(ctl, s_fail);
    // L_D (k-major) for the trailing update: Lt[m][k0 + r] = L_D[r][m]
    for (int q = tid; q < NB * NB; q += kPanelThreads) {
      const int m = q >> 6, rr = q & 63;
      if (m < nb && rr < nb) Lt[(size_t)m * ld + k0 + rr] = rr >= m ? T[rr][m] : 0.0;
    }
    // W = L_D^-T from the identity rows
    for (int q = tid; q < NB * NB; q += kPanelThreads) W[q] = T[NB + (q >> 6)][q & 63];
  } else {
    for (int q = tid; q < NB * NB; q += kPanelThreads) {
      const int rr = q >> 6, c = q & 63;
      if (rbase + rr < n_rows && c < nb) S[(size_t)(rbase + rr) * ld + k0 + c] = T[NB + rr][c];
    }
    for (int q = tid; q < NB * NB; q += kPanelThreads) {
      const int c = q >> 6, rr = q & 63;
      if (rbase + rr < n_rows && c < nb) Lt[(size_t)c * ld + rbase + rr] = T[NB + rr][c];
    }
  }
}

// Trailing update S[r][c] -= sum_m L[r][k0+m] L[c][k0+m] on 64x64 tiles of the lower triangle
// (rows >= cols >= k0+nb, rows < n_rows, cols < c_end).  The diagonal blocks of S keep their
// pre-factor content: nothing reads L_D from S afterwards (the back substitution uses W = L_D^-T).
// c_end closes the current 256-wide outer block: the rest of the trailing matrix waits for the
// rank-256 update on the tensor cores (launch_chol_wide_update).
__global__ void __launch_bounds__(256)
chol_update_kernel(double* __restrict__ S, int ld, int n_rows, int c_end, int k0, int nb,
                   const double* __restrict__ Lt, const ba_lm_state* ctl, int use_ctl) {
  if (use_ctl && ctl->done) return;
  const int tid = threadIdx.x;
  const int t0 = k0 + nb;
  const int ti = blockIdx.y, tj = blockIdx.x;
  if (tj > ti) return;
  const int r0 = t0 + ti * 64, c0 = t0 + tj * 64;
  if (r0 >= n_rows || c0 >= c_end) return;
  constexpr int MH = NB;  // the whole panel depth in one pass: all loads in flight at once
  extern __shared__ double usm[];
  double(*sA)[64 + 1] = reinterpret_cast<double(*)[64 + 1]>(usm);
  double(*sB)[64 + 1] = reinterpret_cast<double(*)[64 + 1]>(usm + MH * 65);
  const int ty = tid / 16, tx = tid % 16;  // thread owns rows ty+16*i, cols tx+16*j
  double acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
  for (int m0 = 0; m0 < nb; m0 += MH) {
    __syncthreads();
    {
      double va[16], vb[16];
      const int x = tid & 63;
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int m = m0 + (tid >> 6) + 4 * u;
        va[u] = (m < nb && r0 + x < n_rows) ? Lt[(size_t)m * ld + r0 + x] : 0.0;
        vb[u] = (m < nb && c0 + x < n_rows) ? Lt[(size_t)m * ld + c0 + x] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        sA[(tid >> 6) + 4 * u][x] = va[u];
        sB[(tid >> 6) + 4 * u][x] = vb[u];
      }
    }
    __syncthreads();
#pragma unroll 8
    for (int m = 0; m < MH; ++m) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = sA[m][ty + 16 * i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = sB[m][tx + 16 * j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] += a[i] * b[j];
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = r0 + ty + 16 * i, c = c0 + tx + 16 * j;
      if (r < n_rows && c <= r && c < c_end) S[(size_t)r * ld + c] -= acc[i][j];
    }
}

// ---- small systems: one step per panel -----------------------------------------------------------
// The factorisation of a small system is a chain of latency-bound panels.  Step p of chol_fused_kernel
// takes the trailing update off that chain:
//   * panel blocks   -- as chol_panel_kernel, but each first applies the PREVIOUS panel's update
//                       to its own 128 x 64 slice (diagonal block + its rows of block column p):
//                       T -= Lp^T Lp on the FP64 tensor cores, operands staged k-major in shared
//                       memory next to T (about 2 us), then the elimination;
//   * update blocks  -- the rest of the previous panel's trailing update (64 x 64 tiles of the
//                       columns beyond block column p), which nothing in step p reads.
// Step p + 1 needs both and gets them after the grid barrier.  Lt alternates between two 64-row
// buffers so the previous panel stays readable while the current one is written.
__device__ __forceinline__ void step_dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

constexpr int kSLD = NB + 4;  // k-major operand rows padded to 68 doubles: conflict-free fragment loads

// acc[i][j] += sum_k A[k][row0 + 8 i] B[k][col0 + 8 j] over the 64-deep panel (DMMA fragments)
template <int FI, int FJ>
__device__ __forceinline__ void panel_product(const double* __restrict__ A, const double* __restrict__ B,
                                              int row0, int col0, int kq, double (&acc)[FI][FJ][2]) {
#pragma unroll 4
  for (int kk = 0; kk < NB; kk += 4) {
    double fa[FI], fb[FJ];
#pragma unroll
    for (int i = 0; i < FI; ++i) fa[i] = A[(kk + kq) * kSLD + row0 + 8 * i];
#pragma unroll
    for (int j = 0; j < FJ; ++j) fb[j] = B[(kk + kq) * kSLD + col0 + 8 * j];
#pragma unroll
    for (int i = 0; i < FI; ++i)
#pragma unroll
      for (int j = 0; j < FJ; ++j) step_dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
  }
}

// One virtual block `vb` of step p (vb < p_blocks: panel block, else update tile vb - p_blocks).
// S and Lp are read with ld.global.cg: other SMs wrote them earlier in the same launch, and the L1 is
// not coherent.
__device__ __forceinline__ void chol_step_body(int vb, double* S, int ld, int n_rows, int k0, int nb, int p_blocks,
                                               double* Lt, const double* Lp, double* W, ba_lm_state* ctl,
                                               double* psm) {
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  if (vb >= p_blocks) {
    // ---- update block: one 64 x 64 tile of the previous panel's trailing update ---------------
    double* sA = psm;              // [64][68] Lp[:, r0 ..]
    double* sB = psm + NB * kSLD;  // [64][68] Lp[:, c0 ..]
    const int t = vb - p_blocks;
    int ti = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
    while ((ti + 1) * (ti + 2) / 2 <= t) ++ti;
    while (ti * (ti + 1) / 2 > t) --ti;
    const int tj = t - ti * (ti + 1) / 2;
    const int t0 = k0 + NB;  // first column beyond the block column the panel blocks handle
    const int r0 = t0 + ti * NB, c0 = t0 + tj * NB;
    for (int q = tid; q < NB * NB; q += kPanelThreads) {
      const int m = q >> 6, x = q & 63;
      sA[m * kSLD + x] = r0 + x < n_rows ? __ldcg(Lp + (size_t)m * ld + r0 + x) : 0.0;
      sB[m * kSLD + x] = c0 + x < n_rows ? __ldcg(Lp + (size_t)m * ld + c0 + x) : 0.0;
    }
    __syncthreads();
    const int rb = warp >> 2, cb = warp & 3;  // 16 x 16 sub-tile per warp
    if (ti == tj && cb > rb) return;          // strictly above the diagonal
    double acc[2][2][2] = {};
    panel_product<2, 2>(sA, sB, rb * 16 + (lane >> 2), cb * 16 + (lane >> 2), lane & 3, acc);
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int r = r0 + rb * 16 + (lane >> 2) + 8 * i, c = c0 + cb * 16 + 2 * (lane & 3) + 8 * j;
        if (r >= n_rows || c > r) continue;
        double* dst = S + (size_t)r * ld + c;
        dst[0] = __ldcg(dst) - acc[i][j][0];
        if (c + 1 <= r) dst[1] = __ldcg(dst + 1) - acc[i][j][1];
      }
    return;
  }
  // ---- panel block (see chol_panel_kernel for the elimination) ----------------------------------
  double(*T)[NB + 1] = reinterpret_cast<double(*)[NB + 1]>(psm);
  double* col = psm + 2 * NB * (NB + 1);  // [2][128]
  double* piv = col + 4 * NB;             // [64]
  double* sB = piv + NB;                  // [64][68] Lp[:, k0 ..]   (previous panel, k-major)
  double* sA = sB + NB * kSLD;            // [64][68] Lp[:, rbase ..]
  __shared__ int s_fail;
  const int rbase = k0 + nb + (vb - 1) * NB;
  if (tid == 0) s_fail = kNoBadPivot;
  {
    double vd[8], va[8];
    const int c = tid & 63;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int r = (tid >> 6) + 8 * u;
      vd[u] = (r == c) ? 1.0 : 0.0;
      if (r < nb && c <= r) vd[u] = __ldcg(S + (size_t)(k0 + r) * ld + k0 + c);
      va[u] = (vb == 0 && r == c) ? 1.0 : 0.0;
      if (vb != 0 && rbase + r < n_rows && c < nb) va[u] = __ldcg(S + (size_t)(rbase + r) * ld + k0 + c);
    }
    if (Lp) {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int m = (tid >> 6) + 8 * u;
        sB[m * kSLD + c] = k0 + c < n_rows ? __ldcg(Lp + (size_t)m * ld + k0 + c) : 0.0;
        sA[m * kSLD + c] = (vb != 0 && rbase + c < n_rows) ? __ldcg(Lp + (size_t)m * ld + rbase + c) : 0.0;
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int r = (tid >> 6) + 8 * u;
      T[r][c] = vd[u];
      T[NB + r][c] = va[u];
    }
  }
  __syncthreads();
  if (Lp) {
    // previous panel's update of this slice: warp -> 16 rows x 32 columns of the 128 x 64 slice
    const int rb = warp >> 1, ch = warp & 1;
    const bool own = rb >= 4;  // rows 64..127 = this block's rows, else the diagonal block
    if (!(own && vb == 0)) {
      double acc[2][4][2] = {};
      panel_product<2, 4>(own ? sA : sB, sB, (own ? rb - 4 : rb) * 16 + (lane >> 2), ch * 32 + (lane >> 2),
                          lane & 3, acc);
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int rl = (own ? rb - 4 : rb) * 16 + (lane >> 2) + 8 * i;  // row inside its 64-block
          const int c = ch * 32 + 2 * (lane & 3) + 8 * j;
          const bool row_ok = own ? rbase + rl < n_rows : rl < nb;
          if (!row_ok) continue;
          double* dst = &T[(own ? NB : 0) + rl][c];
          if (c < nb) dst[0] -= acc[i][j][0];
          if (c + 1 < nb) dst[1] -= acc[i][j][1];
        }
    }
    __syncthreads();
  }
  const int r = tid & (2 * NB - 1);
  const int cg = tid >> 7;
  double a[kPanelCols];
#pragma unroll
  for (int j = 0; j < kPanelCols; ++j) a[j] = T[r][kPanelCols * cg + j];
  // Look-ahead: the thread that owns column k + 1 updates that entry first and publishes it (into the
  // other column buffer) BEFORE its remaining FMAs of step k, so the next step's column is on its way
  // while the bulk of this step's update runs; the barrier of step k + 1 then waits for arithmetic only.
  // Every entry still receives the same FMAs in the same order: the factor is bit-identical.
  if (cg == 0) col[r] = a[0];
  for (int g = 0; g < NB / kPanelCols; ++g) {
#pragma unroll
    for (int kk = 0; kk < kPanelCols; ++kk) {
      const int k = kPanelCols * g + kk;
      double* ck = col + (kk & 1) * (2 * NB);
      double* cn = col + ((kk + 1) & 1) * (2 * NB);
      __syncthreads();
      if (cg >= g) {
        const double d = ck[k];
        if (r == k && cg == g) piv[k] = d;
        const double la = ck[r] * rcp_newton(d);
        const double2* pr = reinterpret_cast<const double2*>(ck + kPanelCols * cg);
        if (cg > g) {
#pragma unroll
          for (int jp = 0; jp < kPanelCols / 2; ++jp) {
            const double2 cv = pr[jp];
            a[2 * jp] = fma(-la, cv.x, a[2 * jp]);
            a[2 * jp + 1] = fma(-la, cv.y, a[2 * jp + 1]);
            if (jp == 0 && kk == kPanelCols - 1 && cg == g + 1) cn[r] = a[0];
          }
        } else {
#pragma unroll
          for (int jp = 0; jp < kPanelCols / 2; ++jp) {
            if (2 * jp + 1 > kk) {
              const double2 cv = pr[jp];
              if (2 * jp > kk) a[2 * jp] = fma(-la, cv.x, a[2 * jp]);
              a[2 * jp + 1] = fma(-la, cv.y, a[2 * jp + 1]);
              if (kk + 1 < kPanelCols && jp == (kk + 1) / 2) cn[r] = a[kk + 1];
            }
          }
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < kPanelCols; ++j) T[r][kPanelCols * cg + j] = a[j];
  __syncthreads();
  if (tid < NB) {
    const double d = piv[tid];
    if (tid < nb && !(d > 0.0)) atomicMin(&s_fail, bad_pivot_code(tid, d));
    piv[tid] = rsqrt(d);
  }
  __syncthreads();
  for (int q = tid; q < 2 * NB * NB; q += kPanelThreads) T[q >> 6][q & 63] *= piv[q & 63];
  __syncthreads();
  if (vb == 0) {
    if (tid == 0) report_bad_pivot(ctl, s_fail);
    for (int q = tid; q < NB * NB; q += kPanelThreads) {
      const int m = q >> 6, rr = q & 63;
      if (m < nb && rr < nb) Lt[(size_t)m * ld + k0 + rr] = rr >= m ? T[rr][m] : 0.0;
    }
    for (int q = tid; q < NB * NB; q += kPanelThreads) W[q] = T[NB + (q >> 6)][q & 63];
  } else {
    for (int q = tid; q < NB * NB; q += kPanelThreads) {
      const int rr = q >> 6, c = q & 63;
      if (rbase + rr < n_rows && c < nb) S[(size_t)(rbase + rr) * ld + k0 + c] = T[NB + rr][c];
    }
    for (int q = tid; q < NB * NB; q += kPanelThreads) {
      const int c = q >> 6, rr = q & 63;
      if (rbase + rr < n_rows && c < nb) Lt[(size_t)c * ld + rbase + rr] = T[NB + rr][c];
    }
  }
}

// Back substitution L^T x = y (y = row rhs_row of the factor) by 64-column blocks from the
// last one: rhs_B = y_B - L[below, B]^T x_below (GEMV), x_B = W_B rhs_B with W_B = L_BB^-T from
// the panel kernel.  One block; x lives in shared memory.
__global__ void __launch_bounds__(1024)
chol_backsolve_kernel(const double* __restrict__ S, int ld, int n, int rhs_row,
                      const double* __restrict__ W, double* __restrict__ dxi,
                      const ba_lm_state* ctl, int use_ctl) {
  if (use_ctl && ctl->done) return;
  extern __shared__ double sm[];
  double* x = sm;             // [n]
  double* red = sm + n;       // [16][64]
  double* rhs = red + 16 * 64;  // [64]
  const int tid = threadIdx.x;
  const int tx = tid & 63, ty = tid >> 6;  // 64 columns x 16 row groups
  const int nblk = (n + 63) / 64;
  for (int blk = nblk - 1; blk >= 0; --blk) {
    const int b0 = blk * 64;
    const int b1 = b0 + 64 < n ? b0 + 64 : n;
    const int w = b1 - b0;
    // W row for the second product and y_B are fetched now so their L2 latency overlaps the GEMV
    const int wj = tid >> 4, wpart = tid & 15;
    const double* Wj = W + (size_t)blk * NB * NB + (size_t)wj * NB;
    double wv[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) wv[i] = Wj[wpart + 16 * i];
    const double yb = (ty == 0 && tx < w) ? S[(size_t)rhs_row * ld + b0 + tx] : 0.0;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;  // independent chains: FP64 latency is long
    if (tx < w) {
      int k = b1 + ty;
      for (; k + 48 < n; k += 64) {
        const double s0 = S[(size_t)k * ld + b0 + tx], s1 = S[(size_t)(k + 16) * ld + b0 + tx];
        const double s2 = S[(size_t)(k + 32) * ld + b0 + tx], s3 = S[(size_t)(k + 48) * ld + b0 + tx];
        a0 = fma(s0, x[k], a0);
        a1 = fma(s1, x[k + 16], a1);
        a2 = fma(s2, x[k + 32], a2);
        a3 = fma(s3, x[k + 48], a3);
      }
      for (; k < n; k += 16) a0 = fma(S[(size_t)k * ld + b0 + tx], x[k], a0);
    }
    red[ty * 64 + tx] = (a0 + a1) + (a2 + a3);
    __syncthreads();
    if (ty == 0) {
      double p[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
      for (int g = 0; g < 16; ++g) p[g & 3] += red[g * 64 + tx];
      rhs[tx] = yb - ((p[0] + p[1]) + (p[2] + p[3]));
    }
    __syncthreads();
    {
      // x_B[j] = sum_c W[j][c] rhs[c]; thread (j = tid / 16, part = tid % 16)
      const int j = wj, part = wpart;
      double s = (wv[0] * rhs[part] + wv[1] * rhs[part + 16]) +
                 (wv[2] * rhs[part + 32] + wv[3] * rhs[part + 48]);
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
      if (part == 0 && j < w) x[b0 + j] = s;
    }
    __syncthreads();
  }
  for (int k = tid; k < n; k += 1024) dxi[k] = x[k];
}

// The same back substitution for large systems, spread over the GPU (the single-block kernel
// above streams n^2/2 doubles through one SM: 4.6 ms at n = 9000).  Right-looking: once x_B of a
// 64-block is known, y[c] -= sum_{r in B} L[r][c] x_B[r] for all columns c before B.  Columns are
// dealt to the CTAs in chunks of 64; after a grid barrier every CTA forms the next x_B itself
// (x_B = W_B y_B, 64x64, redundantly: no second barrier), the owner of the chunk stores it, and
// all CTAs update their own chunks.  The rows L[B][.] a CTA needs for its next update do not
// depend on x, so they are fetched BEFORE the barrier and the HBM latency overlaps the wait.
// One barrier per block; fixed summation order (deterministic).  All CTAs must be co-resident:
// the grid never exceeds the SM count and the kernel runs alone on its stream.
// The kernel is launched cooperatively (all CTAs co-resident or the launch fails), and the spin is
// bounded as well: after kBarrierLimitNs the waiting CTA poisons the counter (every later barrier of
// every CTA falls through) and raises BA_ERR_BARRIER in the control block instead of hanging the GPU.
constexpr unsigned long long kBarrierLimitNs = 10ull * 1000000000ull;
__device__ __forceinline__ void grid_barrier(unsigned int* bar, unsigned int target, ba_lm_state* ctl) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(bar, 1u);
    unsigned int v, polls = 0;
    unsigned long long t0 = 0;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
      if (v >= target) break;
      if ((++polls & 1023u) == 0) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (t0 == 0) t0 = now;
        else if (now - t0 > kBarrierLimitNs) {
          atomicOr(bar, 0x80000000u);
          ctl->status = BA_ERR_BARRIER;
          break;
        }
      }
    } while (true);
  }
  __syncthreads();
}

// ---- small systems: the whole factorisation in ONE persistent launch ------------------------------
// All steps run in one cooperative launch, a grid barrier between them, so the latency-bound panel
// chain pays no launch, drain and first loads per panel.  Panel blocks go to the first CTAs; the
// update tiles of the previous panel, which nothing in the step waits for, are dealt to the CTAs that
// hold no panel block, so that the CTAs on the critical path (slice update, elimination) reach the
// barrier first.
__global__ void __launch_bounds__(kPanelThreads)
chol_fused_kernel(double* S, int ld, int n, int n_rows, double* Lt, double* Winv, unsigned int* bar,
                  ba_lm_state* ctl, int use_ctl) {
  if (use_ctl && ctl->done) return;
  extern __shared__ double psm[];
  const int G = (int)gridDim.x, cta = (int)blockIdx.x;
  unsigned int epoch = 0;
  int panel = 0;
  for (int k0 = 0; k0 < n; k0 += NB, ++panel) {
    const int nb = n - k0 < NB ? n - k0 : NB;
    const int below = n_rows - (k0 + nb);
    const int p_blocks = 1 + (below + NB - 1) / NB;
    int u_blocks = 0;
    if (panel > 0) {
      const int rest = n_rows - (k0 + NB);  // rows / columns beyond block column `panel`
      if (rest > 0) {
        const int nt = (rest + NB - 1) / NB;
        u_blocks = nt * (nt + 1) / 2;
      }
    }
    double* Lt_cur = Lt + (size_t)(panel & 1) * NB * ld;
    const double* Lt_prev = panel > 0 ? Lt + (size_t)((panel - 1) & 1) * NB * ld : nullptr;
    double* W = Winv + (size_t)panel * NB * NB;
    for (int vb = cta; vb < p_blocks; vb += G) {
      chol_step_body(vb, S, ld, n_rows, k0, nb, p_blocks, Lt_cur, Lt_prev, W, ctl, psm);
      __syncthreads();
    }
    if (u_blocks > 0) {
      const bool spare = G > p_blocks;  // CTAs without a panel block take all the tiles
      const int first = spare ? cta - p_blocks : cta;
      const int stride = spare ? G - p_blocks : G;
      if (first >= 0)
        for (int t = first; t < u_blocks; t += stride) {
          chol_step_body(p_blocks + t, S, ld, n_rows, k0, nb, p_blocks, Lt_cur, Lt_prev, W, ctl, psm);
          __syncthreads();
        }
    }
    if (k0 + NB < n) grid_barrier(bar, ++epoch * (unsigned int)G, ctl);
  }
}

__global__ void __launch_bounds__(256)
chol_backsolve_grid_kernel(const double* __restrict__ S, int ld, int n, int rhs_row,
                           const double* __restrict__ W, double* __restrict__ ywork,
                           double* __restrict__ dxi, unsigned int* bar, ba_lm_state* ctl,
                           int use_ctl) {
  if (use_ctl && ctl->done) return;
  __shared__ double xB[NB], yB[NB], part[4][NB];
  const int tid = threadIdx.x, G = gridDim.x, cta = blockIdx.x;
  const int col = tid & 63, rg = tid >> 6;  // update: 64 columns x 4 groups of 16 rows
  const int nblk = (n + NB - 1) / NB;
  // running rhs of the chunks this CTA owns (chunk q belongs to CTA q % G)
  for (int q = cta; q < nblk; q += G)
    if (tid < NB && q * NB + tid < n) ywork[q * NB + tid] = S[(size_t)rhs_row * ld + q * NB + tid];
  // rows of block `blk` restricted to chunk q: 16 values per thread, fetched one step ahead
  double pre[16];
  auto prefetch = [&](int blk, int q) {
    const int b0 = blk * NB;
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const int r = b0 + rg * 16 + u;
      pre[u] = (q < blk && r < n) ? S[(size_t)r * ld + q * NB + col] : 0.0;
    }
  };
  prefetch(nblk - 1, cta);
  unsigned int epoch = 0;
  grid_barrier(bar, ++epoch * G, ctl);
  for (int blk = nblk - 1; blk >= 0; --blk) {
    const int b0 = blk * NB;
    const int w = n - b0 < NB ? n - b0 : NB;
    if (tid < NB) yB[tid] = tid < w ? __ldcg(ywork + b0 + tid) : 0.0;
    __syncthreads();
    {
      const int j = tid >> 2, p4 = tid & 3;  // x_B[j] = sum_c W[j][c] y_B[c]; columns 4 p4 + 16 m + {0..3}: coalesced
      const double2* Wj = reinterpret_cast<const double2*>(W + (size_t)blk * NB * NB + (size_t)j * NB + p4 * 4);
      double a0 = 0.0, a1 = 0.0;
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const double2 lo = Wj[8 * m], hi = Wj[8 * m + 1];
        const double* yq = yB + p4 * 4 + 16 * m;
        a0 = fma(lo.x, yq[0], a0);
        a1 = fma(lo.y, yq[1], a1);
        a0 = fma(hi.x, yq[2], a0);
        a1 = fma(hi.y, yq[3], a1);
      }
      double sx = a0 + a1;
      sx += __shfl_xor_sync(0xffffffffu, sx, 1);
      sx += __shfl_xor_sync(0xffffffffu, sx, 2);
      if (p4 == 0) {
        xB[j] = sx;
        if (blk % G == cta && j < w) dxi[b0 + j] = sx;
      }
    }
    __syncthreads();
    // chunks of this CTA below the block (with G >= nblk, the usual case, exactly one)
    for (int q = cta; q < blk; q += G) {
      double acc = 0.0;
#pragma unroll
      for (int u = 0; u < 16; ++u) acc = fma(pre[u], xB[rg * 16 + u], acc);
      if (q + G < blk) prefetch(blk, q + G);
      part[rg][col] = acc;
      __syncthreads();
      if (rg == 0 && q * NB + col < n)
        ywork[q * NB + col] -= (part[0][col] + part[1][col]) + (part[2][col] + part[3][col]);
      __syncthreads();
    }
    if (blk > 0) prefetch(blk - 1, cta);  // static data: in flight while the barrier is awaited
    if (blk > 0) grid_barrier(bar, ++epoch * G, ctl);
  }
}

// ---- back substitution on one thread-block cluster (1024 <= n < 2048) ------------------------------
// The single-block kernel streams the whole factor through one SM (C3, n = 1793: 12.9 MB, 0.21 ms --
// a quarter of the factor + solve time); the grid-wide kernel pays a ~2 us software barrier and a
// round trip through global memory for the running right-hand side per 64-block and is no faster at
// this size.  Here eight CTAs form ONE CLUSTER: the running right-hand side lives in the shared
// memory of the CTA that owns the chunk (chunk q belongs to CTA q % 8), the other CTAs read the
// block they need through distributed shared memory, and the steps are separated by the hardware
// cluster barrier.  Right-looking like the grid kernel: every CTA forms x_B = W_B y_B itself and
// updates its own chunks; the factor rows and W of the next step are static and fetched before the
// barrier.  Fixed summation order: deterministic.
constexpr int kBsCluster = 8;
constexpr int kBsMaxOwn = 4;  // chunks per CTA
// The cluster from n = 1024: against one CTA it measured 8 us slower at 7 blocks (C2), 37 us faster
// at 29 blocks (C3).
constexpr int kBsClusterMinN = 1024;
constexpr int kBsGridMinN = 2048;  // from here the grid-wide kernel
static_assert((kBsGridMinN - 1 + NB - 1) / NB <= kBsCluster * kBsMaxOwn,
              "every 64-block of an n < kBsGridMinN system needs a chunk slot in the cluster");

__global__ void __launch_bounds__(256)
chol_backsolve_cluster_kernel(const double* __restrict__ S, int ld, int n, int rhs_row,
                              const double* __restrict__ W, double* __restrict__ dxi,
                              const ba_lm_state* ctl, int use_ctl) {
  if (use_ctl && ctl->done) return;  // the same answer in every CTA of the cluster
  cg::cluster_group cluster = cg::this_cluster();
  const int cta = (int)cluster.block_rank(), G = (int)cluster.num_blocks();
  __shared__ double ych[kBsMaxOwn][NB];  // running rhs of the chunks this CTA owns (chunk = cta + G * slot)
  __shared__ double xB[NB], yB[NB], part[4][NB];
  const int tid = threadIdx.x;
  const int col = tid & 63, rg = tid >> 6;  // update: 64 columns x 4 groups of 16 rows
  const int wj = tid >> 2, wp4 = tid & 3;   // x_B: row j, quarter p4 of the dot product
  const int nblk = (n + NB - 1) / NB;
  for (int slot = 0; slot < kBsMaxOwn; ++slot) {
    const int q = cta + G * slot;
    if (tid < NB) ych[slot][tid] = (q < nblk && q * NB + tid < n) ? S[(size_t)rhs_row * ld + q * NB + tid] : 0.0;
  }
  // static data of a step, fetched one step ahead: the rows of block `blk` over this CTA's chunks
  // and this thread's piece of W_blk
  double pre[kBsMaxOwn][16], wv[16];
  auto prefetch = [&](int blk) {
    const int b0 = blk * NB;
#pragma unroll
    for (int slot = 0; slot < kBsMaxOwn; ++slot) {
      const int q = cta + G * slot;
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int r = b0 + rg * 16 + u;
        pre[slot][u] = (q < blk && r < n) ? S[(size_t)r * ld + q * NB + col] : 0.0;
      }
    }
    // thread (j, p4) takes columns 4 p4 + 16 m + {0..3}: the four threads of a row read 64 contiguous
    // bytes per m (with 16 consecutive columns per thread a warp-wide load touched 32 lines -- 4 us per
    // 64-block, more than everything else in the step)
    const double2* Wj = reinterpret_cast<const double2*>(W + (size_t)blk * NB * NB + (size_t)wj * NB + wp4 * 4);
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const double2 lo = Wj[8 * m], hi = Wj[8 * m + 1];
      wv[4 * m] = lo.x; wv[4 * m + 1] = lo.y; wv[4 * m + 2] = hi.x; wv[4 * m + 3] = hi.y;
    }
  };
  __syncthreads();
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  prefetch(nblk - 1);
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
  for (int blk = nblk - 1; blk >= 0; --blk) {
    const int b0 = blk * NB;
    const int w = n - b0 < NB ? n - b0 : NB;
    {
      const double* owner_y = cluster.map_shared_rank(&ych[0][0], blk % G);  // distributed shared memory
      if (tid < NB) yB[tid] = owner_y[(blk / G) * NB + tid];
    }
    __syncthreads();
    {
      double a0 = 0.0, a1 = 0.0;  // x_B[j] = sum_c W[j][c] y_B[c]
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const double* yq = yB + wp4 * 4 + 16 * m;
        a0 = fma(wv[4 * m], yq[0], a0);
        a1 = fma(wv[4 * m + 1], yq[1], a1);
        a0 = fma(wv[4 * m + 2], yq[2], a0);
        a1 = fma(wv[4 * m + 3], yq[3], a1);
      }
      double sx = a0 + a1;
      sx += __shfl_xor_sync(0xffffffffu, sx, 1);
      sx += __shfl_xor_sync(0xffffffffu, sx, 2);
      if (wp4 == 0) {
        xB[wj] = sx;
        if (blk % G == cta && wj < w) dxi[b0 + wj] = sx;
      }
    }
    __syncthreads();
#pragma unroll
    for (int slot = 0; slot < kBsMaxOwn; ++slot) {
      const int q = cta + G * slot;
      if (q < blk) {  // uniform in the CTA
        double acc = 0.0;
#pragma unroll
        for (int u = 0; u < 16; ++u) acc = fma(pre[slot][u], xB[rg * 16 + u], acc);
        part[rg][col] = acc;
        __syncthreads();
        if (rg == 0) ych[slot][col] -= (part[0][col] + part[1][col]) + (part[2][col] + part[3][col]);
        __syncthreads();
      }
    }
    // Split barrier: arrive (release: this step's updates of the running right-hand side) BEFORE the
    // next step's loads are issued -- a release after them would wait for all of them to return --
    // and wait after; the loads then overlap the barrier.
    asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
    if (blk > 0) prefetch(blk - 1);
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
  }
}

// Rows (with the right-hand-side row) from which the factorisation is two-level.
constexpr int kCholTwoLevelRows = 2048;

int launch_cholesky_solve(ba_engine* e, bool conditional, cudaStream_t s) {
  const int use_ctl = conditional ? 1 : 0;
  const int n = e->n_full, n_rows = e->rhs_row + 1, ld = e->n_pad;
  if (n_rows < kCholTwoLevelRows) {
    constexpr size_t kStepSmem = (2 * NB * (NB + 1) + 5 * NB + 2 * NB * kSLD) * sizeof(double);
    // the persistent kernel needs its CTAs co-resident (cooperative launch): ask once how many fit
    static int fused_ctas_per_sm = -1;
    if (fused_ctas_per_sm < 0) {
      BA_CUDA(cudaFuncSetAttribute(chol_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStepSmem));
      int per_sm = 0;
      BA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, chol_fused_kernel, kPanelThreads, kStepSmem));
      fused_ctas_per_sm = per_sm;
    }
    if (fused_ctas_per_sm == 0) {
      set_error("chol_fused_kernel does not fit on an SM (%d threads, %zu B of shared memory)", kPanelThreads,
                kStepSmem);
      return BA_ERR_CUDA;
    }
    // grid: enough CTAs for the busiest step (panel blocks + the tiles of the previous panel's update)
    int want = 1;
    {
      int panel = 0;
      for (int k0 = 0; k0 < n; k0 += NB, ++panel) {
        const int nb = n - k0 < NB ? n - k0 : NB;
        const int below = n_rows - (k0 + nb);
        int blocks = 1 + (below + NB - 1) / NB;
        const int rest = n_rows - (k0 + NB);
        if (panel > 0 && rest > 0) {
          const int nt = (rest + NB - 1) / NB;
          blocks += nt * (nt + 1) / 2;
        }
        if (blocks > want) want = blocks;
      }
    }
    const int fit = e->num_sms * fused_ctas_per_sm;
    const int G = want < fit ? want : fit;
    BA_CUDA(cudaMemsetAsync(e->chol_bar, 0, sizeof(unsigned int), s));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(G);
    cfg.blockDim = dim3(kPanelThreads);
    cfg.dynamicSmemBytes = kStepSmem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    BA_CUDA(cudaLaunchKernelEx(&cfg, chol_fused_kernel, e->P(), ld, n, n_rows, e->Lt, e->Winv, e->chol_bar, e->ctl,
                               use_ctl));
    BA_LAUNCH_CHECK();
  } else {
    // Two-level blocking.  Inside a 256-wide outer block the panels update only the block's own
    // columns; the rest of the trailing matrix then gets ONE rank-256 update on the FP64 tensor cores
    // (the SYRK kernel of K3 with a subtracting epilogue), which reads and writes S a quarter as often.
    constexpr int OB = kCholOB;
    constexpr size_t kPanelSmem = (2 * NB * (NB + 1) + 5 * NB) * sizeof(double);
    BA_CUDA(cudaFuncSetAttribute(chol_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPanelSmem));
    constexpr size_t kUpdateSmem = 2 * NB * 65 * sizeof(double);
    BA_CUDA(cudaFuncSetAttribute(chol_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kUpdateSmem));
    CholSplit split;
    comm_chol_split(e, &split);
    int panel = 0;
    for (int K0 = 0; K0 < n; K0 += OB) {
      // columns the panels of this block update themselves
      const int c_end = K0 + OB < n_rows ? K0 + OB : n_rows;
      for (int k0 = K0; k0 < K0 + OB && k0 < n; k0 += NB, ++panel) {
        const int nb = n - k0 < NB ? n - k0 : NB;
        const int below = n_rows - (k0 + nb);
        const int pblocks = 1 + (below + NB - 1) / NB;
        double* Lt = e->Lt + (size_t)(k0 - K0) * ld;  // k-rows of this panel inside the block column
        chol_panel_kernel<<<pblocks, kPanelThreads, kPanelSmem, s>>>(e->P(), ld, n_rows, k0, nb, Lt,
                                                                     e->Winv + (size_t)panel * NB * NB, e->ctl, use_ctl);
        BA_LAUNCH_CHECK();
        if (below <= 0 || k0 + nb >= c_end) continue;
        dim3 grid((c_end - (k0 + nb) + 63) / 64, (below + 63) / 64);
        chol_update_kernel<<<grid, 256, kUpdateSmem, s>>>(e->P(), ld, n_rows, c_end, k0, nb, Lt, e->ctl, use_ctl);
        BA_LAUNCH_CHECK();
      }
      if (K0 + OB < n_rows) {  // all four panels of the block are full here
        const int t0 = K0 + OB, remaining = n_rows - t0;
        if (split.world > 1 && remaining >= kCholSplitMinRows) {
          // sharded run: every rank updates its own tile rows and sends the part the next panels
          // read -- the next block column, or everything that is left when the following update
          // will not be divided any more -- to all ranks; one flag exchange closes the step
          const bool next_divided = t0 + OB < n_rows && n_rows - (t0 + OB) >= kCholSplitMinRows;
          split.push_cols = next_divided ? OB : (remaining + 127) / 128 * 128;
          // Before the FIRST divided update nothing has ordered the ranks since the sum of `red`:
          // a rank that is ahead would store into a peer's matrix while that peer is still
          // assembling it in place.  One more flag exchange closes the window (the later steps are
          // ordered by the exchange that ends the step before).
          if (K0 == 0) BA_TRY(launch_comm_chol_sync(e, conditional, s));
          BA_TRY(launch_chol_wide_update(e->P(), ld, n_rows, t0, e->Lt, OB, e->ctl, s, &split));
          BA_TRY(launch_comm_chol_sync(e, conditional, s));
        } else {
          BA_TRY(launch_chol_wide_update(e->P(), ld, n_rows, t0, e->Lt, OB, e->ctl, s, nullptr));
        }
      }
    }
  }
  if (n >= kBsGridMinN) {
    const int nblk = (n + NB - 1) / NB;
    const int G = nblk < e->num_sms ? nblk : e->num_sms;
    BA_CUDA(cudaMemsetAsync(e->chol_bar, 0, sizeof(unsigned int), s));
    // cooperative launch: the driver admits the grid only if all G CTAs can be resident together,
    // whatever else the device is running
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(G);
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    BA_CUDA(cudaLaunchKernelEx(&cfg, chol_backsolve_grid_kernel, (const double*)e->P(), ld, n, e->rhs_row,
                               (const double*)e->Winv, e->ywork, e->dxi, e->chol_bar, e->ctl, use_ctl));
    BA_LAUNCH_CHECK();
    return BA_OK;
  }
  if (n >= kBsClusterMinN) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kBsCluster);
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = kBsCluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    BA_CUDA(cudaLaunchKernelEx(&cfg, chol_backsolve_cluster_kernel, (const double*)e->P(), ld, n, e->rhs_row,
                               (const double*)e->Winv, e->dxi, (const ba_lm_state*)e->ctl, use_ctl));
    BA_LAUNCH_CHECK();
    return BA_OK;
  }
  const size_t smem = ((size_t)n + 16 * 64 + 64) * sizeof(double);  // n < 1024: at most 17 KB
  BA_CUDA(cudaFuncSetAttribute(chol_backsolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)smem));
  chol_backsolve_kernel<<<1, 1024, smem, s>>>(e->P(), ld, n, e->rhs_row, e->Winv, e->dxi, e->ctl,
                                              use_ctl);
  BA_LAUNCH_CHECK();
  return BA_OK;
}

}  // namespace ba
