// K8: marginal covariances of the cameras and the points at the current state (ba_covariance).
//
// Everything is taken at the committed state without damping, with the gauge unknowns pinned.
// H = 2 J^T J is the Gauss-Newton Hessian, S = U - sum_j Y_j Y_j^T its reduced camera system and
// L its Cholesky factor (S = L L^T), with Y_j = W_j^T L_j^-T as K2b writes it (V_j = L_j L_j^T).
//   camera i:  [H^-1]_ii = S^-1[9i .. 9i+8]^2,  S^-1[a][b] = <L^-1 e_a, L^-1 e_b>
//   point j:   [H^-1]_jj = L_j^-T (I_3 + Q_j) L_j^-1,  Q_j[d][e] = <L^-1 y_{3j+d}, L^-1 y_{3j+e}>
// with y_r row r of the k-major Y operand.  Both are Gram matrices of consecutive groups of
// forward-substituted rows (9 per camera, 3 per point); S^-1 is never formed.  The covariance is
// sigma^2 (J^T J)^-1 = 2 sigma^2 H^-1 with sigma^2 = E / (2 n_obs - (3N + 9M - 7)).
//
// Pipeline per batch of right-hand-side rows (k-major, [rows][n_pad], columns < 9M):
//   fill      rows of Yt (dense), the 9 x 3 blocks of Ysp scattered into zeros (sparse), or unit rows
//   cov_trsm_kernel  X = B L^-T in place on the FP64 tensor cores, one CTA per 64-row strip
//   cov_gram_kernel  the g x g Gram matrix of every group of g rows, mapped and scaled
#include "ba_common.cuh"

namespace ba {

constexpr int kCovStrip = 64;                          // rows per CTA of the solve = width of L's blocks
constexpr int kCovLd = kCholNB + 4;                    // shared rows padded to 68 doubles
constexpr int kCovTile = kCovStrip * kCovLd;           // doubles per staged 64 x 64 tile
constexpr size_t kCovBatchBytes = (size_t)2 << 30;     // right-hand-side batch: at most 2 GiB
constexpr int kCovBatchQuantum = 576;                  // = lcm(64, 9): whole strips, whole cameras and points
static_assert(kCovStrip == kCholNB, "a strip's column blocks are the factor's 64-column panels");
static_assert(kCovBatchQuantum % kCovStrip == 0 && kCovBatchQuantum % 9 == 0, "batch quantum");

// ---- fill kernels: k-major right-hand sides (the batch is zeroed before) -------------------------
// dense: rows [r0, r0 + rows) of Yt, columns < n (column n = 9M holds z_j, not part of y)
__global__ void cov_fill_dense_kernel(const double* __restrict__ Yt, int ld, int n, int64_t r0, int rows,
                                      double* __restrict__ B) {
  const int64_t total = (int64_t)rows * n;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += stride) {
    const int64_t r = q / n;
    const int c = (int)(q - r * n);
    B[r * ld + c] = Yt[(r0 + r) * ld + c];
  }
}

// sparse: points [j0, j0 + np); observation o of point j puts Ysp[o][d][a] at row 3 (j - j0) + d,
// column 9 cam(o) + a.  One warp per point.
__global__ void cov_fill_sparse_kernel(const int64_t* __restrict__ obs_ptr, const int32_t* __restrict__ obs_cam,
                                       const double* __restrict__ Ysp, int ld, int64_t j0, int np,
                                       double* __restrict__ B) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t jj = warp; jj < np; jj += nwarps) {
    const int64_t lo = obs_ptr[j0 + jj], hi = obs_ptr[j0 + jj + 1];
    for (int64_t k = lo * 27 + lane; k < hi * 27; k += 32) {
      const int64_t o = k / 27;
      const int e = (int)(k - o * 27), d = e / 9, a = e - 9 * d;
      B[(3 * jj + d) * ld + 9 * (int64_t)obs_cam[o] + a] = Ysp[k];
    }
  }
}

// cameras: row r is the unit vector e_{c0 + r}
__global__ void cov_fill_unit_kernel(int n, int c0, int rows, int ld, double* __restrict__ B) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < rows && c0 + r < n) B[(int64_t)r * ld + c0 + r] = 1.0;
}

// ---- blocked forward substitution X = B L^-T ----------------------------------------------------
// One CTA per strip of 64 rows, left-looking over the 64-column blocks J of L:
//   acc = B[:, J] - sum_{K < J} X[:, K] L[J, K]^T,   X[:, J] = acc W_J,   W_J = L_JJ^-T
// L[J, K] (K < J) is read where the factorisation left it (the rows below each diagonal block of S)
// and W_J from Winv; the diagonal blocks of S are not the factor and are never read.  X[:, K] goes
// back to the batch in place and is read again (L2) for the later blocks of the same strip.  Both
// products run on DMMA.8x8x4: 8 warps, warp w owns rows 16 (w / 2) .. +15 and columns 32 (w % 2) .. +31
// of the 64 x 64 block.  The operands are staged row-major (k contiguous, rows padded to 68 doubles:
// conflict-free fragment loads) by cp.async, two stages.  Fixed summation order: bit-reproducible.
// first_col >= 0 (camera pass): row r of the batch is e_{first_col + r}, so X[r][c] = 0 for
// c < first_col + r and the blocks before the strip's first unit column are skipped (they stay zero).
constexpr int kCovThreads = 256;
constexpr size_t kCovSmem = 6 * (size_t)kCovTile * sizeof(double);  // 2 x (X, L) stages, rhs, W: 204 KB

__device__ __forceinline__ void cov_stage_tile(double* dst, const double* src, int64_t ld, int valid_rows,
                                               int valid_cols) {
  // 64 rows x 32 chunks of 16 B; rows >= valid_rows and chunks starting at >= valid_cols read as zero
  for (int q = threadIdx.x; q < kCovStrip * 32; q += kCovThreads) {
    const int r = q >> 5, ch = q & 31;
    const bool ok = r < valid_rows && 2 * ch < valid_cols;
    cp_async16_zfill(dst + r * kCovLd + 2 * ch, ok ? src + (int64_t)r * ld + 2 * ch : src, ok ? 16 : 0);
  }
}

// acc[i][j] += sum_k A[row0 + 8 i][k] Bt[col0 + 8 j][k] over 64 k (both row-major, k contiguous)
__device__ __forceinline__ void cov_tile_product(const double* __restrict__ A, const double* __restrict__ Bt,
                                                 int row0, int col0, int kq, double (&acc)[2][4][2]) {
#pragma unroll 4
  for (int kk = 0; kk < kCholNB; kk += 4) {
    double fa[2], fb[4];
#pragma unroll
    for (int i = 0; i < 2; ++i) fa[i] = A[(row0 + 8 * i) * kCovLd + kk + kq];
#pragma unroll
    for (int j = 0; j < 4; ++j) fb[j] = Bt[(col0 + 8 * j) * kCovLd + kk + kq];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
  }
}

__global__ void __launch_bounds__(kCovThreads, 1)
cov_trsm_kernel(double* __restrict__ B, int ld, int n, const double* __restrict__ S, int lds,
                const double* __restrict__ Winv, int first_col) {
  extern __shared__ double csm[];
  double* const sX = csm;                  // [2] stages of X[:, K]
  double* const sL = csm + 2 * kCovTile;   // [2] stages of L[J, K]
  double* sR = csm + 4 * kCovTile;  // rhs block, then acc
  double* sW = csm + 5 * kCovTile;  // W_J, row-major [c][j]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rb = warp >> 1, ch = warp & 1;
  const int row0 = rb * 16 + (lane >> 2), col0 = ch * 32 + (lane >> 2), kq = lane & 3;
  double* Bs = B + (int64_t)blockIdx.x * kCovStrip * ld;
  const int nblk = (n + kCholNB - 1) / kCholNB;
  const int jb0 = first_col >= 0 ? (first_col + (int)blockIdx.x * kCovStrip) / kCholNB : 0;
  for (int J = jb0; J < nblk; ++J) {
    const int c0 = J * kCholNB;
    const int nbJ = n - c0 < kCholNB ? n - c0 : kCholNB;
    // rhs block and W_J travel with the first stage
    cov_stage_tile(sR, Bs + c0, ld, kCovStrip, nbJ);
    for (int q = threadIdx.x; q < kCovStrip * 32; q += kCovThreads) {
      const int r = q >> 5, c2 = q & 31;
      cp_async16_zfill(sW + r * kCovLd + 2 * c2, Winv + (size_t)J * kCholNB * kCholNB + r * kCholNB + 2 * c2, 16);
    }
    if (jb0 < J) {
      cov_stage_tile(sX, Bs + jb0 * kCholNB, ld, kCovStrip, kCholNB);
      cov_stage_tile(sL, S + (int64_t)c0 * lds + jb0 * kCholNB, lds, nbJ, kCholNB);
    }
    cp_async_commit();
    double acc[2][4][2] = {};
    for (int K = jb0; K < J; ++K) {
      const int st = (K - jb0) & 1;
      if (K + 1 < J) {  // next stage while this one is multiplied
        cov_stage_tile(sX + (st ^ 1) * kCovTile, Bs + (K + 1) * kCholNB, ld, kCovStrip, kCholNB);
        cov_stage_tile(sL + (st ^ 1) * kCovTile, S + (int64_t)c0 * lds + (K + 1) * kCholNB, lds, nbJ, kCholNB);
      }
      cp_async_commit();
      cp_async_wait<1>();
      __syncthreads();
      cov_tile_product(sX + st * kCovTile, sL + st * kCovTile, row0, col0, kq, acc);
      __syncthreads();
    }
    cp_async_wait<0>();
    __syncthreads();
    // acc = B[:, J] - X[:, <J] L[J, <J]^T, in place over the rhs block (every entry has one owner)
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        double* p = sR + (row0 + 8 * i) * kCovLd + 2 * kq + 8 * j + ch * 32;
        p[0] -= acc[i][j][0];
        p[1] -= acc[i][j][1];
      }
    __syncthreads();
    // X[:, J] = acc W_J; the B operand is read straight from W's rows (b = W[k][col])
    double x[2][4][2] = {};
#pragma unroll 4
    for (int kk = 0; kk < kCholNB; kk += 4) {
      double fa[2], fb[4];
#pragma unroll
      for (int i = 0; i < 2; ++i) fa[i] = sR[(row0 + 8 * i) * kCovLd + kk + kq];
#pragma unroll
      for (int j = 0; j < 4; ++j) fb[j] = sW[(kk + kq) * kCovLd + col0 + 8 * j];
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma884(x[i][j][0], x[i][j][1], fa[i], fb[j]);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = ch * 32 + 8 * j + 2 * kq;  // column inside the block
        double* dst = Bs + (int64_t)(row0 + 8 * i) * ld + c0 + c;
        if (c < nbJ) dst[0] = x[i][j][0];
        if (c + 1 < nbJ) dst[1] = x[i][j][1];
      }
    // the stores must land before the next block stages them (cp.async reads L2) and before the
    // shared buffers are refilled
    __threadfence_block();
    __syncthreads();
  }
}

// ---- Gram matrices of row groups --------------------------------------------------------------
// One warp per group of G consecutive rows: Gram[d][e] = sum_k X[d][k] X[e][k], lane l summing
// k = k_lo + l + 32 t, then a fixed shuffle tree.  G == 3: point j = j0 + group, out = scale *
// m^T (I + Q) m with m = L_j^-1 from LINV; G == 9: camera i = i0 + group, out = scale * Q with the
// gauge-pinned rows and columns zero.
template <int G>
__global__ void __launch_bounds__(256)
cov_gram_kernel(const double* __restrict__ X, int ld, int n, int groups, int64_t g0, int axis,
                const double* __restrict__ LINV, double scale, double* __restrict__ out) {
  constexpr int NP = G * (G + 1) / 2;
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t gi = warp; gi < groups; gi += nwarps) {
    const double* Xg = X + gi * G * ld;
    // camera rows are zero before their own unit column (forward substitution of e_c)
    const int k_lo = G == 9 ? (int)(9 * (g0 + gi)) & ~31 : 0;
    double acc[NP];
#pragma unroll
    for (int p = 0; p < NP; ++p) acc[p] = 0.0;
    for (int k = k_lo + lane; k < n; k += 32) {
      double v[G];
#pragma unroll
      for (int d = 0; d < G; ++d) v[d] = Xg[(int64_t)d * ld + k];
      int p = 0;
#pragma unroll
      for (int d = 0; d < G; ++d)
#pragma unroll
        for (int e = d; e < G; ++e, ++p) acc[p] = fma(v[d], v[e], acc[p]);
    }
#pragma unroll
    for (int p = 0; p < NP; ++p) acc[p] = warp_sum(acc[p]);
    if (lane != 0) continue;
    double Q[G][G];
    {
      int p = 0;
#pragma unroll
      for (int d = 0; d < G; ++d)
#pragma unroll
        for (int e = d; e < G; ++e) { Q[d][e] = acc[p]; Q[e][d] = acc[p]; ++p; }
    }
    if (G == 3) {
      const int64_t j = g0 + gi;
      const double* li = LINV + 6 * j;
      const double m[3][3] = {{li[0], 0.0, 0.0}, {li[1], li[2], 0.0}, {li[3], li[4], li[5]}};
      double T[3][3];  // (I + Q) m
#pragma unroll
      for (int d = 0; d < 3; ++d)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
          double s = m[d][b];
#pragma unroll
          for (int e = 0; e < 3; ++e) s = fma(Q[d][e], m[e][b], s);
          T[d][b] = s;
        }
      double* o = out + 9 * j;
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = a; b < 3; ++b) {  // upper triangle, mirrored: the block is exactly symmetric
          double s = 0.0;
#pragma unroll
          for (int d = 0; d < 3; ++d) s = fma(m[d][a], T[d][b], s);
          o[3 * a + b] = scale * s;
          o[3 * b + a] = scale * s;
        }
    } else {
      const int64_t i = g0 + gi;
      const uint32_t mask = gauge_mask((int)i, axis);
      double* o = out + 81 * i;
#pragma unroll
      for (int a = 0; a < G; ++a)
#pragma unroll
        for (int b = 0; b < G; ++b) o[G * a + b] = (((mask >> a) | (mask >> b)) & 1u) ? 0.0 : scale * Q[a][b];
    }
  }
}

// Rows per batch: the whole pass when it fits, else the budget rounded down to whole quanta.
static int64_t cov_batch_rows(int64_t rows, int ld) {
  const int64_t cap = (int64_t)(kCovBatchBytes / ((size_t)8 * ld)) / kCovBatchQuantum * kCovBatchQuantum;
  const int64_t whole = (rows + kCovStrip - 1) / kCovStrip * kCovStrip;
  const int64_t q = cap > kCovBatchQuantum ? cap : kCovBatchQuantum;
  return whole < q ? whole : q;
}

// One pass: `rows` right-hand-side rows in groups of G, batch by batch.
template <int G>
static int cov_pass(ba_engine* e, double* batch, int64_t batch_rows, double scale, double* out, cudaStream_t s) {
  const int n = e->n_full, ld = e->n_pad;
  const int64_t rows = G == 9 ? (int64_t)n : 3 * e->N;
  for (int64_t r0 = 0; r0 < rows; r0 += batch_rows) {
    const int nr = (int)(rows - r0 < batch_rows ? rows - r0 : batch_rows);
    const int strips = (nr + kCovStrip - 1) / kCovStrip;
    BA_CUDA(cudaMemsetAsync(batch, 0, (size_t)strips * kCovStrip * ld * sizeof(double), s));
    if (G == 9) {
      cov_fill_unit_kernel<<<(nr + 255) / 256, 256, 0, s>>>(n, (int)r0, nr, ld, batch);
    } else if (e->dense) {
      cov_fill_dense_kernel<<<e->num_sms * 8, 256, 0, s>>>(e->Yt, ld, n, r0, nr, batch);
    } else {
      cov_fill_sparse_kernel<<<balanced_blocks((nr / 3 + 7) / 8, (int64_t)e->num_sms * 16), 256, 0, s>>>(
          e->obs_ptr, e->obs_cam, e->Ysp, ld, r0 / 3, nr / 3, batch);
    }
    BA_LAUNCH_CHECK();
    cov_trsm_kernel<<<strips, kCovThreads, kCovSmem, s>>>(batch, ld, n, e->P(), ld, e->Winv, G == 9 ? (int)r0 : -1);
    BA_LAUNCH_CHECK();
    const int groups = nr / G;
    cov_gram_kernel<G><<<balanced_blocks((groups + 7) / 8, (int64_t)e->num_sms * 16), 256, 0, s>>>(
        batch, ld, n, groups, r0 / G, e->axis, e->LINV, scale, out);
    BA_LAUNCH_CHECK();
  }
  return BA_OK;
}

// The undamped system at the current state, factored; E into cost_buf[3] (the spare slot).
// Runs against a scratch control block so that the LM loop's own stays untouched.
static int cov_factor(ba_engine* e, cudaStream_t s) {
  BA_TRY(launch_cam_prep(e, 0, s));
  BA_TRY(launch_cost(e, 0, 3, s));
  BA_TRY(launch_k1(e, s, false));
  BA_TRY(launch_k2a(e, s, false));
  BA_TRY(launch_camera_blocks(e, s, false));
  BA_TRY(launch_k2b(e, false, 0.0, s));
  BA_TRY(launch_k3(e, false, s));
  BA_TRY(launch_assemble(e, false, 0.0, s));
  return launch_cholesky_solve(e, false, s);
}

int covariance(ba_engine* e, double* point_cov, double* cam_cov, double* sigma2, int mem, cudaStream_t s) {
  if (e->comm) {
    set_error("covariance of a sharded engine is not supported (the undamped system would need the exchange)");
    return BA_ERR_STATE;
  }
  const int64_t dof = 2 * e->nobs - (3 * e->N + 9 * (int64_t)e->M - 7);
  if (dof <= 0) {
    set_error("covariance needs more residuals than unknowns (2 n_obs = %lld, unknowns = %lld)",
              (long long)(2 * e->nobs), (long long)(3 * e->N + 9 * (int64_t)e->M - 7));
    return BA_ERR_INVALID;
  }
  if (!e->dense) {
    std::vector<int64_t> ptr((size_t)e->N + 1);
    BA_CUDA(cudaMemcpyAsync(ptr.data(), e->obs_ptr, ptr.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    BA_CUDA(cudaStreamSynchronize(s));
    for (int64_t j = 0; j < e->N; ++j)
      if (ptr[(size_t)j + 1] - ptr[(size_t)j] < 2) {
        set_error("point %lld has fewer than two views: its covariance is unbounded", (long long)j);
        return BA_ERR_SINGULAR;
      }
  }
  ba_lm_state* scratch = nullptr;
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&scratch), sizeof(ba_lm_state), s));
  BA_CUDA(cudaMemsetAsync(scratch, 0, sizeof(ba_lm_state), s));
  ba_lm_state* const lm_ctl = e->ctl;
  e->ctl = scratch;
  int st = cov_factor(e, s);
  e->ctl = lm_ctl;
  ba_lm_state ctl_h;
  double E = 0.0;
  if (st == BA_OK && (cudaMemcpyAsync(&ctl_h, scratch, sizeof(ctl_h), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
                      cudaMemcpyAsync(&E, e->cost_buf + 3, sizeof(double), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
                      cudaStreamSynchronize(s) != cudaSuccess)) {
    set_error("covariance: reading the factorisation status failed: %s", cudaGetErrorString(cudaGetLastError()));
    st = BA_ERR_CUDA;
  }
  cudaFreeAsync(scratch, s);
  if (st != BA_OK) return st;
  if (ctl_h.status != BA_OK || ctl_h.chol_fail) {
    set_error(ctl_h.status == BA_ERR_SINGULAR && !ctl_h.chol_fail
                  ? "a point block of the undamped system is not positive definite"
                  : "the undamped reduced camera system is not positive definite");
    return BA_ERR_SINGULAR;
  }
  const double s2 = E / (double)dof;
  if (sigma2) *sigma2 = s2;
  const double scale = 2.0 * s2;

  const bool dev = mem == BA_MEM_DEVICE;
  double *pc = nullptr, *cc = nullptr, *batch = nullptr;
  if (point_cov) {
    if (dev) pc = point_cov;
    else BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&pc), (size_t)9 * e->N * sizeof(double), s));
  }
  if (cam_cov) {
    if (dev) cc = cam_cov;
    else BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&cc), (size_t)81 * e->M * sizeof(double), s));
  }
  const int64_t want = point_cov ? (3 * e->N > e->n_full ? 3 * e->N : e->n_full) : e->n_full;
  const int64_t batch_rows = cov_batch_rows(want, e->n_pad);
  BA_CUDA(cudaFuncSetAttribute(cov_trsm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCovSmem));
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&batch), (size_t)batch_rows * e->n_pad * sizeof(double), s));
  if (cam_cov) st = cov_pass<9>(e, batch, batch_rows, scale, cc, s);
  if (st == BA_OK && point_cov) st = cov_pass<3>(e, batch, batch_rows, scale, pc, s);
  if (st == BA_OK && !dev) {
    if (point_cov && cudaMemcpyAsync(point_cov, pc, (size_t)9 * e->N * sizeof(double), cudaMemcpyDeviceToHost, s) != cudaSuccess)
      st = BA_ERR_CUDA;
    if (cam_cov && cudaMemcpyAsync(cam_cov, cc, (size_t)81 * e->M * sizeof(double), cudaMemcpyDeviceToHost, s) != cudaSuccess)
      st = BA_ERR_CUDA;
    if (st != BA_OK) set_error("covariance: copy to the host failed: %s", cudaGetErrorString(cudaGetLastError()));
  }
  cudaFreeAsync(batch, s);
  if (!dev) {
    if (pc) cudaFreeAsync(pc, s);
    if (cc) cudaFreeAsync(cc, s);
  }
  if (cudaStreamSynchronize(s) != cudaSuccess && st == BA_OK) {
    set_error("covariance failed: %s", cudaGetErrorString(cudaGetLastError()));
    st = BA_ERR_CUDA;
  }
  return st;
}

}  // namespace ba
