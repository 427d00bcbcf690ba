// K1: per-observation reprojection residuals and analytic Jacobians, plus the cost-only
// variant and the per-camera derived table they read.
//
// Replaces (reference lib/bundle_adjustment.py): _get_K :283-289, _calc_pqr :291-307,
// _calc_X_diff_pqr :309-322, _calc_f/u/t/R_diff_pqr :324-398, _calc_camera_params_diff_pqr
// :400-427, the residual terms of _calc_d_P/_calc_d_F :445,:454 and _calc_reprojection_error
// :666-677.  The reference tiles per-camera rows to (N, M, 3) arrays (:318-320, :368-376);
// here the per-camera values live in a 128-byte table row staged in shared memory and are
// never materialised per observation.
//
// Memory roofline (HBM): per observation 16 B read (x, y) [+8 B indices when sparse] and
// 64 B + 160 B written (the point-side and camera-side Jacobian rows, each carrying the
// residual so that the two consumers stream one row each).
//
// The row arithmetic itself is obs_jacobian / obs_residual / obs_cost in ba_common.cuh (one
// division per observation, every operation pinned), shared with the kernels that re-derive the
// rows: dense scenes are linearised matrix-free (k2_point_blocks.cu), K1 then only refreshes the
// camera table and writes the rows when somebody reads the JP / JC buffers.
#include "ba_common.cuh"

namespace ba {

// ---- per-camera derived table -----------------------------------------------------------
// row: gp(3) gq(3) gr(3) t(3) 1/f u0/f0 v0/f0 1/f0, with gp = f R[:,0] + u0 R[:,2] etc. = rows of
// K R^T (:283-302); p = gp . (X - t) reproduces P [X;1] with P[:, 3] = -K R^T t.
__global__ void cam_prep_kernel(int M, const double* __restrict__ f, const double* __restrict__ u,
                                const double* __restrict__ R, const double* __restrict__ t,
                                double f0, double* __restrict__ tab, const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const double fi = f[i], u0 = u[2 * i], v0 = u[2 * i + 1];
  const double* Ri = R + 9 * i;
  double* T = tab + (size_t)i * kCamTab;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double r0 = Ri[3 * k + 0], r1 = Ri[3 * k + 1], r2 = Ri[3 * k + 2];
    T[k] = fi * r0 + u0 * r2;
    T[3 + k] = fi * r1 + v0 * r2;
    T[6 + k] = f0 * r2;
    T[9 + k] = t[3 * i + k];
  }
  // per-camera quotients of the Jacobian formulas (:336-356), so that no kernel divides by them per
  // observation: 1 / f, u0 / f0, v0 / f0, 1 / f0
  T[12] = 1.0 / fi;
  T[13] = u0 / f0;
  T[14] = v0 / f0;
  T[15] = 1.0 / f0;
}

int launch_cam_prep(ba_engine* e, int which, cudaStream_t s) {
  const CamState& c = e->cam[which];
  cam_prep_kernel<<<(e->M + 127) / 128, 128, 0, s>>>(e->M, c.f, c.u, c.R, c.t, e->f0,
                                                      e->camtab[which], nullptr);
  BA_LAUNCH_CHECK();
  return BA_OK;
}

// (kTabStride / tab_smem_doubles: the padded shared-memory camera table, see ba_common.cuh; at the
// table's own stride of 16 doubles ncu counted 8.7 bank conflicts per observation.)
constexpr int kK1Stage = 32 * 8 + 32 * 21;  // staging doubles per warp: point rows, camera rows

// ---- K1 -------------------------------------------------------------------------------------
template <bool DENSE, bool SMEM_TAB>
__global__ void __launch_bounds__(256)
k1_residual_jacobian_kernel(int64_t nobs, int M, const int32_t* __restrict__ obs_cam,
                            const int32_t* __restrict__ obs_pt, const double2* __restrict__ xy,
                            const double* __restrict__ X, const double* __restrict__ camtab,
                            double f0, double* __restrict__ JP, double* __restrict__ JC,
                            double* __restrict__ cost_part, const ba_lm_state* ctl) {
  if (ctl && (ctl->done || !ctl->need_linearize)) return;
  extern __shared__ double2 s_tab2[];
  const double* tab = camtab;
  constexpr int TS = SMEM_TAB ? kTabStride : kCamTab;  // row stride of the table being read
  if (SMEM_TAB) {
    double* dst = reinterpret_cast<double*>(s_tab2);
    for (int k = threadIdx.x; k < M * kCamTab; k += blockDim.x) dst[(k >> 4) * kTabStride + (k & 15)] = camtab[k];
    __syncthreads();
    tab = dst;
  }
  __shared__ double scratch[32];
  // per-warp staging of the 32 x (8 + 20) output doubles, so the Jacobian rows leave the SM as
  // whole contiguous runs instead of per-lane 16-byte pieces.  Point rows: [32][8] with the column
  // XOR-swizzled by (lane >> 1) & 7 -- lanes write one column at a time (16 distinct bank pairs per
  // half-warp) and the read-out walks consecutive addresses.  Camera rows: [32][21] (odd stride).
  // (The first version used one [32][29] array: ncu counted 8.7 bank conflicts per observation.)
  const int lane = threadIdx.x & 31;
  const int swz = (lane >> 1) & 7;
  double* st = reinterpret_cast<double*>(s_tab2) + (SMEM_TAB ? tab_smem_doubles(M) : 0) +
               (size_t)(threadIdx.x >> 5) * kK1Stage;

  // contiguous slab of observations per block, 256 at a time (coalesced xy reads)
  const int64_t per = (nobs + gridDim.x - 1) / gridDim.x;
  const int64_t lo = per * blockIdx.x;
  const int64_t hi = lo + per < nobs ? lo + per : nobs;
  double acc = 0.0;
  for (int64_t o0 = lo + (threadIdx.x & ~31); o0 < hi; o0 += blockDim.x) {
    const int64_t o = o0 + lane;
    const int cnt = (int)(hi - o0 < 32 ? hi - o0 : 32);
    if (o < hi) {
    int i, j;
    if (DENSE) {
      j = (int)(o / M);
      i = (int)(o - (int64_t)j * M);
    } else {
      i = obs_cam[o];
      j = obs_pt[o];
    }
    ObsJacobian J;
    obs_jacobian(tab + (size_t)i * TS, X[3 * (size_t)j + 0], X[3 * (size_t)j + 1], X[3 * (size_t)j + 2], J);
    const double2 m = xy[o];
    double e0, e1;
    obs_residual(J, m.x, m.y, e0, e1);  // :445, :454
    acc += fma(e1, e1, __dmul_rn(e0, e0));

    double* wp = st + lane * 8;
    wp[0 ^ swz] = e0; wp[1 ^ swz] = e1;
    wp[2 ^ swz] = J.ax[0]; wp[3 ^ swz] = J.ax[1]; wp[4 ^ swz] = J.ax[2];
    wp[5 ^ swz] = J.bx[0]; wp[6 ^ swz] = J.bx[1]; wp[7 ^ swz] = J.bx[2];
    // camera row: e, then the nine entries of row a and of row b
    double* w = st + 256 + lane * 21;
    w[0] = e0; w[1] = e1;
#pragma unroll
    for (int a = 0; a < 9; ++a) {
      w[2 + a] = J.ja[a];
      w[11 + a] = J.jb[a];
    }
    }
    __syncwarp();
    {
      double* dp = JP + (size_t)o0 * kJP;
      for (int k = lane; k < kJP * cnt; k += 32) {
        const int row = k >> 3;
        dp[k] = st[row * 8 + ((k & 7) ^ ((row >> 1) & 7))];
      }
      double* dc = JC + (size_t)o0 * kJC;
      for (int k = lane; k < kJC * cnt; k += 32) {
        const int row = k / kJC;
        dc[k] = st[256 + row * 21 + (k - row * kJC)];
      }
    }
    __syncwarp();
  }
  const double tot = block_sum(acc, scratch);
  if (threadIdx.x == 0) cost_part[blockIdx.x] = tot;
}

// ---- cost only (:666-677) ---------------------------------------------------------------------
template <bool DENSE, bool SMEM_TAB>
__global__ void __launch_bounds__(256)
cost_kernel(int64_t nobs, int M, const int32_t* __restrict__ obs_cam,
            const int32_t* __restrict__ obs_pt, const double2* __restrict__ xy,
            const double* __restrict__ X, const double* __restrict__ camtab, double f0,
            double* __restrict__ cost_part, const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;
  extern __shared__ double2 s_tab2[];
  const double* tab = camtab;
  constexpr int TS = SMEM_TAB ? kTabStride : kCamTab;
  if (SMEM_TAB) {
    double* dst = reinterpret_cast<double*>(s_tab2);
    for (int k = threadIdx.x; k < M * kCamTab; k += blockDim.x) dst[(k >> 4) * kTabStride + (k & 15)] = camtab[k];
    __syncthreads();
    tab = dst;
  }
  __shared__ double scratch[32];
  const int64_t per = (nobs + gridDim.x - 1) / gridDim.x;
  const int64_t lo = per * blockIdx.x;
  const int64_t hi = lo + per < nobs ? lo + per : nobs;
  double acc = 0.0;
  for (int64_t o = lo + threadIdx.x; o < hi; o += blockDim.x) {
    int i, j;
    if (DENSE) {
      j = (int)(o / M);
      i = (int)(o - (int64_t)j * M);
    } else {
      i = obs_cam[o];
      j = obs_pt[o];
    }
    const double2 m = xy[o];
    acc += obs_cost(tab + (size_t)i * TS, X[3 * (size_t)j + 0], X[3 * (size_t)j + 1], X[3 * (size_t)j + 2], m.x, m.y);
  }
  const double tot = block_sum(acc, scratch);
  if (threadIdx.x == 0) cost_part[blockIdx.x] = tot;
}

// Fixed-order final sum of the per-block partials into cost_buf[slot].
__global__ void cost_finish_kernel(const double* __restrict__ part, int n, double* out,
                                   const ba_lm_state* ctl, int lin_only) {
  if (ctl && (ctl->done || (lin_only && !ctl->need_linearize))) return;
  __shared__ double scratch[32];
  double acc = 0.0;
  for (int k = threadIdx.x; k < n; k += blockDim.x) acc += part[k];
  const double tot = block_sum(acc, scratch);
  if (threadIdx.x == 0) *out = tot;
}

// The camera table is staged in shared memory whenever it fits next to K1's output staging.
// (Reading a large table -- C4: 1000 cameras, 136 KB -- through L1 instead, to keep three blocks
// per SM resident, was measured and is no faster: K1 7.9 vs 8.1 ms, cost kernel 1.48 vs 1.12 ms.)
static inline size_t tab_smem_bytes(const ba_engine* e) {
  const size_t bytes = tab_smem_doubles(e->M) * sizeof(double);
  return bytes <= 160 * 1024 ? bytes : 0;
}

int launch_cost(ba_engine* e, int which, int slot, cudaStream_t s) {
  const size_t smem = tab_smem_bytes(e);
  const double2* xy = reinterpret_cast<const double2*>(e->obs_xy);
  const int grid = e->cost_blocks;
  // the 48 KB default limit counts the static block_sum scratch too: at 360 and 361 cameras the table
  // alone fits under it, table and scratch do not
#define BA_COST_LAUNCH(D, T)                                                                   \
  do {                                                                                         \
    if (smem + 32 * sizeof(double) > 48 * 1024)                                                \
      BA_CUDA(cudaFuncSetAttribute(cost_kernel<D, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                   (int)smem));                                                \
    cost_kernel<D, T><<<grid, 256, smem, s>>>(e->nobs, e->M, e->obs_cam, e->obs_pt, xy,        \
                                              e->X[which], e->camtab[which], e->f0,            \
                                              e->cost_part, nullptr);                          \
  } while (0)
  if (e->dense) {
    if (smem) BA_COST_LAUNCH(true, true); else BA_COST_LAUNCH(true, false);
  } else {
    if (smem) BA_COST_LAUNCH(false, true); else BA_COST_LAUNCH(false, false);
  }
#undef BA_COST_LAUNCH
  BA_LAUNCH_CHECK();
  cost_finish_kernel<<<1, 256, 0, s>>>(e->cost_part, grid, e->cost_buf + slot, nullptr, 0);
  BA_LAUNCH_CHECK();
  return BA_OK;
}

// Dense matrix-free scenes (dense_matrix_free) never read JP / JC back -- K2a, the camera blocks,
// K2b and the point update re-derive the rows -- so only the camera table is refreshed; `force_rows`
// writes them all the same (ba_buffer_read of JP / JC: tests, diagnostics).
int launch_k1(ba_engine* e, cudaStream_t s, bool conditional, bool force_rows) {
  const size_t tab_bytes = tab_smem_bytes(e);
  const size_t smem = tab_bytes + 8 * kK1Stage * sizeof(double);
  const double2* xy = reinterpret_cast<const double2*>(e->obs_xy);
  const int grid = e->cost_blocks;
  const ba_lm_state* ctl = conditional ? e->ctl : nullptr;
  // the table of the *current* state must be fresh
  {
    const CamState& c = e->cam[0];
    cam_prep_kernel<<<(e->M + 127) / 128, 128, 0, s>>>(e->M, c.f, c.u, c.R, c.t, e->f0,
                                                        e->camtab[0], ctl);
    BA_LAUNCH_CHECK();
  }
  if (dense_matrix_free(e) && !force_rows) return BA_OK;
#define BA_K1_LAUNCH(D, T)                                                                     \
  do {                                                                                         \
    if (smem > 48 * 1024)                                                                      \
      BA_CUDA(cudaFuncSetAttribute(k1_residual_jacobian_kernel<D, T>,                          \
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   \
    k1_residual_jacobian_kernel<D, T><<<grid, 256, smem, s>>>(                                 \
        e->nobs, e->M, e->obs_cam, e->obs_pt, xy, e->X[0], e->camtab[0], e->f0, e->JP, e->JC,  \
        e->cost_part, ctl);                                                                    \
  } while (0)
  if (e->dense) {
    if (tab_bytes) BA_K1_LAUNCH(true, true); else BA_K1_LAUNCH(true, false);
  } else {
    if (tab_bytes) BA_K1_LAUNCH(false, true); else BA_K1_LAUNCH(false, false);
  }
#undef BA_K1_LAUNCH
  BA_LAUNCH_CHECK();
  return BA_OK;
}

}  // namespace ba
