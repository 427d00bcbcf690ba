// K2: per-point and per-camera Gauss-Newton blocks.
//
//   k2a  V_j = 2 sum_i Jx^T Jx (matE, reference :519-556), g_j = 2 sum_i Jx^T e (d_P, :429-469)
//        -- one warp per point, warp-level reductions, once per linearisation.
//   cam  U_i = 2 sum_j Jc^T Jc (diagonal blocks of matG, :618-653), dF_i = 2 sum_j Jc^T e (d_F,
//        :471-509) -- segmented reduction over the camera-major order, fixed summation order.
//   k2b  per inner solve: damp V_j (:120-122), Cholesky V_j(1+c) = L L^T instead of the
//        reference's general inverse (:128), z_j = L^-1 g_j and
//        Y_ij = W_ij^T L^-T  with W_ij = 2 Jx^T Jc (matF block, :598-605), so that
//        sum_j F_j^T E_j^-1 F_j = sum_j Y_j Y_j^T (:132-135) becomes a SYRK (K3) and
//        sum_j F_j^T E_j^-1 d_P_j = sum_j Y_j z_j (:143) rides along as one extra column.
//
// Gauge: the 7 removed unknowns (:62-72) are pinned instead of deleted -- their Jc columns are
// masked here, so the corresponding rows/columns of the reduced system vanish and K4 puts a
// unit diagonal there (delta = 0, algebraically identical to deletion).
//
// Memory roofline (HBM), stored-row form (sparse scenes): k2a reads 64 B/obs; cam reads 160 B/obs;
// k2b reads 64+160 B/obs and writes 216 B/obs (Y).
//
// Matrix-free form (template flag MF; dense scenes whose camera table fits 48 KB of shared memory,
// dense_matrix_free): the three kernels re-derive the Jacobian rows with obs_jacobian (ba_common.cuh)
// from the camera table, X_j and the observed point instead of reading what K1 stored -- the same
// pinned arithmetic, the same summation orders, hence the same bits; K1 then stores nothing, k2a and
// cam read 16 B/obs, k2b only writes its 216 B/obs.
#include "ba_common.cuh"

namespace ba {

// ---- k2a --------------------------------------------------------------------------------------
// MF (dense_matrix_free): the point-side rows and the residual are re-derived from the camera table
// (shared memory), X_j and the observed points instead of being read from JP -- K1 then has nothing
// to store; same arithmetic (obs_jacobian, K1's residual expression), same order: the same V, d_P.
template <bool DENSE, bool MF>
__global__ void __launch_bounds__(256)
k2a_point_blocks_kernel(int64_t N, int M, const int64_t* __restrict__ obs_ptr,
                        const double* __restrict__ JP, double* __restrict__ V,
                        double* __restrict__ GPT, const ba_lm_state* ctl,
                        const double* __restrict__ camtab, const double* __restrict__ X,
                        const double2* __restrict__ xy, double f0) {
  static_assert(DENSE || !MF, "the matrix-free variant is the dense one");
  if (ctl && (ctl->done || !ctl->need_linearize)) return;
  extern __shared__ double k2a_tab[];
  if (MF) {
    for (int k = threadIdx.x; k < M * kCamTab; k += blockDim.x) k2a_tab[(k >> 4) * kTabStride + (k & 15)] = camtab[k];
    __syncthreads();
  }
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t j = warp; j < N; j += nwarps) {
    const int64_t lo = DENSE ? j * M : obs_ptr[j];
    const int64_t hi = DENSE ? lo + M : obs_ptr[j + 1];
    double vxx = 0, vxy = 0, vxz = 0, vyy = 0, vyz = 0, vzz = 0, g0 = 0, g1 = 0, g2 = 0;
    const double xj0 = MF ? X[3 * (size_t)j] : 0.0, xj1 = MF ? X[3 * (size_t)j + 1] : 0.0,
                 xj2 = MF ? X[3 * (size_t)j + 2] : 0.0;
    for (int64_t o = lo + lane; o < hi; o += 32) {
      double e0, e1, a0, a1, a2, b0, b1, b2;
      if (MF) {
        ObsJacobian J;
        obs_jacobian(k2a_tab + (size_t)(o - lo) * kTabStride, xj0, xj1, xj2, J);
        const double2 m = xy[o];
        obs_residual(J, m.x, m.y, e0, e1);  // :445, :454, as K1
        a0 = J.ax[0]; a1 = J.ax[1]; a2 = J.ax[2];
        b0 = J.bx[0]; b1 = J.bx[1]; b2 = J.bx[2];
      } else {
        const double2* row = reinterpret_cast<const double2*>(JP + (size_t)o * kJP);
        const double2 r0 = row[0], r1 = row[1], r2 = row[2], r3 = row[3];
        e0 = r0.x; e1 = r0.y;
        a0 = r1.x; a1 = r1.y; a2 = r2.x; b0 = r2.y; b1 = r3.x; b2 = r3.y;
      }
      vxx = pair_accumulate(vxx, a0, a0, b0, b0);
      vxy = pair_accumulate(vxy, a0, a1, b0, b1);
      vxz = pair_accumulate(vxz, a0, a2, b0, b2);
      vyy = pair_accumulate(vyy, a1, a1, b1, b1);
      vyz = pair_accumulate(vyz, a1, a2, b1, b2);
      vzz = pair_accumulate(vzz, a2, a2, b2, b2);
      g0 = pair_accumulate(g0, e0, a0, e1, b0);
      g1 = pair_accumulate(g1, e0, a1, e1, b1);
      g2 = pair_accumulate(g2, e0, a2, e1, b2);
    }
    vxx = warp_sum(vxx); vxy = warp_sum(vxy); vxz = warp_sum(vxz);
    vyy = warp_sum(vyy); vyz = warp_sum(vyz); vzz = warp_sum(vzz);
    g0 = warp_sum(g0); g1 = warp_sum(g1); g2 = warp_sum(g2);
    if (lane == 0) {
      double* v = V + 6 * (size_t)j;
      v[0] = 2.0 * vxx; v[1] = 2.0 * vxy; v[2] = 2.0 * vxz;
      v[3] = 2.0 * vyy; v[4] = 2.0 * vyz; v[5] = 2.0 * vzz;
      double* g = GPT + 3 * (size_t)j;
      g[0] = 2.0 * g0; g[1] = 2.0 * g1; g[2] = 2.0 * g2;
    }
  }
}

int launch_k2a(ba_engine* e, cudaStream_t s, bool conditional) {
  const ba_lm_state* ctl = conditional ? e->ctl : nullptr;
  const int grid = balanced_blocks((e->N + 7) / 8, (int64_t)e->num_sms * 16);  // 8 warps per block
  const double2* xy = reinterpret_cast<const double2*>(e->obs_xy);
  if (dense_matrix_free(e))
    k2a_point_blocks_kernel<true, true><<<grid, 256, tab_smem_doubles(e->M) * sizeof(double), s>>>(
        e->N, e->M, e->obs_ptr, e->JP, e->V, e->GPT, ctl, e->camtab[0], e->X[0], xy, e->f0);
  else if (e->dense)
    k2a_point_blocks_kernel<true, false><<<grid, 256, 0, s>>>(e->N, e->M, e->obs_ptr, e->JP, e->V, e->GPT, ctl,
                                                              e->camtab[0], e->X[0], xy, e->f0);
  else
    k2a_point_blocks_kernel<false, false><<<grid, 256, 0, s>>>(e->N, e->M, e->obs_ptr, e->JP, e->V, e->GPT, ctl,
                                                               e->camtab[0], e->X[0], xy, e->f0);
  BA_LAUNCH_CHECK();
  return BA_OK;
}

// ---- camera blocks ----------------------------------------------------------------------------
// grid (chunks, M); block (i, c) reduces chunk c of camera i's observations into 54 numbers.
// MF (dense_matrix_free): the camera-side rows and the residual are re-derived (the block's camera
// table row in registers, X_q and the observed point read per observation: 40 B instead of 160 B).
template <bool DENSE, bool MF>
__global__ void __launch_bounds__(128, MF ? 3 : 1)
camera_blocks_kernel(int64_t N, int M, const int64_t* __restrict__ cam_ptr,
                     const int32_t* __restrict__ cm_perm, const double* __restrict__ JC,
                     double* __restrict__ Upart, const ba_lm_state* ctl,
                     const double* __restrict__ camtab, const double* __restrict__ X,
                     const double2* __restrict__ xy, double f0) {
  static_assert(DENSE || !MF, "the matrix-free variant is the dense one");
  if (ctl && (ctl->done || !ctl->need_linearize)) return;
  const int i = blockIdx.y;
  double T[kCamTab];
  if (MF) {
#pragma unroll
    for (int k = 0; k < kCamTab; ++k) T[k] = camtab[(size_t)i * kCamTab + k];
  }
  const int chunk = blockIdx.x, nchunks = gridDim.x;
  const int64_t seg_lo = DENSE ? 0 : cam_ptr[i];
  const int64_t seg_n = DENSE ? N : cam_ptr[i + 1] - seg_lo;
  const int64_t per = (seg_n + nchunks - 1) / nchunks;
  const int64_t lo = per * chunk;
  const int64_t hi = lo + per < seg_n ? lo + per : seg_n;

  double acc[kUPart];
#pragma unroll
  for (int k = 0; k < kUPart; ++k) acc[k] = 0.0;
  for (int64_t q = lo + threadIdx.x; q < hi; q += blockDim.x) {
    const int64_t o = DENSE ? q * M + i : (int64_t)cm_perm[seg_lo + q];
    double v[kJC];
    if (MF) {
      ObsJacobian J;
      obs_jacobian(T, X[3 * (size_t)q], X[3 * (size_t)q + 1], X[3 * (size_t)q + 2], J);
      const double2 m = xy[o];
      obs_residual(J, m.x, m.y, v[0], v[1]);  // :445, :454, as K1
#pragma unroll
      for (int k = 0; k < 9; ++k) {
        v[2 + k] = J.ja[k];
        v[11 + k] = J.jb[k];
      }
    } else {
      const double2* row = reinterpret_cast<const double2*>(JC + (size_t)o * kJC);
#pragma unroll
      for (int k = 0; k < kJC / 2; ++k) {
        const double2 t2 = row[k];
        v[2 * k] = t2.x;
        v[2 * k + 1] = t2.y;
      }
    }
    const double e0 = v[0], e1 = v[1];
    const double* a = v + 2;
    const double* b = v + 11;
    int idx = 0;
#pragma unroll
    for (int r = 0; r < 9; ++r)
#pragma unroll
      for (int c = r; c < 9; ++c, ++idx) acc[idx] = pair_accumulate(acc[idx], a[r], a[c], b[r], b[c]);
#pragma unroll
    for (int r = 0; r < 9; ++r) acc[45 + r] = pair_accumulate(acc[45 + r], e0, a[r], e1, b[r]);
  }
  // block reduction, fixed order: lanes by xor-tree, then warps 0..3 in sequence
  __shared__ double sred[4][kUPart];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < kUPart; ++k) {
    const double s = warp_sum(acc[k]);
    if (lane == 0) sred[warp][k] = s;
  }
  __syncthreads();
  if (threadIdx.x < kUPart) {
    const double s = ((sred[0][threadIdx.x] + sred[1][threadIdx.x]) + sred[2][threadIdx.x]) +
                     sred[3][threadIdx.x];
    Upart[((size_t)i * nchunks + chunk) * kUPart + threadIdx.x] = s;
  }
}

// Sum the chunks in order, expand to the full symmetric 9x9, apply factor 2 and the gauge mask.
__global__ void camera_blocks_finish_kernel(int M, int nchunks, int axis,
                                            const double* __restrict__ Upart,
                                            double* __restrict__ U, double* __restrict__ GCAM,
                                            const ba_lm_state* ctl) {
  if (ctl && (ctl->done || !ctl->need_linearize)) return;
  const int i = blockIdx.x;
  const int k = threadIdx.x;  // 0..89: 81 entries of U, 9 of dF
  if (k >= 90) return;
  const uint32_t mask = gauge_mask(i, axis);
  int src;
  bool pinned;
  if (k < 81) {
    int r = k / 9, c = k % 9;
    pinned = ((mask >> r) & 1u) || ((mask >> c) & 1u);
    if (r > c) { int t = r; r = c; c = t; }
    src = r * 9 - r * (r - 1) / 2 + (c - r);  // index in the packed upper triangle
  } else {
    pinned = (mask >> (k - 81)) & 1u;
    src = 45 + (k - 81);
  }
  double s = 0.0;
  for (int ch = 0; ch < nchunks; ++ch) s += Upart[((size_t)i * nchunks + ch) * kUPart + src];
  s = pinned ? 0.0 : 2.0 * s;
  if (k < 81) U[(size_t)i * 81 + k] = s;
  else GCAM[(size_t)i * 9 + (k - 81)] = s;
}

int launch_camera_blocks(ba_engine* e, cudaStream_t s, bool conditional) {
  const ba_lm_state* ctl = conditional ? e->ctl : nullptr;
  dim3 grid(e->cam_chunks, e->M);
  const double2* xy = reinterpret_cast<const double2*>(e->obs_xy);
  if (dense_matrix_free(e))
    camera_blocks_kernel<true, true><<<grid, 128, 0, s>>>(e->N, e->M, e->cam_ptr, e->cm_perm, e->JC, e->Upart, ctl,
                                                          e->camtab[0], e->X[0], xy, e->f0);
  else if (e->dense)
    camera_blocks_kernel<true, false><<<grid, 128, 0, s>>>(e->N, e->M, e->cam_ptr, e->cm_perm, e->JC, e->Upart, ctl,
                                                           e->camtab[0], e->X[0], xy, e->f0);
  else
    camera_blocks_kernel<false, false><<<grid, 128, 0, s>>>(e->N, e->M, e->cam_ptr, e->cm_perm, e->JC, e->Upart, ctl,
                                                            e->camtab[0], e->X[0], xy, e->f0);
  BA_LAUNCH_CHECK();
  camera_blocks_finish_kernel<<<e->M, 96, 0, s>>>(e->M, e->cam_chunks, e->axis, e->Upart, e->Uloc,
                                                   e->Uloc + (size_t)e->M * 81, ctl);
  BA_LAUNCH_CHECK();
  return BA_OK;
}

// ---- k2b --------------------------------------------------------------------------------------
// One warp per point.  Dense layout of Y: Yt[(3j+d) * ld + 9i + a] (k-major operand of the
// SYRK) with z_j in column rhs_col; sparse layout: Ysp[o][d][a].
// MF (dense scenes, camera table small enough for shared memory): matrix-free -- the Jacobian rows
// are re-derived from the camera table and X_j (obs_jacobian, the arithmetic K1 stored them with:
// the same bits) instead of being read back, 224 B per observation; the kernel then only writes.
//
// colmax (dense, when K3 runs on the INT8 emulation; nullptr otherwise): the column maxima of |Yt| that
// set the emulation's column exponents, gathered as Yt is written.  Only ilogb of a maximum is used,
// and for a normal double that is its exponent field: a CTA keeps the largest top 16 bits (exponent and
// four mantissa bits) of every column in shared memory (2 bytes per column: room for the stored-row
// kernel's three CTAs per SM up to n_pad 10 752, for the matrix-free one's two at every M it takes),
// then raises colmax[a] to them << 48 with one atomicMax per column.  A subnormal entry (exponent field
// 0) goes straight to colmax with its full bit pattern, so ilogb of colmax[a] is that of max |Yt[k][a]|
// in every case, and an all-zero column keeps 0.
__device__ __forceinline__ unsigned colmax_top16(double y, unsigned long long* __restrict__ colmax, int col) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(y) & 0x7FFFFFFFFFFFFFFFull;
  if (u != 0 && u < (1ull << 52)) atomicMax(colmax + col, u);  // subnormal: rare
  return (unsigned)(u >> 48);
}
__device__ __forceinline__ void colmax_smem_max(unsigned short* cm, int col, unsigned v) {
  unsigned short old = *reinterpret_cast<volatile unsigned short*>(cm + col);
  while (v > old) {  // the maximum rarely grows after a CTA's first points: mostly one load
    const unsigned short prev = atomicCAS(cm + col, old, (unsigned short)v);
    if (prev == old) break;
    old = prev;
  }
}

template <bool DENSE, bool MF>
__global__ void __launch_bounds__(256, MF ? 2 : 3)
k2b_point_solve_kernel(int64_t N, int M, int axis, const int64_t* __restrict__ obs_ptr,
                       const int32_t* __restrict__ obs_cam, const double* __restrict__ JP,
                       const double* __restrict__ JC, const double* __restrict__ V,
                       const double* __restrict__ GPT, double c_host, ba_lm_state* ctl,
                       int use_ctl, double* __restrict__ LINV, double* __restrict__ Z,
                       double* __restrict__ Yt, int ld, int rhs_col, double* __restrict__ Ysp,
                       const double* __restrict__ X, double* __restrict__ PT,
                       const double* __restrict__ camtab, double f0, unsigned long long* __restrict__ colmax) {
  static_assert(DENSE || !MF, "the matrix-free variant is the dense one");
  if (use_ctl && ctl->done) return;
  const double c = use_ctl ? ctl->c : c_host;
  const double damp = 1.0 + c;
  const int lane = threadIdx.x & 31;
  extern __shared__ double k2b_stage[];
  double* tab = k2b_stage;  // MF: the camera table, rows padded to kTabStride
  double* st0 = k2b_stage + (MF ? tab_smem_doubles(M) : 0);
  unsigned short* cm = reinterpret_cast<unsigned short*>(st0 + 8 * 864);  // colmax: [ld] top 16 bits
  if (DENSE && colmax)
    for (int k = threadIdx.x; k < ld; k += blockDim.x) cm[k] = 0;
  if (MF)
    for (int k = threadIdx.x; k < M * kCamTab; k += blockDim.x) tab[(k >> 4) * kTabStride + (k & 15)] = camtab[k];
  if (MF || (DENSE && colmax)) __syncthreads();
  double* st = st0 + (threadIdx.x >> 5) * 864;  // 32 observations x 27 doubles per warp
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t j = warp; j < N; j += nwarps) {
    const double* v = V + 6 * (size_t)j;
    // damped block (:120-122) and its Cholesky factor
    const double vxx = v[0] * damp, vxy = v[1], vxz = v[2], vyy = v[3] * damp, vyz = v[4],
                 vzz = v[5] * damp;
    const double l00 = sqrt(vxx);
    const double l10 = vxy / l00, l20 = vxz / l00;
    const double d11 = vyy - l10 * l10;
    const double l11 = sqrt(d11);
    const double l21 = (vyz - l20 * l10) / l11;
    const double d22 = vzz - l20 * l20 - l21 * l21;
    const double l22 = sqrt(d22);
    if (!(vxx > 0.0) || !(d11 > 0.0) || !(d22 > 0.0)) {
      // singular / indefinite point block: the reference's inv() raises LinAlgError (:128)
      if (lane == 0) atomicExch(&ctl->status, (int)BA_ERR_SINGULAR);
    }
    // inverse of L (lower): m = L^-1
    const double m00 = 1.0 / l00, m11 = 1.0 / l11, m22 = 1.0 / l22;
    const double m10 = -l10 * m00 * m11;
    const double m21 = -l21 * m11 * m22;
    const double m20 = -(l20 * m00 + l21 * m10) * m22;
    const double* g = GPT + 3 * (size_t)j;
    const double z0 = m00 * g[0];
    const double z1 = m10 * g[0] + m11 * g[1];
    const double z2 = m20 * g[0] + m21 * g[1] + m22 * g[2];
    if (lane == 0) {
      double* li = LINV + 6 * (size_t)j;
      li[0] = m00; li[1] = m10; li[2] = m11; li[3] = m20; li[4] = m21; li[5] = m22;
      double* z = Z + 3 * (size_t)j;
      z[0] = z0; z[1] = z1; z[2] = z2;
      if (!DENSE) {
        // point table of the pair kernel: X_j and the damped inverse block V^-1 = L^-T L^-1
        double* pt = PT + (size_t)j * kPT;
        pt[0] = X[3 * (size_t)j];
        pt[1] = X[3 * (size_t)j + 1];
        pt[2] = X[3 * (size_t)j + 2];
        pt[3] = m00 * m00 + m10 * m10 + m20 * m20;
        pt[4] = m10 * m11 + m20 * m21;
        pt[5] = m20 * m22;
        pt[6] = m11 * m11 + m21 * m21;
        pt[7] = m21 * m22;
        pt[8] = m22 * m22;
      }
      if (DENSE) {
        Yt[(size_t)(3 * j + 0) * ld + rhs_col] = z0;
        Yt[(size_t)(3 * j + 1) * ld + rhs_col] = z1;
        Yt[(size_t)(3 * j + 2) * ld + rhs_col] = z2;
        if (colmax) {
          const unsigned h0 = colmax_top16(z0, colmax, rhs_col), h1 = colmax_top16(z1, colmax, rhs_col),
                         h2 = colmax_top16(z2, colmax, rhs_col);
          colmax_smem_max(cm, rhs_col, max(max(h0, h1), h2));
        }
      }
    }
    const int64_t lo = DENSE ? j * M : obs_ptr[j];
    const int64_t hi = DENSE ? lo + M : obs_ptr[j + 1];
    const double xj0 = MF ? X[3 * (size_t)j] : 0.0, xj1 = MF ? X[3 * (size_t)j + 1] : 0.0,
                 xj2 = MF ? X[3 * (size_t)j + 2] : 0.0;
    for (int64_t o0 = lo; o0 < hi; o0 += 32) {
      const int64_t o = o0 + lane;
      const int cnt = (int)(hi - o0 < 32 ? hi - o0 : 32);
      const bool on = o < hi;
      // masked camera Jacobian rows (gauge-pinned parameters zeroed) and T = 2 Jx L^-T (2x3):
      // T[k][d] = 2 sum_b Jx[k][b] m[d][b]
      double ja[9], jb[9];
      double ta0 = 0, ta1 = 0, ta2 = 0, tb0 = 0, tb1 = 0, tb2 = 0;
      if (on) {
        const int i = DENSE ? (int)(o - lo) : obs_cam[o];
        const uint32_t mask = gauge_mask(i, axis);
        double a0, a1, a2, b0, b1, b2;
        if (MF) {
          ObsJacobian J;
          obs_jacobian(tab + (size_t)i * kTabStride, xj0, xj1, xj2, J);
          a0 = J.ax[0]; a1 = J.ax[1]; a2 = J.ax[2];
          b0 = J.bx[0]; b1 = J.bx[1]; b2 = J.bx[2];
#pragma unroll
          for (int a = 0; a < 9; ++a) {
            const bool pin = (mask >> a) & 1u;
            ja[a] = pin ? 0.0 : J.ja[a];
            jb[a] = pin ? 0.0 : J.jb[a];
          }
        } else {
          const double2* rp = reinterpret_cast<const double2*>(JP + (size_t)o * kJP);
          const double2 p1 = rp[1], p2 = rp[2], p3 = rp[3];
          a0 = p1.x; a1 = p1.y; a2 = p2.x; b0 = p2.y; b1 = p3.x; b2 = p3.y;
          const double2* rc = reinterpret_cast<const double2*>(JC + (size_t)o * kJC);
          double jc[kJC];
#pragma unroll
          for (int k = 1; k < kJC / 2; ++k) {
            const double2 t2 = rc[k];
            jc[2 * k] = t2.x;
            jc[2 * k + 1] = t2.y;
          }
#pragma unroll
          for (int a = 0; a < 9; ++a) {
            const bool pin = (mask >> a) & 1u;
            ja[a] = pin ? 0.0 : jc[2 + a];
            jb[a] = pin ? 0.0 : jc[11 + a];
          }
        }
        const double axr[3] = {a0, a1, a2}, bxr[3] = {b0, b1, b2};
        double ta[3], tb[3];
        scaled_point_rows(axr, bxr, m00, m10, m11, m20, m21, m22, ta, tb);
        ta0 = ta[0]; ta1 = ta[1]; ta2 = ta[2];
        tb0 = tb[0]; tb1 = tb[1]; tb2 = tb[2];
      }
      if (on) {
        // Y[a][d] = Jc0[a] T[0][d] + Jc1[a] T[1][d], staged in shared memory so that the warp
        // writes whole contiguous runs (the per-lane 72-byte pieces would be partial sectors)
#pragma unroll
        for (int a = 0; a < 9; ++a) {
          const double y0 = y_entry(ja[a], jb[a], ta0, tb0);
          const double y1 = y_entry(ja[a], jb[a], ta1, tb1);
          const double y2 = y_entry(ja[a], jb[a], ta2, tb2);
          if (DENSE) {
            st[9 * lane + a] = y0;
            st[288 + 9 * lane + a] = y1;
            st[576 + 9 * lane + a] = y2;
          } else {
            st[27 * lane + a] = y0;
            st[27 * lane + 9 + a] = y1;
            st[27 * lane + 18 + a] = y2;
          }
        }
      }
      __syncwarp();
      if (DENSE) {
        const int col0 = 9 * (int)(o0 - lo);
        double* dst = Yt + (size_t)(3 * j) * ld + col0;
        for (int k = lane; k < 9 * cnt; k += 32) {
          const double y0 = st[k], y1 = st[288 + k], y2 = st[576 + k];
          dst[k] = y0;
          dst[(size_t)ld + k] = y1;
          dst[2 * (size_t)ld + k] = y2;
          if (colmax) {
            const unsigned h0 = colmax_top16(y0, colmax, col0 + k), h1 = colmax_top16(y1, colmax, col0 + k),
                           h2 = colmax_top16(y2, colmax, col0 + k);
            colmax_smem_max(cm, col0 + k, max(max(h0, h1), h2));
          }
        }
      } else {
        double* dst = Ysp + (size_t)o0 * 27;
        for (int k = lane; k < 27 * cnt; k += 32) dst[k] = st[k];
      }
      __syncwarp();
    }
  }
  if (DENSE && colmax) {
    __syncthreads();
    for (int k = threadIdx.x; k < ld; k += blockDim.x)
      if (cm[k]) atomicMax(colmax + k, (unsigned long long)cm[k] << 48);
  }
}

// Dense scenes whose camera table fits next to the staging rows re-derive the Jacobian rows.
bool dense_matrix_free(const ba_engine* e) {
  return e->dense && tab_smem_doubles(e->M) * sizeof(double) <= 48 * 1024;
}

// Every path that runs K2b (LM graph, eager loop, covariance, sharded phases) comes through here, so the
// column maxima are reset before each launch that gathers them.
int launch_k2b(ba_engine* e, bool conditional, double c_host, cudaStream_t s) {
  const int use_ctl = conditional ? 1 : 0;
  const bool mf = dense_matrix_free(e);
  unsigned long long* colmax = e->syrk.colmax;  // null unless the dense product is emulated
  if (colmax) BA_CUDA(cudaMemsetAsync(colmax, 0, (size_t)e->n_pad * sizeof(unsigned long long), s));
  const size_t kStage = 8 * 864 * sizeof(double) + (mf ? tab_smem_doubles(e->M) * sizeof(double) : 0) +
                        (colmax ? ((size_t)e->n_pad * sizeof(unsigned short) + 15) / 16 * 16 : 0);
  const int grid = balanced_blocks((e->N + 7) / 8, (int64_t)e->num_sms * 16);
#define BA_K2B_LAUNCH(D, F)                                                                                  \
  do {                                                                                                       \
    BA_CUDA(cudaFuncSetAttribute(k2b_point_solve_kernel<D, F>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                 (int)kStage));                                                              \
    k2b_point_solve_kernel<D, F><<<grid, 256, kStage, s>>>(                                                  \
        e->N, e->M, e->axis, e->obs_ptr, e->obs_cam, e->JP, e->JC, e->V, e->GPT, c_host, e->ctl, use_ctl,   \
        e->LINV, e->Z, e->Yt, e->n_pad, e->rhs_row, e->Ysp, e->X[0], e->pairs.PT, e->camtab[0], e->f0,        \
        colmax);                                                                                             \
  } while (0)
  if (mf) BA_K2B_LAUNCH(true, true);
  else if (e->dense) BA_K2B_LAUNCH(true, false);
  else BA_K2B_LAUNCH(false, false);
#undef BA_K2B_LAUNCH
  BA_LAUNCH_CHECK();
  return BA_OK;
}

}  // namespace ba
