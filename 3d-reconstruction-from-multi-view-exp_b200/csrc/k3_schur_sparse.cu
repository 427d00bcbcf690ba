// K3 for sparse visibility: matrix-free, pair-stationary Schur products.
//
//   P[9i+a][9k+b] = sum over points j seen by both camera i and camera k (k <= i) of
//                   sum_d Y_ij[a][d] Y_kj[b][d]                (reference :132-135)
//   P[rhs][9i+a]  = sum_j sum_d Y_ij[a][d] z_j[d]               (reference :138-143)
//
// With Y_ij = Jc_ij^T (2 Jx_ij) L_j^-T (Jc the 2x9 camera Jacobian, Jx the 2x3 point Jacobian of
// observation (i, j), L_j L_j^T the damped V_j) the product of a camera pair through point j is
//
//   Y_ij Y_kj^T = Jc_ij^T G Jc_kj,    G = 4 Jx_ij Vd_j^-1 Jx_kj^T   (2x2),
//
// and Jc, Jx are functions of the camera parameters and X_j alone (reference :309-398; they do not
// involve the observed image point).  So nothing per observation has to be read: the kernel
// re-derives both Jacobians from the two cameras' table rows (shared memory) and the per-point row
// PT[j] = [X_j | Vd_j^-1] (96 B; 96 MB for 10^6 points: resident in the 126 MB L2), i.e. ~310 FP64
// operations and 96 B of L2 traffic per pair-point instead of 2 x 216 B of gathered Y blocks,
// which at C4 (19 GB of blocks, each read m_j = 100 times) made the kernel latency/HBM bound.
//
// ONE WARP PER CAMERA PAIR (i, k), k < i; every 32 common points make a round: their rows PT[j] are
// gathered into shared memory with 16-byte cp.async (five lanes per row), double buffered so that the
// gather of round r + 1 is in flight while round r is computed; every lane takes ONE common point.
// No shared-memory or global read-modify-write; the per-lane sums meet once per pair in a fixed order.
// Order of summation depends on the data only: runs are bit-reproducible.
//
// The camera-pair product is one PairProduct (ba_common.cuh) of the engine; two pair kernels, and where
// the common points come from decides which one runs (its `kind`; measurements: DESIGN.md section 3b):
//   * pairs_prepare           at engine creation: the pair-item count (refused past the launch limit),
//                             the bitmaps and the point table PT.
//   * pairs_index             with the observations: bitmaps per camera and -- memory permitting -- the
//                             STATIC PAIR LISTS: the ascending ids of the points every pair shares
//                             (pair_count_kernel, exclusive sum, pair_fill_kernel; 4 B per pair-point).
//                             Visibility does not change between iterations; intersecting the bitmaps
//                             and compacting the hits every solve was more than half of the kernel.
//   * schur_pairs_reg_kernel  PAIRS_LISTS: 32 ids per round with one coalesced load; the pair's 9 x 9
//                             block lives in 81 FP64 registers per lane (144 DFMAs per point).
//   * schur_pairs_kernel      PAIRS_SCAN, when the lists do not fit a third of the free memory (or
//                             BA_PAIRS_NO_LIST is set): it scans the bitmaps itself (4096 points per step,
//                             warp prefix sum, ring queue) and sums the leading 8 x 8 of the block on
//                             DMMA.8x8x4 (operands transposed through shared memory).  Register
//                             accumulators lose with the scan (40.0 against 35.9 ms at 1000 x 200k): at
//                             255 registers two warps per scheduler cannot overlap the scan's serial
//                             phases.  Without the scan they win (27.0 against 27.8 ms).
// Both take their per-point arithmetic from pair_point, so they differ only in how they sum.
//
// Bound: FP64 pipe (~316 instructions per pair-point; sum_j m_j (m_j - 1) / 2 pair-points).  DMMA runs
// on the same FP64 datapath as DFMA on this GPU (fp64_peak.cu, mode 2), so the tensor form buys no
// arithmetic, only issue slots -- and costs the fragment traffic.
//
// schur_diag_kernel: the diagonal blocks P[9i..][9i..] and the rhs row, a segmented reduction over
// the camera's observations in camera-major order (fixed chunking and order).
#include <cub/device/device_scan.cuh>

#include <cstdlib>

#include "ba_common.cuh"

namespace ba {

constexpr int kPS = 14;            // doubles per point row in shared memory (112 B = 7 x 16: odd -> conflict-free LDS.128)
constexpr int kPieces = 5;         // 16-byte pieces gathered per point row (the 9 doubles in use)
constexpr int kPairTile = 32;      // pairs are scheduled in kPairTile x kPairTile tiles of (i, k)
constexpr int kDiagPart = 54;      // 45 unique entries of the diagonal block + 9 rhs entries
constexpr int kQueue = 128;        // queue capacity (point ids); a power of two: the queue is a ring
constexpr int kFragX = 32 * 8 + 4; // doubles between the two rows of a fragment array (+4: conflict-free fragment loads)

// ---- index: per camera bitmap over points -------------------------------------------------------
__global__ void bitmap_fill_kernel(int64_t nobs, int64_t Wp, const int32_t* __restrict__ obs_cam,
                                   const int32_t* __restrict__ obs_pt, uint32_t* __restrict__ bits) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < nobs; o += stride) {
    const int j = obs_pt[o];
    atomicOr(&bits[(size_t)obs_cam[o] * Wp + (j >> 5)], 1u << (j & 31));
  }
}

// ---- static pair lists ----------------------------------------------------------------------------
// Which points two cameras share does not change between iterations, but intersecting the bitmaps,
// compacting the hits and queueing them was 55-60 % of the pair kernel's time (stall samples, DESIGN.md
// section 3b) -- every solve.  The intersection is therefore done ONCE per engine: pair_count_kernel
// counts the common points of every pair item, an exclusive sum gives the offsets, pair_fill_kernel
// writes the ascending point ids.  4 B per pair-point (C4: 19.8 GB of the 180 GB); if that exceeds a
// third of the free memory the lists are not built and the pair kernel scans the bitmaps instead.
__device__ __forceinline__ bool pair_from_linear(int64_t t, int M, int& i, int& k);

__global__ void __launch_bounds__(256)
pair_count_kernel(int M, int64_t Wp, int64_t n_items, const uint32_t* __restrict__ bits, int64_t* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (t > n_items) return;
  int i, k;
  int64_t acc = 0;
  if (t < n_items && pair_from_linear(t, M, i, k)) {
    const uint4* bi = reinterpret_cast<const uint4*>(bits + (size_t)i * Wp);
    const uint4* bk = reinterpret_cast<const uint4*>(bits + (size_t)k * Wp);
    for (int64_t w = lane; w < Wp / 4; w += 32) {
      const uint4 a = bi[w], b = bk[w];
      acc += __popc(a.x & b.x) + __popc(a.y & b.y) + __popc(a.z & b.z) + __popc(a.w & b.w);
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if (lane == 0) counts[t] = acc;  // counts[n_items] = 0: the exclusive sum then ends with the total
}

__global__ void __launch_bounds__(256)
pair_fill_kernel(int M, int64_t Wp, int64_t n_items, const uint32_t* __restrict__ bits,
                 const int64_t* __restrict__ ptr, int32_t* __restrict__ pts) {
  const int lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  int i, k;
  if (t >= n_items || !pair_from_linear(t, M, i, k)) return;
  const uint4* bi = reinterpret_cast<const uint4*>(bits + (size_t)i * Wp) + lane;
  const uint4* bk = reinterpret_cast<const uint4*>(bits + (size_t)k * Wp) + lane;
  int64_t running = ptr[t];
  for (int64_t w0 = 0; w0 < Wp; w0 += 128) {  // 4096 points per batch, 128 per lane: ascending over the lanes
    const uint4 a = bi[w0 >> 2], b = bk[w0 >> 2];
    uint64_t c0 = ((uint64_t)(a.y & b.y) << 32) | (a.x & b.x);
    uint64_t c1 = ((uint64_t)(a.w & b.w) << 32) | (a.z & b.z);
    const int n = __popcll(c0) + __popcll(c1);
    int incl = n;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, off);
      if (lane >= off) incl += v;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    int32_t* dst = pts + running + (incl - n);
    const int jbase = (int)(w0 + 4 * lane) * 32;
    while (c0 != 0ull) {
      *dst++ = jbase + __ffsll((long long)c0) - 1;
      c0 &= c0 - 1;
    }
    while (c1 != 0ull) {
      *dst++ = jbase + 64 + __ffsll((long long)c1) - 1;
      c1 &= c1 - 1;
    }
    running += total;
  }
}

// ---- off-diagonal pairs -------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_addr), "l"(gmem));
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// 1 / d to <= ~1 ulp: hardware seed and two Newton steps (a full division is ~20 instructions)
__device__ __forceinline__ double rcp_nr(double d) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
  r = fma(r, fma(-d, r, 1.0), r);
  r = fma(r, fma(-d, r, 1.0), r);
  return r;
}

// Pair number t -> (i, k), k < i.  Pairs are ordered tile by tile (kPairTile x kPairTile cameras),
// so that the warps resident at any time share few bitmaps and walk the points in step.
__device__ __forceinline__ bool pair_from_linear(int64_t t, int M, int& i, int& k) {
  const int64_t per_tile = (int64_t)kPairTile * kPairTile;
  const int64_t tile = t / per_tile;
  const int r = (int)(t - tile * per_tile);
  int ti = (int)((sqrt(8.0 * (double)tile + 1.0) - 1.0) * 0.5);
  while ((int64_t)(ti + 1) * (ti + 2) / 2 <= tile) ++ti;
  while ((int64_t)ti * (ti + 1) / 2 > tile) --ti;
  const int tk = (int)(tile - (int64_t)ti * (ti + 1) / 2);
  i = ti * kPairTile + r / kPairTile;
  k = tk * kPairTile + r % kPairTile;
  return i < M && k < i;
}

struct PairSmem {
  double stage[2][32 * kPS];  // [stage][point of the round][kPS]: X (3), Vd^-1 (6: 00 01 02 11 12 22)
  double cam[2][20];          // table rows of camera i and k (K1's layout) + 1/f, u0/f0, v0/f0, 1/f0
  double ifrag[2 * kFragX];   // [x][lane][8]: first 8 entries of Jc_i row x of the lane's point (DMMA A operand)
  double tfrag[2 * kFragX];   // [x][lane][8]: first 8 entries of row x of G Jc_k            (DMMA B operand)
  int32_t queue[kQueue];      // point ids; [0, 32) = the next round
};

// Unscaled Jacobian pieces of one camera at one point (K1's formulas without the 1/r^2 factor):
// camera row a = [af, au, 0, -aX, aX x d], row b = [bf, 0, au, -bX, bX x d]; point rows aX, bX.
struct SideJac {
  double aX[3], bX[3], d[3], af, bf, au, r;
};

__device__ __forceinline__ SideJac side_jacobian(const double* __restrict__ c, double x0, double x1,
                                                 double x2) {
  SideJac s;
  s.d[0] = x0 - c[9];
  s.d[1] = x1 - c[10];
  s.d[2] = x2 - c[11];
  const double p = c[0] * s.d[0] + c[1] * s.d[1] + c[2] * s.d[2];
  const double q = c[3] * s.d[0] + c[4] * s.d[1] + c[5] * s.d[2];
  const double r = c[6] * s.d[0] + c[7] * s.d[1] + c[8] * s.d[2];
#pragma unroll
  for (int m = 0; m < 3; ++m) {
    s.aX[m] = r * c[m] - p * c[6 + m];      // :450
    s.bX[m] = r * c[3 + m] - q * c[6 + m];  // :459
  }
  s.af = r * ((p - c[17] * r) * c[16]);  // :336  (c[16] = 1/f, c[17] = u0/f0)
  s.bf = r * ((q - c[18] * r) * c[16]);  // :337  (c[18] = v0/f0)
  s.au = r * (r * c[19]);                // :350-356 (c[19] = 1/f0)
  s.r = r;
  return s;
}

// Table rows of cameras i and k into cam[0] and cam[1] (one warp).
__device__ __forceinline__ void stage_cameras(double (*cam)[20], const double* __restrict__ camtab, int i, int k,
                                              int lane) {
  const int which = lane >> 4, c = lane & 15;
  const double v = camtab[(size_t)(which ? k : i) * kCamTab + c];
  cam[which][c] = v;
  __syncwarp();
  if (c >= 12) cam[which][c + 4] = v;  // 1 / f, u0 / f0, v0 / f0, 1 / f0 (cam_prep_kernel) where side_jacobian reads them
  __syncwarp();
}

// The arithmetic of one pair-point, shared by both pair kernels: from the staged rows of cameras i and k
// and the point's staged row pt, Jc_i's pieces si and the rows t0, t1 of G Jc_k.
__device__ __forceinline__ void pair_point(const double* __restrict__ cam_i, const double* __restrict__ cam_k,
                                           const double* __restrict__ pt, SideJac& si, double* t0, double* t1) {
  const double2 x01 = *reinterpret_cast<const double2*>(pt);
  const double2 x2v = *reinterpret_cast<const double2*>(pt + 2);  // X2, V00
  const double2 v12 = *reinterpret_cast<const double2*>(pt + 4);  // V01, V02
  const double2 v34 = *reinterpret_cast<const double2*>(pt + 6);  // V11, V12
  const double v22 = pt[8];
  const double v00 = x2v.y, v01 = v12.x, v02 = v12.y, v11 = v34.x, v12_ = v34.y;
  si = side_jacobian(cam_i, x01.x, x01.y, x2v.x);
  const SideJac sk = side_jacobian(cam_k, x01.x, x01.y, x2v.x);
  // G = 4 Jx_i Vd^-1 Jx_k^T with the four 1 / r^2 factors folded into one scale
  const double rr = si.r * sk.r;
  const double rr2 = rr * rr;
  const double sc = 4.0 * rcp_nr(rr2 * rr2);
  double g00, g01, g10, g11;
  {
    const double m0 = v00 * sk.aX[0] + v01 * sk.aX[1] + v02 * sk.aX[2];
    const double m1 = v01 * sk.aX[0] + v11 * sk.aX[1] + v12_ * sk.aX[2];
    const double m2 = v02 * sk.aX[0] + v12_ * sk.aX[1] + v22 * sk.aX[2];
    g00 = sc * (si.aX[0] * m0 + si.aX[1] * m1 + si.aX[2] * m2);
    g10 = sc * (si.bX[0] * m0 + si.bX[1] * m1 + si.bX[2] * m2);
  }
  {
    const double m0 = v00 * sk.bX[0] + v01 * sk.bX[1] + v02 * sk.bX[2];
    const double m1 = v01 * sk.bX[0] + v11 * sk.bX[1] + v12_ * sk.bX[2];
    const double m2 = v02 * sk.bX[0] + v12_ * sk.bX[1] + v22 * sk.bX[2];
    g01 = sc * (si.aX[0] * m0 + si.aX[1] * m1 + si.aX[2] * m2);
    g11 = sc * (si.bX[0] * m0 + si.bX[1] * m1 + si.bX[2] * m2);
  }
  // rows of G Jc_k; Jc_k row a = [af, au, 0, -aX, aX x d], row b = [bf, 0, au, -bX, bX x d]
  t0[0] = g00 * sk.af + g01 * sk.bf;  t1[0] = g10 * sk.af + g11 * sk.bf;
  t0[1] = g00 * sk.au;                t1[1] = g10 * sk.au;
  t0[2] = g01 * sk.au;                t1[2] = g11 * sk.au;
#pragma unroll
  for (int m = 0; m < 3; ++m) {
    t0[3 + m] = -(g00 * sk.aX[m] + g01 * sk.bX[m]);
    t1[3 + m] = -(g10 * sk.aX[m] + g11 * sk.bX[m]);
  }
#pragma unroll
  for (int m = 0; m < 3; ++m) {
    const int m1 = (m + 1) % 3, m2 = (m + 2) % 3;
    const double aw = sk.aX[m1] * sk.d[m2] - sk.aX[m2] * sk.d[m1];
    const double bw = sk.bX[m1] * sk.d[m2] - sk.bX[m2] * sk.d[m1];
    t0[6 + m] = g00 * aw + g01 * bw;
    t1[6 + m] = g10 * aw + g11 * bw;
  }
}

// ---- bitmap scan (no pair lists) ------------------------------------------------------------------
// The lanes intersect the two cameras' bitmaps 128 points each per step, a warp prefix sum of the hit
// counts gives their slots in a ring queue of point ids, and every 32 queued ids make a round.
// 12 warps per SM at 168 registers.
__global__ void __launch_bounds__(32, 12)
schur_pairs_kernel(int M, int axis, int64_t Wp, const uint32_t* __restrict__ bits,
                   const double* __restrict__ camtab, double f0, const double* __restrict__ PT,
                   double* __restrict__ P, int ld, const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;
  int i, k;
  if (!pair_from_linear(blockIdx.x, M, i, k)) return;
  __shared__ __align__(16) PairSmem sm;
  const int lane = threadIdx.x;
  stage_cameras(sm.cam, camtab, i, k, lane);

  // four bitmap words (128 points) per lane and batch
  const uint4* bi = reinterpret_cast<const uint4*>(bits + (size_t)i * Wp) + lane;
  const uint4* bk = reinterpret_cast<const uint4*>(bits + (size_t)k * Wp) + lane;
  const uint32_t q_addr = (uint32_t)__cvta_generic_to_shared(sm.queue);
  const uint32_t s_addr = (uint32_t)__cvta_generic_to_shared(sm.stage[0]);

  // Accumulators.  The 8x8 leading part of the block is summed over the 32 lanes' points by the
  // FP64 tensor cores (DMMA.8x8x4, K = 2 rows x 32 points per round): 2 registers per lane in the
  // m8n8 C-fragment layout (row lane / 4, columns 2 (lane % 4) + {0, 1}).  Row 8, column 8 and the
  // corner stay per lane and meet in a fixed-order butterfly at the end.
  double c0 = 0.0, c1 = 0.0;
  double r8[8], c8[8], c88 = 0.0;
#pragma unroll
  for (int a = 0; a < 8; ++a) r8[a] = c8[a] = 0.0;
  const int fg = lane >> 2, fkq = lane & 3;
  const int frag_base = (fkq & 1) * kFragX + (fkq >> 1) * 8;

  int qn = 0;           // entries queued
  int head = 0;         // ring position of the first queued entry
  int rounds = 0;       // rounds whose gather has been issued
  int cnt_prev = 0;     // valid lanes of the round waiting in stage (rounds - 1) & 1

  auto compute = [&](int st, int cnt) {
    double2* i0 = reinterpret_cast<double2*>(sm.ifrag + lane * 8);
    double2* i1 = reinterpret_cast<double2*>(sm.ifrag + kFragX + lane * 8);
    double2* t0s = reinterpret_cast<double2*>(sm.tfrag + lane * 8);
    double2* t1s = reinterpret_cast<double2*>(sm.tfrag + kFragX + lane * 8);
    const int sw = (lane >> 1) & 3;
    if (lane < cnt) {
      SideJac si;
      double t0[9], t1[9];
      pair_point(sm.cam[0], sm.cam[1], sm.stage[st] + lane * kPS, si, t0, t1);
      double ia[9], ib[9];
      ia[0] = si.af;  ib[0] = si.bf;
      ia[1] = si.au;  ib[1] = 0.0;
      ia[2] = 0.0;    ib[2] = si.au;
#pragma unroll
      for (int m = 0; m < 3; ++m) {
        ia[3 + m] = -si.aX[m];
        ib[3 + m] = -si.bX[m];
      }
      ia[6] = si.aX[1] * si.d[2] - si.aX[2] * si.d[1];  ib[6] = si.bX[1] * si.d[2] - si.bX[2] * si.d[1];
      ia[7] = si.aX[2] * si.d[0] - si.aX[0] * si.d[2];  ib[7] = si.bX[2] * si.d[0] - si.bX[0] * si.d[2];
      ia[8] = si.aX[0] * si.d[1] - si.aX[1] * si.d[0];  ib[8] = si.bX[0] * si.d[1] - si.bX[1] * si.d[0];
      // 16-byte pieces swizzled by (lane / 2) % 4: the lanes of a quarter-warp hit distinct banks
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        i0[u ^ sw] = make_double2(ia[2 * u], ia[2 * u + 1]);
        i1[u ^ sw] = make_double2(ib[2 * u], ib[2 * u + 1]);
        t0s[u ^ sw] = make_double2(t0[2 * u], t0[2 * u + 1]);
        t1s[u ^ sw] = make_double2(t1[2 * u], t1[2 * u + 1]);
      }
      // row 8, column 8 and the corner of the block stay with the lane
#pragma unroll
      for (int a = 0; a < 8; ++a) {
        r8[a] = fma(ia[8], t0[a], fma(ib[8], t1[a], r8[a]));
        c8[a] = fma(ia[a], t0[8], fma(ib[a], t1[8], c8[a]));
      }
      c88 = fma(ia[8], t0[8], fma(ib[8], t1[8], c88));
    } else {
      const double2 z = make_double2(0.0, 0.0);
#pragma unroll
      for (int u = 0; u < 4; ++u) i0[u] = i1[u] = t0s[u] = t1s[u] = z;
    }
    __syncwarp();
    // leading 8x8: C += A B with A[a][kappa] = Jc_i row (kappa & 1) of point kappa / 2, entry a,
    // and B[kappa][b] likewise from G Jc_k; 16 steps of K = 4 (two points each)
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      // the two points of step u are rows 2u, 2u + 1: their swizzle is u % 4
      const int o = frag_base + 16 * u + ((((fg >> 1) ^ (u & 3)) << 1) | (fg & 1));
      const double fa = sm.ifrag[o];
      const double fb = sm.tfrag[o];
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                   : "+d"(c0), "+d"(c1)
                   : "d"(fa), "d"(fb));
    }
  };

  // Issue the gather of the next round (the first cnt entries of the ring), then compute the previous
  // round.
  auto round = [&](int cnt) {
    const uint32_t sa = s_addr + (uint32_t)(rounds & 1) * (32 * kPS * 8);
#pragma unroll
    for (int u = 0; u < kPieces; ++u) {  // X (3) + V^-1 (6) = 72 B: the first five 16-byte pieces of the row
      const int p = lane + 32 * u;
      const int row = (p * 205) >> 10;  // p / 5 for p < 160
      const int piece = p - kPieces * row;
      int j;
      asm volatile("ld.shared.s32 %0, [%1];\n" : "=r"(j) : "r"(q_addr + 4u * (uint32_t)((head + row) & (kQueue - 1))));
      if (row < cnt) cp_async16(sa + (row * kPS + 2 * piece) * 8, PT + (size_t)j * kPT + 2 * piece);
    }
    cp_commit();
    qn -= cnt;
    head = (head + cnt) & (kQueue - 1);  // the queue is a ring: nothing moves
    if (rounds > 0) {
      cp_wait<1>();
      __syncwarp();
      compute((rounds & 1) ^ 1, cnt_prev);
    }
    __syncwarp();
    cnt_prev = cnt;
    ++rounds;
  };

  // bitmap words are fetched one batch ahead
  uint4 wi = bi[0], wk = bk[0];
  for (int64_t w0 = 0; w0 < Wp; w0 += 128) {
    const uint4 ci = wi, ck = wk;
    if (w0 + 128 < Wp) {
      wi = bi[(w0 + 128) >> 2];
      wk = bk[(w0 + 128) >> 2];
    }
    uint64_t c0 = ((uint64_t)(ci.y & ck.y) << 32) | (ci.x & ck.x);
    uint64_t c1 = ((uint64_t)(ci.w & ck.w) << 32) | (ci.z & ck.z);
    const int jbase = (int)(w0 + 4 * lane) * 32;
    while (__any_sync(0xffffffffu, (c0 | c1) != 0ull)) {
      // exclusive prefix of the hit counts -> queue slots; hits that do not fit wait for the next pass
      const int n = __popcll(c0) + __popcll(c1);
      int incl = n;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += v;
      }
      const int total = __shfl_sync(0xffffffffu, incl, 31);
      int pos = qn + incl - n;
      while (c0 != 0ull && pos < kQueue) {
        const int b = __ffsll((long long)c0) - 1;
        c0 &= c0 - 1;
        sm.queue[(head + pos++) & (kQueue - 1)] = jbase + b;
      }
      while (c0 == 0ull && c1 != 0ull && pos < kQueue) {
        const int b = __ffsll((long long)c1) - 1;
        c1 &= c1 - 1;
        sm.queue[(head + pos++) & (kQueue - 1)] = jbase + 64 + b;
      }
      qn = qn + total < kQueue ? qn + total : kQueue;
      __syncwarp();
      while (qn >= 32) round(32);
    }
  }
  if (qn > 0) round(qn);
  if (rounds > 0) {
    cp_wait<0>();
    __syncwarp();
    compute((rounds - 1) & 1, cnt_prev);
  }

  // leading 8x8 straight from the C fragments; row 8, column 8 and the corner after a fixed-order
  // butterfly over the 32 lanes.  Rows / columns of gauge-pinned parameters (:62-72) are zero.
  const uint32_t mask_i = gauge_mask(i, axis), mask_k = gauge_mask(k, axis);
  {
    double* dst = P + (size_t)(9 * i + fg) * ld + 9 * k + 2 * fkq;
    const bool pin_r = (mask_i >> fg) & 1u;
    dst[0] = (pin_r || ((mask_k >> (2 * fkq)) & 1u)) ? 0.0 : c0;
    dst[1] = (pin_r || ((mask_k >> (2 * fkq + 1)) & 1u)) ? 0.0 : c1;
  }
#pragma unroll
  for (int a = 0; a < 8; ++a) {
    double v = r8[a], w = c8[a];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      v += __shfl_xor_sync(0xffffffffu, v, off);
      w += __shfl_xor_sync(0xffffffffu, w, off);
    }
    if (((mask_i >> 8) | (mask_k >> a)) & 1u) v = 0.0;
    if (((mask_i >> a) | (mask_k >> 8)) & 1u) w = 0.0;
    if (lane == a) P[(size_t)(9 * i + 8) * ld + 9 * k + a] = v;
    if (lane == 8 + a) P[(size_t)(9 * i + a) * ld + 9 * k + 8] = w;
  }
  {
    double v = c88;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (((mask_i >> 8) | (mask_k >> 8)) & 1u) v = 0.0;
    if (lane == 16) P[(size_t)(9 * i + 8) * ld + 9 * k + 8] = v;
  }
}

// ---- pair lists: register accumulators ------------------------------------------------------------
// DMMA shares the FP64 datapath with DFMA (fp64_peak mode 2: 32 TF/s in sum), so the tensor
// instructions of the kernel above buy no arithmetic, and building their fragments costs 128
// shared-memory wavefronts per 32 pair-points.  Here every lane keeps the whole 9 x 9 block of the pair
// in 81 FP64 registers and adds its point's Jc_i^T (G Jc_k) with 144 DFMAs (the structural zeros of
// Jc_i skipped): no fragments, no shuffles, 255 registers, eight warps per SM, independent accumulator
// chains.  The ids of a round come from the static lists (pairs_index): 32 with one coalesced
// load, fetched a round ahead.
// The 81 per-lane sums meet once per pair, through shared memory (the staging rows, free by then),
// in lane order.  Order of summation depends on the data only: bit-reproducible.
struct PairRegSmem {
  double stage[2][32 * kPS];  // [parity][lane][kPS] the rows of the round's points; reduction scratch [27][33] at the end
  double cam[2][20];
};
static_assert(27 * 33 <= 2 * 32 * kPS, "reduction scratch must fit the staging buffers");

__global__ void __launch_bounds__(32, 8)
schur_pairs_reg_kernel(int M, int axis, const double* __restrict__ camtab, double f0, const double* __restrict__ PT,
                       double* __restrict__ P, int ld, const ba_lm_state* ctl,
                       const int64_t* __restrict__ pair_ptr, const int32_t* __restrict__ pair_pts) {
  if (ctl && ctl->done) return;
  int i, k;
  if (!pair_from_linear(blockIdx.x, M, i, k)) return;
  __shared__ __align__(16) PairRegSmem sm;
  const int lane = threadIdx.x;
  stage_cameras(sm.cam, camtab, i, k, lane);

  double acc[9][9];
#pragma unroll
  for (int a = 0; a < 9; ++a)
#pragma unroll
    for (int b = 0; b < 9; ++b) acc[a][b] = 0.0;

  auto compute = [&](int st) {
    SideJac si;
    double t0[9], t1[9];
    pair_point(sm.cam[0], sm.cam[1], sm.stage[st] + lane * kPS, si, t0, t1);
    // block += Jc_i^T [t0; t1], row by row of Jc_i^T; its structural zeros are skipped
#pragma unroll
    for (int b = 0; b < 9; ++b) {
      acc[0][b] = fma(si.af, t0[b], fma(si.bf, t1[b], acc[0][b]));
      acc[1][b] = fma(si.au, t0[b], acc[1][b]);
      acc[2][b] = fma(si.au, t1[b], acc[2][b]);
    }
#pragma unroll
    for (int m = 0; m < 3; ++m) {
#pragma unroll
      for (int b = 0; b < 9; ++b) acc[3 + m][b] = fma(-si.aX[m], t0[b], fma(-si.bX[m], t1[b], acc[3 + m][b]));
    }
#pragma unroll
    for (int m = 0; m < 3; ++m) {
      const int m1 = (m + 1) % 3, m2 = (m + 2) % 3;
      const double aw = si.aX[m1] * si.d[m2] - si.aX[m2] * si.d[m1];
      const double bw = si.bX[m1] * si.d[m2] - si.bX[m2] * si.d[m1];
#pragma unroll
      for (int b = 0; b < 9; ++b) acc[6 + m][b] = fma(aw, t0[b], fma(bw, t1[b], acc[6 + m][b]));
    }
  };

  const uint32_t stage0 = (uint32_t)__cvta_generic_to_shared(sm.stage[0]);
  const int64_t lo = pair_ptr[blockIdx.x], hi = pair_ptr[blockIdx.x + 1];
  int jnext = lo + lane < hi ? pair_pts[lo + lane] : -1;
  int rounds = 0, cnt_prev = 0;
  for (int64_t base = lo; base < hi; base += 32) {
    const int cnt = hi - base < 32 ? (int)(hi - base) : 32;
    const int jcur = jnext;
    if (base + 32 < hi) jnext = base + 32 + lane < hi ? pair_pts[base + 32 + lane] : -1;
    const uint32_t dst = stage0 + (uint32_t)(rounds & 1) * (32 * kPS * 8);
#pragma unroll
    for (int u = 0; u < kPieces; ++u) {
      const int p = lane + 32 * u;
      const int row = (p * 205) >> 10;  // p / 5 for p < 160
      const int piece = p - kPieces * row;
      const int jr = __shfl_sync(0xffffffffu, jcur, row);
      if (row < cnt) cp_async16(dst + (uint32_t)(row * kPS + 2 * piece) * 8u, PT + (size_t)jr * kPT + 2 * piece);
    }
    cp_commit();
    if (rounds > 0) {
      cp_wait<1>();
      __syncwarp();
      if (lane < cnt_prev) compute((rounds & 1) ^ 1);
    }
    __syncwarp();
    cnt_prev = cnt;
    ++rounds;
  }
  if (rounds > 0) {
    cp_wait<0>();
    __syncwarp();
    if (lane < cnt_prev) compute((rounds - 1) & 1);
  }
  __syncwarp();

  // 81 sums over the 32 lanes, 27 at a time through the (now free) staging buffers: lane e adds
  // entry e of every lane in lane order.  Rows / columns of gauge-pinned parameters (:62-72) are zero.
  const uint32_t mask_i = gauge_mask(i, axis), mask_k = gauge_mask(k, axis);
  double* scratch = sm.stage[0];
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
    for (int e = 0; e < 27; ++e) scratch[e * 33 + lane] = acc[3 * pass + e / 9][e % 9];
    __syncwarp();
    if (lane < 27) {
      const double* row = scratch + lane * 33;
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
      for (int q = 0; q < 32; q += 4) {
        s0 += row[q];
        s1 += row[q + 1];
        s2 += row[q + 2];
        s3 += row[q + 3];
      }
      const int a = 3 * pass + lane / 9, b = lane % 9;
      const bool pin = ((mask_i >> a) | (mask_k >> b)) & 1u;
      P[(size_t)(9 * i + a) * ld + 9 * k + b] = pin ? 0.0 : (s0 + s1) + (s2 + s3);
    }
    __syncwarp();
  }
}

// ---- diagonal blocks and rhs --------------------------------------------------------------------
// grid (chunks, M): block (c, i) reduces chunk c of camera i's observations into 54 numbers.
__global__ void __launch_bounds__(128)
schur_diag_kernel(const int64_t* __restrict__ cam_ptr, const int32_t* __restrict__ cm_perm,
                  const int32_t* __restrict__ obs_pt, const double* __restrict__ Ysp,
                  const double* __restrict__ Z, double* __restrict__ Dpart, const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;
  const int i = blockIdx.y;
  const int chunk = blockIdx.x, nchunks = gridDim.x;
  const int64_t seg_lo = cam_ptr[i], seg_n = cam_ptr[i + 1] - seg_lo;
  const int64_t per = (seg_n + nchunks - 1) / nchunks;
  const int64_t lo = per * chunk;
  const int64_t hi = lo + per < seg_n ? lo + per : seg_n;
  double acc[kDiagPart];
#pragma unroll
  for (int q = 0; q < kDiagPart; ++q) acc[q] = 0.0;
  for (int64_t q = lo + threadIdx.x; q < hi; q += blockDim.x) {
    const int o = cm_perm[seg_lo + q];
    const double* y = Ysp + (size_t)o * 27;  // [d][a]
    const double* z = Z + 3 * (size_t)obs_pt[o];
    double v[27];
#pragma unroll
    for (int u = 0; u < 27; ++u) v[u] = y[u];
    const double z0 = z[0], z1 = z[1], z2 = z[2];
    int idx = 0;
#pragma unroll
    for (int r = 0; r < 9; ++r)
#pragma unroll
      for (int c = r; c < 9; ++c) acc[idx++] += v[r] * v[c] + v[9 + r] * v[9 + c] + v[18 + r] * v[18 + c];
#pragma unroll
    for (int r = 0; r < 9; ++r) acc[45 + r] += v[r] * z0 + v[9 + r] * z1 + v[18 + r] * z2;
  }
  __shared__ double sred[4][kDiagPart];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < kDiagPart; ++q) {
    const double s = warp_sum(acc[q]);
    if (lane == 0) sred[warp][q] = s;
  }
  __syncthreads();
  if (threadIdx.x < kDiagPart) {
    const double s = ((sred[0][threadIdx.x] + sred[1][threadIdx.x]) + sred[2][threadIdx.x]) +
                     sred[3][threadIdx.x];
    Dpart[((size_t)i * nchunks + chunk) * kDiagPart + threadIdx.x] = s;
  }
}

__global__ void schur_diag_finish_kernel(int nchunks, const double* __restrict__ Dpart,
                                         double* __restrict__ P, int ld, int rhs_row,
                                         const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;
  const int i = blockIdx.x;
  const int q = threadIdx.x;  // 0..89: 81 entries of the block, 9 of the rhs
  if (q >= 90) return;
  int src, r = 0, c = 0;
  if (q < 81) {
    r = q / 9;
    c = q % 9;
    const int lo = r < c ? r : c, hi = r < c ? c : r;
    src = lo * 9 - lo * (lo - 1) / 2 + (hi - lo);
  } else {
    src = 45 + (q - 81);
  }
  double s = 0.0;
  for (int ch = 0; ch < nchunks; ++ch) s += Dpart[((size_t)i * nchunks + ch) * kDiagPart + src];
  if (q < 81) {
    if (c <= r) P[(size_t)(9 * i + r) * ld + 9 * i + c] = s;
  } else {
    P[(size_t)rhs_row * ld + 9 * i + (q - 81)] = s;
  }
}

// ---- the camera-pair product: index, choice, launch -------------------------------------------------
int pairs_prepare(PairProduct* p, int M, int64_t N, cudaStream_t s) {
  *p = PairProduct();
  const int nt = (M + kPairTile - 1) / kPairTile;
  const int64_t n_items = (int64_t)nt * (nt + 1) / 2 * kPairTile * kPairTile;
  if (n_items >= ((int64_t)1 << 31)) {  // one block per pair item
    set_error("%d cameras exceed the camera-pair limit: %lld pair items, one launch takes fewer than 2^31 "
              "(at most %d cameras)", M, (long long)n_items, 2047 * kPairTile);
    return BA_ERR_INVALID;
  }
  p->M = M;
  p->N = N;
  p->n_items = n_items;
  p->Wp = ((N + 31) / 32 + 255) / 256 * 256;  // whole groups of 256 words: 32 lanes x 8 words
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&p->bits), (size_t)M * p->Wp * sizeof(uint32_t), s));
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&p->PT), (size_t)N * kPT * sizeof(double), s));
  return BA_OK;
}

static void free_lists(PairProduct* p, cudaStream_t s) {
  if (p->pair_ptr) cudaFreeAsync(p->pair_ptr, s);
  if (p->pair_pts) cudaFreeAsync(p->pair_pts, s);
  p->pair_ptr = nullptr;
  p->pair_pts = nullptr;
  p->kind = PAIRS_SCAN;
}

int pairs_index(PairProduct* p, int64_t nobs, const int32_t* obs_cam, const int32_t* obs_pt, int num_sms,
                cudaStream_t s) {
  free_lists(p, s);
  BA_CUDA(cudaMemsetAsync(p->bits, 0, (size_t)p->M * p->Wp * sizeof(uint32_t), s));
  BA_CUDA(cudaMemsetAsync(p->PT, 0, (size_t)p->N * kPT * sizeof(double), s));
  bitmap_fill_kernel<<<num_sms * 8, 256, 0, s>>>(nobs, p->Wp, obs_cam, obs_pt, p->bits);
  BA_LAUNCH_CHECK();
  // BA_PAIRS_NO_LIST: no lists, the pair kernel scans the bitmaps every solve (tests of that fallback)
  if (std::getenv("BA_PAIRS_NO_LIST")) return BA_OK;
  const int64_t n_items = p->n_items;
  if (cudaMallocAsync(reinterpret_cast<void**>(&p->pair_ptr), (size_t)(n_items + 1) * sizeof(int64_t), s) != cudaSuccess) {
    cudaGetLastError();
    p->pair_ptr = nullptr;
    return BA_OK;
  }
  const unsigned blocks = (unsigned)((n_items + 1 + 7) / 8);
  pair_count_kernel<<<blocks, 256, 0, s>>>(p->M, p->Wp, n_items, p->bits, p->pair_ptr);
  BA_LAUNCH_CHECK();
  {
    size_t tmp_bytes = 0;
    BA_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, p->pair_ptr, p->pair_ptr, (int)(n_items + 1), s));
    void* tmp = nullptr;
    BA_CUDA(cudaMallocAsync(&tmp, tmp_bytes, s));
    BA_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, p->pair_ptr, p->pair_ptr, (int)(n_items + 1), s));
    BA_CUDA(cudaFreeAsync(tmp, s));
  }
  int64_t total = 0;
  BA_CUDA(cudaMemcpyAsync(&total, p->pair_ptr + n_items, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  BA_CUDA(cudaStreamSynchronize(s));
  size_t free_b = 0, total_b = 0;
  BA_CUDA(cudaMemGetInfo(&free_b, &total_b));
  const size_t need = (size_t)(total > 0 ? total : 1) * sizeof(int32_t);
  if (need > free_b / 3 || cudaMallocAsync(reinterpret_cast<void**>(&p->pair_pts), need, s) != cudaSuccess) {
    cudaGetLastError();
    p->pair_pts = nullptr;
    free_lists(p, s);
    return BA_OK;
  }
  pair_fill_kernel<<<(unsigned)((n_items + 7) / 8), 256, 0, s>>>(p->M, p->Wp, n_items, p->bits, p->pair_ptr,
                                                                 p->pair_pts);
  BA_LAUNCH_CHECK();
  p->kind = PAIRS_LISTS;
  return BA_OK;
}

int pairs_launch(const PairProduct* p, const double* camtab, double f0, int axis, double* P, int ld,
                 const ba_lm_state* ctl, cudaStream_t s) {
  if (p->kind == PAIRS_LISTS) {
    BA_CUDA(cudaFuncSetAttribute(schur_pairs_reg_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                 (int)cudaSharedmemCarveoutMaxShared));
    schur_pairs_reg_kernel<<<(unsigned)p->n_items, 32, 0, s>>>(p->M, axis, camtab, f0, p->PT, P, ld, ctl, p->pair_ptr,
                                                              p->pair_pts);
  } else {
    BA_CUDA(cudaFuncSetAttribute(schur_pairs_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                 (int)cudaSharedmemCarveoutMaxShared));
    schur_pairs_kernel<<<(unsigned)p->n_items, 32, 0, s>>>(p->M, axis, p->Wp, p->bits, camtab, f0, p->PT, P, ld, ctl);
  }
  BA_LAUNCH_CHECK();
  return BA_OK;
}

void pairs_release(PairProduct* p, cudaStream_t s) {
  free_lists(p, s);
  if (p->bits) cudaFreeAsync(p->bits, s);
  if (p->PT) cudaFreeAsync(p->PT, s);
  *p = PairProduct();
}

int launch_schur_sparse(ba_engine* e, const ba_lm_state* ctl, cudaStream_t s) {
  ProfScope ps(e, PG_SYRK, s);
  dim3 dgrid(e->cam_chunks, e->M);
  schur_diag_kernel<<<dgrid, 128, 0, s>>>(e->cam_ptr, e->cm_perm, e->obs_pt, e->Ysp, e->Z, e->Upart, ctl);
  BA_LAUNCH_CHECK();
  schur_diag_finish_kernel<<<e->M, 96, 0, s>>>(e->cam_chunks, e->Upart, e->P(), e->n_pad, e->rhs_row, ctl);
  BA_LAUNCH_CHECK();
  return pairs_launch(&e->pairs, e->camtab[0], e->f0, e->axis, e->P(), e->n_pad, ctl, s);
}

}  // namespace ba
