// Shared definitions of the bundle-adjustment engine: engine object, error handling,
// launch bookkeeping and small device helpers.  sm_100a only.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "ba_b200.h"

namespace ba {

// ------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);

#define BA_CUDA(expr)                                                                      \
  do {                                                                                     \
    cudaError_t _err = (expr);                                                             \
    if (_err != cudaSuccess) {                                                             \
      ::ba::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_err), __FILE__,  \
                      __LINE__);                                                           \
      return BA_ERR_CUDA;                                                                  \
    }                                                                                      \
  } while (0)

#define BA_TRY(expr)                 \
  do {                               \
    int _st = (expr);                \
    if (_st != BA_OK) return _st;    \
  } while (0)

// ------------------------------------------------------------------------------------
// constants of the data layout
// ------------------------------------------------------------------------------------
constexpr int kCamTab = 16;   // doubles per camera in the derived table (128 B rows)
constexpr int kJP = 8;        // doubles per observation, point-side row: e(2), de/dX (2x3)
constexpr int kJC = 20;       // doubles per observation, camera-side row: e(2), de/dcam (2x9)
constexpr int kUPart = 54;    // 45 unique entries of U_i + 9 of dF_i
constexpr int kPT = 12;       // doubles per point in the pair kernel's point table (sparse):
                              // X (3), damped V^-1 (00 01 02 11 12 22), 3 pad = 96 B = 3 sectors
constexpr int kCholNB = 64;   // panel width of the blocked Cholesky
constexpr int kCholOB = 256;  // outer block (4 panels) of the two-level variant for large systems
constexpr int kCholSplitMinRows = 2560;  // trailing rows from which the rank-256 update runs on 128-tiles
constexpr int kMaxRecords = 4096;
constexpr int kMaxRanks = 8;    // ranks of one peer-memory exchange (one NVSwitch domain)

// Pinned camera parameters (gauge): camera 0 keeps f,u0,v0 only; camera 1 loses one
// translation component (reference lib/bundle_adjustment.py:62-72).  Bit a set = parameter a
// of that camera is removed from the unknowns.
__host__ __device__ inline uint32_t gauge_mask(int cam, int axis) {
  return cam == 0 ? 0x1F8u : (cam == 1 ? (1u << (3 + axis)) : 0u);
}

struct CamState {
  double* f = nullptr;  // [M]
  double* u = nullptr;  // [M][2]
  double* R = nullptr;  // [M][3][3] row-major, camera-to-world
  double* t = nullptr;  // [M][3]
};

// "k3" brackets the whole Schur phase; "syrk" only the dense product inside it (the DMMA kernels, or
// the INT8 emulation's conversion, product and reconstruction kernels; nested scopes use their own
// event pair).
enum ProfGroup { PG_K1 = 0, PG_K2, PG_K3, PG_K4, PG_COST, PG_OTHER, PG_SYRK, PG_CHOL, PG_COMM, PG_COUNT };

// One CTA of the dense Schur product: tile (ti, tj) of P and the k-chunks [c_lo, c_hi) of Y^T.
struct SyrkItem {
  int ti, tj, c_lo, c_hi;
  int slot2;  // >= 0: a "tall" item also computes the ragged rows below its tile (the thin tile
              // (ti + 1, tj)); their partial results go to this slot of the partial-tile store
};

// One two-CTA cluster of the emulated Schur product: modulus `mod`, 256-tile (ti, tj) of P, 128-row
// k-blocks [kb_lo, kb_hi) of the residue planes.
struct EmuItem {
  int mod, ti, tj, kb_lo, kb_hi;
};

struct Comm;  // peer-memory exchange of a sharded run (comm_peer.cu)

struct ProfSlot {
  double ms = 0.0;
  int64_t launches = 0;
};

// A timed scope whose events have been recorded but not read yet: reading them needs a host
// synchronisation, and a synchronisation after every scope would let the GPU drain between
// kernels (launch latency inside the brackets).  They are resolved when the profile is read.
struct ProfPending {
  int group;
  cudaEvent_t a, b;
};

}  // namespace ba

// The opaque engine of the C ABI.
struct ba_engine {
  ba_problem prob{};
  int64_t N = 0, nobs = 0;
  int M = 0, dense = 0, axis = 0, device = 0;
  double f0 = 1.0;
  int num_sms = 148;

  // reduced system layout: n_full = 9M unknown slots (gauge entries pinned, not deleted),
  // row rhs_row = 9M carries the right-hand side, n_pad = padded order = leading dimension
  int n_full = 0, rhs_row = 0, n_pad = 0;
  int syrk_tile = 128;
  int syrk_n_items = 0, syrk_n_tiles = 0;
  int syrk_n_ctas = 0;                 // CTAs of the SYRK launch (= items unless stream-K planned)
  int* syrk_cta_first = nullptr;       // [syrk_n_ctas + 1] stream-K: first item of every CTA (else null)
  ba::SyrkItem* syrk_items = nullptr;  // [syrk_n_items] launch order
  int* syrk_tile_first = nullptr;      // [syrk_n_tiles + 1]
  int* syrk_tile_items = nullptr;      // items of each tile in ascending k order
  int64_t k_pad = 0;  // padded 3N (rows of Yt)
  // dense Schur product emulated on the INT8 tensor cores (k3_schur_syrk.cu): chosen at engine creation
  int syrk_emu = 0;
  int emu_bits = 0;                      // b: |scaled entry| <= 2^b, exact CRT lift for k_pad rows
  int emu_n_items = 0;
  int emu_n_full = 0;                    // items of whole 256-row tile rows; the ragged row's items follow
  ba::EmuItem* emu_items = nullptr;      // [emu_n_items] launch order
  int8_t* Yq = nullptr;                  // [kEmuModuli][n_pad][k_pad] residue planes, K-major
  uint32_t* Pmod = nullptr;              // [kEmuModuli][lower 128-tiles][128 cols][128 rows] residue sums
  unsigned long long* colmax = nullptr;  // [n_pad] bit pattern of max |Yt[k][a]| over k

  // observations (CSR by point) and camera-major index
  int64_t* obs_ptr = nullptr;
  int32_t* obs_cam = nullptr;  // null when dense
  int32_t* obs_pt = nullptr;   // null when dense
  double* obs_xy = nullptr;
  int64_t* cam_ptr = nullptr;  // [M+1] (sparse)
  int32_t* cm_perm = nullptr;  // [nobs] observation ids sorted by camera (sparse)
  uint32_t* bits = nullptr;    // [M][Wp] per camera: bitmap over points (sparse)
  int64_t Wp = 0;              // words per camera bitmap, padded to a multiple of 256
  bool have_obs = false, have_state = false;

  // state: [0] current, [1] trial
  double* X[2] = {nullptr, nullptr};
  ba::CamState cam[2];
  double* camtab[2] = {nullptr, nullptr};
  double* gauge = nullptr;  // [16] R0, t0, divisor s, baseline length (k6_gauge.cu)
  bool have_gauge = false;

  // linearisation
  double *JP = nullptr, *JC = nullptr, *V = nullptr, *GPT = nullptr;
  double *Upart = nullptr;  // [M][cam_chunks][54]
  double *Uloc = nullptr;   // [M*81 | M*9] this engine's U_i and dF_i (before any all-reduce)
  int cam_chunks = 1;

  // per solve
  double *LINV = nullptr, *Z = nullptr;
  double* Yt = nullptr;   // dense: [k_pad][n_pad]
  double* Ysp = nullptr;  // sparse: [nobs][27]
  double* PT = nullptr;   // sparse: [N][kPT] point table of the pair kernel (X, damped V^-1)
  // sparse: the common points of every camera pair, compacted once per engine (visibility does not
  // change between iterations): pair_ptr [n_pair_items + 1], pair_pts [pair_total] ascending point ids;
  // null when the lists would not fit the memory budget (the pair kernel then scans the bitmaps)
  int64_t* pair_ptr = nullptr;
  int32_t* pair_pts = nullptr;
  int64_t pair_total = 0;
  double* red = nullptr;  // [n_pad*n_pad | M*81 | M*9]
  int64_t red_len = 0;
  bool red_in_window = false;  // red lives in the exchange window (freed with it)
  ba::Comm* comm = nullptr;    // non-null: sharded run, sums go through peer memory
  double* Spart = nullptr;  // partial tiles, one per work item of the Schur product
  double* Lt = nullptr;     // Cholesky block column, k-major copy [kCholOB][n_pad]
  double* ywork = nullptr;  // [n_pad] running right-hand side of the grid-wide back substitution
  unsigned int* chol_bar = nullptr;  // grid barrier counter of that kernel
  double* Winv = nullptr;   // [panels][64][64] L_D^-T of every diagonal block (back substitution)
  double* dxi = nullptr;    // [M][9]
  double* cost_part = nullptr;
  int cost_blocks = 0;
  double* cost_buf = nullptr;  // [4]: cost of the current / initial state, trial cost, "singular block" flag of the trial solve (summed over ranks with the cost), pad

  ba_lm_state* ctl = nullptr;       // device
  ba_iter_record* rec = nullptr;    // device [kMaxRecords]
  ba_lm_state* ctl_host = nullptr;  // pinned [4]: [0] read_ctl, [1], [2] the two solve graphs

  // the LM loop as CUDA graphs (ba_lm_run): one inner solve per graph, two instances (A/B) so
  // that each has its own pinned control-block slot and completion event
  cudaStream_t own_stream = nullptr;
  cudaGraphExec_t solve_graph[2] = {nullptr, nullptr};
  cudaEvent_t solve_ev[2] = {nullptr, nullptr};
  int64_t graph_launches = 0;  // kernels per graph

  // profiling
  bool profiling = false;
  ba::ProfSlot prof[ba::PG_COUNT];
  std::vector<ba::ProfPending> prof_pending;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;

  double* P() const { return red; }
  double* U() const { return red + (int64_t)n_pad * n_pad; }
  double* GCAM() const { return red + (int64_t)n_pad * n_pad + (int64_t)M * 81; }
};

namespace ba {

extern int64_t g_launch_count;

// Brackets a group of launches with CUDA events when profiling is on.
struct ProfScope {
  ba_engine* e;
  int group;
  cudaStream_t s;
  int64_t launches_before;
  cudaEvent_t a = nullptr, b = nullptr;  // own pair: scopes may nest
  ProfScope(ba_engine* e_, int group_, cudaStream_t s_) : e(e_), group(group_), s(s_) {
    launches_before = g_launch_count;
    if (e->profiling) {
      cudaEventCreate(&a);
      cudaEventCreate(&b);
      cudaEventRecord(a, s);
    }
  }
  ~ProfScope() {
    e->prof[group].launches += g_launch_count - launches_before;
    if (a) {
      cudaEventRecord(b, s);
      e->prof_pending.push_back({group, a, b});
    }
  }
};

// Read the recorded scopes (synchronises on their events) into the per-group totals.
inline void prof_resolve(ba_engine* e, bool keep) {
  for (const ProfPending& p : e->prof_pending) {
    if (keep) {
      cudaEventSynchronize(p.b);
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) e->prof[p.group].ms += ms;
    }
    cudaEventDestroy(p.a);
    cudaEventDestroy(p.b);
  }
  e->prof_pending.clear();
}

#define BA_LAUNCH_CHECK()                                                       \
  do {                                                                          \
    ::ba::g_launch_count++;                                                     \
    cudaError_t _err = cudaGetLastError();                                      \
    if (_err != cudaSuccess) {                                                  \
      ::ba::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_err), \
                      __FILE__, __LINE__);                                      \
      return BA_ERR_CUDA;                                                       \
    }                                                                           \
  } while (0)

// ------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// Deterministic block sum (fixed tree): every thread gets the result.  `scratch` >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  double r = 0.0;
  for (int w = 0; w < nw; ++w) r += scratch[w];
  return r;
}
#endif

#ifdef __CUDACC__
// Shared-memory copy of a camera table: rows padded to 17 doubles (conflict-free when the lanes of a
// warp read one column of 32 consecutive rows, the dense-visibility pattern).
constexpr int kTabStride = kCamTab + 1;
__host__ __device__ constexpr size_t tab_smem_doubles(int M) { return ((size_t)M * kTabStride + 1) & ~(size_t)1; }

// Jacobian rows of ONE observation from the camera's table row T (rows of K R^T (9), t (3), f, u0,
// v0) and the point X -- reference :283-427 (_calc_pqr, _calc_X_diff_pqr, _calc_{f,u,t,R}_diff_pqr).
// K1 stores these rows (JP, JC); the dense K2b and the dense point update re-derive them instead of
// reading 224 B per observation back.  Every operation is pinned (explicit fma / __dmul_rn, no
// compiler contraction), so all callers get the same bits.
struct ObsJacobian {
  double p, q, r;       // projection before the division
  double ir, inv_f0;    // 1 / r; 1 / f0 (from the table)
  double ax[3], bx[3];  // d e0 / dX, d e1 / dX                         = JP[2..4], JP[5..7]
  double ja[9], jb[9];  // d e0 / d(f, u0, v0, t, w), d e1 / d(...)     = JC[2..10], JC[11..19]
};
// One division per observation (1 / r): the per-camera quotients 1 / f, u0 / f0, v0 / f0, 1 / f0 come
// with the table row (cam_prep_kernel), and 1 / r^2 = (1 / r)^2.
__device__ __forceinline__ void obs_jacobian(const double* T, double x0, double x1, double x2, ObsJacobian& J) {
  const double gp0 = T[0], gp1 = T[1], gp2 = T[2];
  const double gq0 = T[3], gq1 = T[4], gq2 = T[5];
  const double gr0 = T[6], gr1 = T[7], gr2 = T[8];
  const double inv_f = T[12], uf = T[13], vf = T[14], inv_f0 = T[15];
  const double d0 = x0 - T[9], d1 = x1 - T[10], d2 = x2 - T[11];
  const double p = fma(gp2, d2, fma(gp1, d1, __dmul_rn(gp0, d0)));
  const double q = fma(gq2, d2, fma(gq1, d1, __dmul_rn(gq0, d0)));
  const double r = fma(gr2, d2, fma(gr1, d1, __dmul_rn(gr0, d0)));
  const double ir = 1.0 / r;
  J.p = p; J.q = q; J.r = r; J.ir = ir; J.inv_f0 = inv_f0;
  // a_theta = r dp/dtheta - p dr/dtheta, b_theta = r dq/dtheta - q dr/dtheta; J = (a, b) / r^2
  const double ir2 = __dmul_rn(ir, ir);
  const double a0 = fma(r, gp0, -__dmul_rn(p, gr0)), a1 = fma(r, gp1, -__dmul_rn(p, gr1)),
               a2 = fma(r, gp2, -__dmul_rn(p, gr2));  // :450
  const double b0 = fma(r, gq0, -__dmul_rn(q, gr0)), b1 = fma(r, gq1, -__dmul_rn(q, gr1)),
               b2 = fma(r, gq2, -__dmul_rn(q, gr2));  // :459
  const double af = __dmul_rn(r, __dmul_rn(fma(-uf, r, p), inv_f));  // :336
  const double bf = __dmul_rn(r, __dmul_rn(fma(-vf, r, q), inv_f));  // :337
  const double au = __dmul_rn(r, __dmul_rn(r, inv_f0));              // :350-356
  // rotation: d(p, q, r) / dw = grad x (X - t) (:391-396)  =>  a_w = a_X x d, b_w = b_X x d
  const double aw0 = fma(a1, d2, -__dmul_rn(a2, d1)), aw1 = fma(a2, d0, -__dmul_rn(a0, d2)),
               aw2 = fma(a0, d1, -__dmul_rn(a1, d0));
  const double bw0 = fma(b1, d2, -__dmul_rn(b2, d1)), bw1 = fma(b2, d0, -__dmul_rn(b0, d2)),
               bw2 = fma(b0, d1, -__dmul_rn(b1, d0));
  J.ax[0] = __dmul_rn(a0, ir2); J.ax[1] = __dmul_rn(a1, ir2); J.ax[2] = __dmul_rn(a2, ir2);
  J.bx[0] = __dmul_rn(b0, ir2); J.bx[1] = __dmul_rn(b1, ir2); J.bx[2] = __dmul_rn(b2, ir2);
  // camera row a: f, u0, v0, t (3) = -a_X (:368-376), w (3); row b likewise
  J.ja[0] = __dmul_rn(af, ir2); J.ja[1] = __dmul_rn(au, ir2); J.ja[2] = 0.0;
  J.ja[3] = -J.ax[0]; J.ja[4] = -J.ax[1]; J.ja[5] = -J.ax[2];
  J.ja[6] = __dmul_rn(aw0, ir2); J.ja[7] = __dmul_rn(aw1, ir2); J.ja[8] = __dmul_rn(aw2, ir2);
  J.jb[0] = __dmul_rn(bf, ir2); J.jb[1] = 0.0; J.jb[2] = J.ja[1];
  J.jb[3] = -J.bx[0]; J.jb[4] = -J.bx[1]; J.jb[5] = -J.bx[2];
  J.jb[6] = __dmul_rn(bw0, ir2); J.jb[7] = __dmul_rn(bw1, ir2); J.jb[8] = __dmul_rn(bw2, ir2);
}
// Squared reprojection residual of one observation (:666-677), the same residual expression as the
// linearisation's (one division): cost kernels and the trial cost of the point update.
__device__ __forceinline__ double obs_cost(const double* T, double x0, double x1, double x2, double mx, double my) {
  const double d0 = x0 - T[9], d1 = x1 - T[10], d2 = x2 - T[11];
  const double p = fma(T[2], d2, fma(T[1], d1, __dmul_rn(T[0], d0)));
  const double q = fma(T[5], d2, fma(T[4], d1, __dmul_rn(T[3], d0)));
  const double r = fma(T[8], d2, fma(T[7], d1, __dmul_rn(T[6], d0)));
  const double ir = 1.0 / r, inv_f0 = T[15];
  const double e0 = fma(p, ir, -__dmul_rn(mx, inv_f0));
  const double e1 = fma(q, ir, -__dmul_rn(my, inv_f0));
  return fma(e1, e1, __dmul_rn(e0, e0));
}
// residual of the linearisation (:445, :454): e = (p, q) / r - (x, y) / f0
__device__ __forceinline__ void obs_residual(const ObsJacobian& J, double mx, double my, double& e0, double& e1) {
  e0 = fma(J.p, J.ir, -__dmul_rn(mx, J.inv_f0));
  e1 = fma(J.q, J.ir, -__dmul_rn(my, J.inv_f0));
}
#endif

#ifdef __CUDACC__
// T = 2 Jx L^-T (2 x 3) from the point-side rows and m = L^-1 (lower), and one entry of
// Y = Jc^T T (reference :128-132 through the Cholesky factor): pinned like obs_jacobian, K2b writes
// Y with these and the dense point update re-derives the same bits.
__device__ __forceinline__ void scaled_point_rows(const double* ax, const double* bx, double m00, double m10,
                                                  double m11, double m20, double m21, double m22, double* ta,
                                                  double* tb) {
  ta[0] = 2.0 * __dmul_rn(ax[0], m00);
  ta[1] = 2.0 * fma(ax[1], m11, __dmul_rn(ax[0], m10));
  ta[2] = 2.0 * fma(ax[2], m22, fma(ax[1], m21, __dmul_rn(ax[0], m20)));
  tb[0] = 2.0 * __dmul_rn(bx[0], m00);
  tb[1] = 2.0 * fma(bx[1], m11, __dmul_rn(bx[0], m10));
  tb[2] = 2.0 * fma(bx[2], m22, fma(bx[1], m21, __dmul_rn(bx[0], m20)));
}
__device__ __forceinline__ double y_entry(double ja, double jb, double ta, double tb) {
  return fma(ja, ta, __dmul_rn(jb, tb));
}
// acc += x0 y0 + x1 y1 as two chained FMAs, pinned: the block sums of K2a / the camera blocks, stored
// rows or re-derived
__device__ __forceinline__ double pair_accumulate(double acc, double x0, double y0, double x1, double y1) {
  return fma(x1, y1, fma(x0, y0, acc));
}
#endif

// Grid of a kernel whose blocks loop over `items` work units with a stride of the grid: at most
// `cap` blocks, and every block gets the same number of units (to within one) -- with the plain
// min(items, cap) a count just above the cap gives a few blocks two units and everybody else one,
// i.e. a second pass at a few percent occupancy (C2: 1250 point groups on 1184 blocks).
inline int balanced_blocks(int64_t items, int64_t cap) {
  if (items <= cap) return (int)(items > 0 ? items : 1);
  const int64_t rounds = (items + cap - 1) / cap;
  return (int)((items + rounds - 1) / rounds);
}

// kernel launchers implemented in the .cu files (each returns a ba_status)
int launch_cam_prep(ba_engine* e, int which, cudaStream_t s);
int launch_cost(ba_engine* e, int which, int slot, cudaStream_t s);
int launch_k1(ba_engine* e, cudaStream_t s, bool conditional, bool force_rows = false);
int launch_k2a(ba_engine* e, cudaStream_t s, bool conditional);
int launch_camera_blocks(ba_engine* e, cudaStream_t s, bool conditional);
int launch_k2b(ba_engine* e, bool conditional, double c_host, cudaStream_t s);
bool dense_matrix_free(const ba_engine* e);  // dense K2b / point update re-derive the Jacobian rows
int launch_k3(ba_engine* e, bool conditional, cudaStream_t s);
int syrk_plan_engine(ba_engine* e);
int syrk_emu_info(int64_t k_pad, int32_t* moduli, int* n_moduli, int* bits);
int syrk_feed_is_tma();  // 1: the 128-tile SYRK is fed by TMA + mbarriers, 0: by cp.async (BA_SYRK_NO_TMA)
// Gram matrix P = Yt^T Yt of a k-major operand outside an engine (k3_schur_syrk.cu)
struct GramWorkspace {
  int n_pad = 0, num_sms = 0, n_items = 0, n_tiles = 0;
  int64_t k_pad = 0;
  SyrkItem* items = nullptr;
  int* tile_first = nullptr;
  int* tile_items = nullptr;
  double* Spart = nullptr;
};
int gram_prepare(GramWorkspace* ws, int n_pad, int64_t k_pad, int num_sms, cudaStream_t s);
int gram_launch(const GramWorkspace* ws, const double* Yt, double* P, cudaStream_t s);
void gram_release(GramWorkspace* ws, cudaStream_t s);
int syrk_plan_selftest(int n_cams, int64_t n_points, int tile, int num_sms, int* n_items, int* n_tiles,
                       double* makespan_rows, double* ideal_rows);
int launch_assemble(ba_engine* e, bool conditional, double c_host, cudaStream_t s);
int launch_cholesky_solve(ba_engine* e, bool conditional, cudaStream_t s);
// How the rank-256 trailing updates of a sharded run's (replicated) Cholesky are divided over
// the ranks: tile row g of the global 128-tile grid belongs to rank g % world; the owner updates
// its tiles only and stores those within `push_cols` columns of the update's origin -- the next
// block column, which every rank's panels read -- into every rank's S over NVLink.
struct CholSplit {
  int rank = 0, world = 1;  // world == 1: every rank updates everything (no split)
  int push_cols = 0;
  double* S_peer[kMaxRanks] = {};
};
int launch_chol_wide_update(double* S, int ld, int n_rows, int t0, const double* Lt, int depth,
                            const ba_lm_state* ctl, cudaStream_t s, const CholSplit* split);
void comm_chol_split(ba_engine* e, CholSplit* out);
int launch_comm_chol_sync(ba_engine* e, bool conditional, cudaStream_t s);
int launch_update_trial(ba_engine* e, bool conditional, cudaStream_t s);
int launch_decide(ba_engine* e, cudaStream_t s);
int launch_lm_begin(ba_engine* e, double scale, double tol, int max_iter, int max_retries,
                    cudaStream_t s);
int build_camera_major_index(ba_engine* e, cudaStream_t s);
int build_pair_index(ba_engine* e, cudaStream_t s);
int launch_schur_sparse(ba_engine* e, const ba_lm_state* ctl, cudaStream_t s);
int fp64_peak(int device, int use_dmma, double* tflops);
int launch_comm_allreduce_red(ba_engine* e, bool conditional, cudaStream_t s);
int launch_comm_allreduce_cost(ba_engine* e, int slot, bool conditional, cudaStream_t s);
void comm_free(ba_engine* e);

}  // namespace ba
