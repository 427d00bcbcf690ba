// K3: Schur-complement products  P = sum_j Y_j Y_j^T  (and the rhs row sum_j z_j^T Y_j^T).
//
// Replaces reference lib/bundle_adjustment.py:132-143 -- `(FtEinv @ matF).sum(axis=0)`, which
// materialises an (N, n, n) temporary, and `(FtEinv @ delta_X_E).sum(axis=0)`.
//
// Dense visibility: Y^T is stored k-major, Yt[3N_pad][ld] (ld = n_pad, a multiple of 8), and
// P = Yt^T Yt is a symmetric rank-k update on the FP64 tensor cores (DMMA.8x8x4 through
// mma.sync.m8n8k4.f64; tcgen05 has no f64 kind).  Only lower-triangle tiles are computed; edge
// tiles skip the 8x8 fragments beyond n_pad.  K (= 3 x points) is split over many more CTAs than
// SM slots so the hardware block scheduler evens out the tail, and the per-split partial tiles are
// summed in a fixed order (deterministic; no FP64 atomics).  z_j occupies column `rhs_row` of
// Yt, so row `rhs_row` of P is the rhs term for free.
//
// Two kernels, one per tile size: 128-tiles (syrk_tma_kernel, one CTA per SM) are fed by TMA
// tensor copies (see "128-tiles fed by TMA" below); 64-tiles (syrk_dmma_kernel, four CTAs per SM)
// by cp.async (LDGSTS) 16-byte copies, 3 stages of KC k-rows, shared-memory rows padded to TILE+4
// doubles (stride = 4 mod 16: the 8-byte fragment loads of a half-warp hit 16 distinct bank pairs
// -- ncu: 0 bank conflicts).
//
// Compute roofline (FP64 tensor): algorithmic flops = 3N * n (n + 1), n = 9M - 7.
//
// Large dense products (C3: n_pad^2 k_pad = 9.8e11) run instead on the INT8 tensor cores, FP64-accurate
// through the modular Ozaki scheme (see "FP64-accurate product on the INT8 tensor cores" below):
// emu_residue_kernel turns Yt into 16 int8 residue planes (with the column maxima K2b gathers as it
// writes Yt), syrk_i8_pair_kernel (tcgen05.mma kind::i8 on pairs of SMs) forms one SYRK per modulus,
// emu_reconstruct_kernel lifts the exact integer products back to FP64 into P.  The DMMA kernels stay for smaller products (C2), the Cholesky's
// trailing updates and the projective-depth Gram matrix.  BA_SYRK_EMU=0|1 overrides the size rule.
//
// Sparse visibility: see k3_schur_sparse.cu (output-stationary, no atomics).
#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <functional>
#include <mutex>
#include <optional>
#include <queue>
#include <vector>

#include "ba_common.cuh"

namespace ba {

constexpr int kStages = 3;

__device__ __forceinline__ void tile_from_linear(int t, int& ti, int& tj) {
  ti = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while ((ti + 1) * (ti + 2) / 2 <= t) ++ti;
  while (ti * (ti + 1) / 2 > t) --ti;
  tj = t - ti * (ti + 1) / 2;
}

// Division of a trailing update over the ranks of a sharded run (see CholSplit): the CTA of a tile
// row this rank does not own exits at once; tiles that start within push_cols columns are also
// stored into every other rank's matrix (peer[q] = that rank's S at the update's origin).
struct SubSplit {
  int rank, world, tile_row0, push_cols;
  double* peer[kMaxRanks];
};

// Epilogue of one accumulator pair at tile-local (rl, cl), cl even: into the item's partial tile
// (`part` points at it), or (SUB) subtracted in place from the lower triangle of S (`part`), with
// the peer stores of a divided update.
template <int TILE, bool SUB>
__device__ __forceinline__ void syrk_store_pair(double v0, double v1, int ti, int tj, int rl, int cl, int ld,
                                                int n_store, double* __restrict__ part, const SubSplit& sp) {
  if (SUB) {
    const int r = ti * TILE + rl, c = tj * TILE + cl;
    if (r >= n_store || c > r) return;
    const size_t off = (size_t)r * ld + c;
    double* p = part + off;
    const bool push = sp.world > 1 && tj * TILE < sp.push_cols;
    if (c + 1 <= r) {
      double2 v = *reinterpret_cast<double2*>(p);
      v.x -= v0;
      v.y -= v1;
      *reinterpret_cast<double2*>(p) = v;
      if (push)
        for (int q = 0; q < sp.world; ++q)
          if (q != sp.rank) *reinterpret_cast<double2*>(sp.peer[q] + off) = v;
    } else {
      const double v = *p - v0;
      *p = v;
      if (push)
        for (int q = 0; q < sp.world; ++q)
          if (q != sp.rank) sp.peer[q][off] = v;
    }
  } else {
    // `part` is the item's own partial tile
    *reinterpret_cast<double2*>(part + (size_t)rl * TILE + cl) = make_double2(v0, v1);
  }
}

// 64-tiles: 2 x 2 warps, each owning a 32 x 32 sub-tile, KC k-rows per stage; four CTAs per SM.
constexpr int kDmmaTile = 64, kDmmaWR = 2, kDmmaWC = 2, kDmmaKC = 16;
constexpr int kDmmaThreads = kDmmaWR * kDmmaWC * 32;
constexpr size_t kDmmaSmemBytes = (size_t)2 * kStages * kDmmaKC * (kDmmaTile + 4) * sizeof(double);

// TILE x TILE output tile per CTA; WR x WC warps, each owning a (TILE/WR) x (TILE/WC) sub-tile.
// SUB = false: the tile of this split is written to part[split][tile] (Schur product).
// SUB = true:  one split; the tile is subtracted in place from the lower triangle of the n_store x
//              n_store matrix `part` (leading dimension ld) -- the rank-k trailing update of the
//              blocked Cholesky (k4_cholesky.cu), where Yt is the k-major copy of a block column.
template <bool SUB>
__global__ void __launch_bounds__(kDmmaThreads)
syrk_dmma_kernel(const double* __restrict__ Yt, int ld, int n_valid, int64_t n_chunks,
                 const SyrkItem* __restrict__ items, double* __restrict__ part,
                 const ba_lm_state* ctl, int n_store, SubSplit sp) {
  if (ctl && ctl->done) return;
  constexpr int TILE = kDmmaTile, WR = kDmmaWR, WC = kDmmaWC, KC = kDmmaKC;
  constexpr int NT = kDmmaThreads;
  constexpr int LDS = TILE + 4;
  constexpr int WM = TILE / WR, WN = TILE / WC;
  constexpr int FM = WM / 8, FN = WN / 8;
  constexpr int CPR = TILE / 2;               // 16-byte pieces per row
  constexpr int PER_THREAD = KC * CPR / NT;   // pieces per thread per operand per stage
  static_assert(KC * CPR % NT == 0, "stage copy must divide evenly");
  extern __shared__ __align__(16) double smem[];

  // work item: a tile and a range of k-chunks (Schur product), or the whole depth of tile
  // blockIdx.x (trailing update)
  int ti, tj;
  int64_t c_lo, c_hi;
  if (SUB) {
    tile_from_linear(blockIdx.x, ti, tj);
    if (sp.world > 1 && (sp.tile_row0 + ti) % sp.world != sp.rank) return;  // another rank's tile row
    c_lo = 0;
    c_hi = n_chunks;
  } else {
    const SyrkItem it = items[blockIdx.x];
    ti = it.ti; tj = it.tj; c_lo = it.c_lo; c_hi = it.c_hi;
  }
  const bool diag = ti == tj;
  const int nk = (int)(c_hi > c_lo ? c_hi - c_lo : 0);

  double* sA = smem;                                // [stage][KC][LDS]
  double* sB = smem + (size_t)kStages * KC * LDS;   // unused for diagonal tiles

  // per-thread copy slots: fixed (row, piece) positions; columns beyond n_valid are zero-filled
  int soff[PER_THREAD];
  int goffA[PER_THREAD], goffB[PER_THREAD];
  int bytesA[PER_THREAD], bytesB[PER_THREAD];
#pragma unroll
  for (int u = 0; u < PER_THREAD; ++u) {
    const int q = threadIdx.x + u * NT;
    const int row = q / CPR, pc = q % CPR;
    soff[u] = row * LDS + 2 * pc;
    const int ca = ti * TILE + 2 * pc, cb = tj * TILE + 2 * pc;
    bytesA[u] = ca < n_valid ? 16 : 0;
    bytesB[u] = cb < n_valid ? 16 : 0;
    goffA[u] = row * ld + (ca < n_valid ? ca : 0);
    goffB[u] = row * ld + (cb < n_valid ? cb : 0);
  }
  const double* gbase = Yt + (size_t)c_lo * KC * ld;

  auto load_stage = [&](int stage, int chunk) {
    const double* g = gbase + (size_t)chunk * KC * ld;
    double* da = sA + (size_t)stage * KC * LDS;
    double* db = sB + (size_t)stage * KC * LDS;
#pragma unroll
    for (int u = 0; u < PER_THREAD; ++u) {
      cp_async16_zfill(da + soff[u], g + goffA[u], bytesA[u]);
      if (!diag) cp_async16_zfill(db + soff[u], g + goffB[u], bytesB[u]);
    }
  };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Sub-tile of this warp.  Off the diagonal: row-major over the WR x WC grid.  On a diagonal
  // tile only the WR (WR + 1) / 2 sub-tiles on or below the diagonal are needed (nothing above
  // the diagonal is read anywhere); they are dealt to warps 0, 1, 2, ... -- consecutive warps sit
  // on different scheduler partitions -- and the remaining warps only help with the copies.
  int wr = warp / WC, wc = warp % WC;
  bool live = true;
  if (diag && WR == WC) {
    live = warp < WR * (WR + 1) / 2;
    if (live) {
      wr = 0;
      while ((wr + 1) * (wr + 2) / 2 <= warp) ++wr;
      wc = warp - wr * (wr + 1) / 2;
    }
  }
  const int row0 = wr * WM + (lane >> 2);
  const int col0 = wc * WN + (lane >> 2);
  const int kq = lane & 3;

  // fragments of this warp inside the valid part of P (n_valid is a multiple of 8)
  int vm = 0, vn = 0;
#pragma unroll
  for (int i = 0; i < FM; ++i) vm += (ti * TILE + wr * WM + 8 * i) < n_valid;
#pragma unroll
  for (int j = 0; j < FN; ++j) vn += (tj * TILE + wc * WN + 8 * j) < n_valid;
  if (!live) vm = 0;
  const bool full = vm == FM && vn == FN;

  double acc[FM][FN][2];
#pragma unroll
  for (int i = 0; i < FM; ++i)
#pragma unroll
    for (int j = 0; j < FN; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

#pragma unroll
  for (int s = 0; s < kStages - 1; ++s) {
    if (s < nk) load_stage(s, s);
    cp_async_commit();
  }
  for (int kc = 0; kc < nk; ++kc) {
    cp_async_wait<kStages - 2>();
    __syncthreads();
    const int nxt = kc + kStages - 1;
    if (nxt < nk) load_stage(nxt % kStages, nxt);
    cp_async_commit();
    const double* a = sA + (size_t)(kc % kStages) * KC * LDS;
    const double* b = diag ? a : sB + (size_t)(kc % kStages) * KC * LDS;
    if (full) {
#pragma unroll
      for (int kk = 0; kk < KC; kk += 4) {
        double fa[FM], fb[FN];
#pragma unroll
        for (int i = 0; i < FM; ++i) fa[i] = a[(kk + kq) * LDS + row0 + 8 * i];
#pragma unroll
        for (int j = 0; j < FN; ++j) fb[j] = b[(kk + kq) * LDS + col0 + 8 * j];
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
      }
    } else if (vm > 0 && vn > 0) {
#pragma unroll
      for (int kk = 0; kk < KC; kk += 4) {
        double fa[FM], fb[FN];
#pragma unroll
        for (int i = 0; i < FM; ++i) fa[i] = a[(kk + kq) * LDS + row0 + 8 * i];
#pragma unroll
        for (int j = 0; j < FN; ++j) fb[j] = b[(kk + kq) * LDS + col0 + 8 * j];
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j)
            if (i < vm && j < vn) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
      }
    }
  }
  cp_async_wait<0>();

  const int orow = wr * WM + (lane >> 2);
  const int ocol = wc * WN + 2 * (lane & 3);
  if (!live) return;  // the sub-tiles above the diagonal of a diagonal tile are never read
  // partial tile of this item: part[item][TILE][TILE]
  double* const out = SUB ? part : part + (size_t)blockIdx.x * TILE * TILE;
#pragma unroll
  for (int i = 0; i < FM; ++i)
#pragma unroll
    for (int j = 0; j < FN; ++j)
      syrk_store_pair<TILE, SUB>(acc[i][j][0], acc[i][j][1], ti, tj, orow + 8 * i, ocol + 8 * j, ld, n_store, out, sp);
}

// ---- 128-tiles fed by TMA ------------------------------------------------------------------------
// The product with a Blackwell-native operand feed.  ncu on a cp.async-fed 128-tile kernel at C3: every
// chunk starts with all 16 warps issuing their LDGSTS (128 warp instructions, ~8 LSU cycles each)
// right behind the block barrier, and the fragment loads of the chunk's first k-steps queue behind
// them in the same LSU pipe -- ~1000 of every 8192 cycles the FP64 tensor pipes wait (tiles without
// ragged edges ran at 85 % of the DMMA peak).  Here the copies are tensor copies
// (cp.async.bulk.tensor.2d -> SASS UTMALDG): ONE instruction per operand and chunk, issued by one
// elected thread; the TMA engine writes shared memory and completes the stage's `full` mbarrier
// with the byte count, no LSU copy instruction and no block barrier is involved.  All 16 warps wait
// on `full`, run their DMMAs, and release the stage through the `empty` mbarrier (one arrival per
// warp); the elected thread refills a stage one chunk after it was consumed, when every warp has
// long moved on, so it practically never waits for `empty`.
//
// Shared-memory layout per stage and operand: [KC k-rows][132 doubles] -- the box is 132 columns
// wide, four more than the tile, so that the dense rows the TMA unit writes have the stride (1056 B
// = 8 banks mod 32) that makes the DMMA fragment loads conflict-free: the 16 lanes of a half-warp
// (4 k-rows x 4 columns) hit 16 distinct bank pairs.  (The first version used one box of 8 columns
// per column group, [group][k][8]: ncu showed 2.2e9 bank conflicts -- k-rows 64 B apart collide two
// by two -- and 32 UTMALDG per chunk.)  Columns beyond n_valid lie outside the tensor and are
// zero-filled by the TMA unit.
//
// Ragged last tile row.  With n_pad = 1808 (200 cameras) the last tile row has 16 valid rows: as
// tiles of their own those 15 thin tiles cost 4.9 % of the kernel for 1.9 % of its flops (each is
// bound by the latency of the three-stage ring, not by its DMMAs).  When at most kTmaTallRows rows
// are left over, the tiles of the row above are "tall": their A box is 148 columns wide (for every
// tile -- the 16 extra columns cost nothing measurable), and every warp computes two more fragments
// -- fragment row 16 or 17 against two of the B fragments it already holds.  Only the two thin
// tiles next to the diagonal remain items of their own.
constexpr int kTmaTile = 128, kTmaKC = 32, kTmaStages = 3, kTmaTallRows = 16;
constexpr int kTmaLda = kTmaTile + kTmaTallRows + 4, kTmaLdb = kTmaTile + 4;   // 148, 132: both = 8 banks mod 32
constexpr int kTmaThreads = 512;
constexpr int kTmaADoubles = kTmaKC * kTmaLda, kTmaBDoubles = kTmaKC * kTmaLdb;
constexpr unsigned kTmaABytes = kTmaADoubles * (unsigned)sizeof(double);    // 37 888
constexpr unsigned kTmaBBytes = kTmaBDoubles * (unsigned)sizeof(double);    // 33 792
constexpr unsigned kTmaStageBytes = kTmaABytes + kTmaBBytes;                // 71 680
constexpr size_t kTmaSmemBytes = (size_t)kTmaStages * kTmaStageBytes + 128 /*alignment*/ + 64 /*barriers*/;

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Wait for the phase of the given parity.  The spin is bounded: a copy that never lands (a wrong
// byte count, a bad descriptor) becomes a trap -- a failed launch -- instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  unsigned ok = 0;
  for (unsigned spins = 0; !ok; ++spins) {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (!ok && spins > (1u << 26)) __trap();
  }
}
__device__ __forceinline__ void tma_load_2d(unsigned dst, const CUtensorMap* map, int c0, int c1, unsigned bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}

// One CTA runs one work item: a tile and a range of k-chunks (Schur product: items[blockIdx.x], its
// partial tile goes to slot blockIdx.x), or the whole depth of tile blockIdx.x (trailing update).
// The elected thread fills the three-stage ring with the item's first chunks and, before chunk kc
// is computed, refills the stage of chunk kc - 1 with chunk kc + 2.
template <bool SUB>
__global__ void __launch_bounds__(kTmaThreads, 1)
syrk_tma_kernel(const __grid_constant__ CUtensorMap tmapA, const __grid_constant__ CUtensorMap tmapB, int ld,
                int n_valid, int64_t n_chunks, const SyrkItem* __restrict__ items, double* __restrict__ part,
                const ba_lm_state* ctl, int n_store, SubSplit sp) {
  if (ctl && ctl->done) return;
  constexpr int TILE = kTmaTile, KC = kTmaKC, LDA = kTmaLda, LDB = kTmaLdb, WR = 4, WC = 4;
  constexpr int WM = TILE / WR, WN = TILE / WC, FM = WM / 8, FN = WN / 8;
  extern __shared__ unsigned char smem_raw[];

  int ti, tj, c_lo = 0, nk;
  bool tall = false;
  if (SUB) {
    tile_from_linear(blockIdx.x, ti, tj);
    if (sp.world > 1 && (sp.tile_row0 + ti) % sp.world != sp.rank) return;  // another rank's tile row
    nk = (int)n_chunks;
  } else {
    const SyrkItem it = items[blockIdx.x];
    ti = it.ti; tj = it.tj; c_lo = it.c_lo; nk = it.c_hi > it.c_lo ? it.c_hi - it.c_lo : 0; tall = it.slot2 >= 0;
  }
  const bool diag = ti == tj;

  // carve shared memory: operand stages (128-byte aligned for the TMA unit), then the mbarriers
  const unsigned base = (smem_u32(smem_raw) + 127u) & ~127u;
  const double* stages = reinterpret_cast<const double*>(smem_raw + (base - smem_u32(smem_raw)));
  constexpr int kStageDoubles = kTmaADoubles + kTmaBDoubles;
  const unsigned bars = base + kTmaStages * kTmaStageBytes;
  auto full_bar = [&](int st) { return bars + 8u * st; };
  auto empty_bar = [&](int st) { return bars + 8u * (kTmaStages + st); };

  auto issue = [&](int kc) {  // thread 0 only: chunk kc of the item into stage kc % kTmaStages
    const int st = kc % kTmaStages;
    const unsigned dst = base + (unsigned)st * kTmaStageBytes;
    const int row = (c_lo + kc) * KC;
    mbar_arrive_expect_tx(full_bar(st), kTmaABytes + (diag ? 0u : kTmaBBytes));
    tma_load_2d(dst, &tmapA, ti * TILE, row, full_bar(st));
    if (!diag) tma_load_2d(dst + kTmaABytes, &tmapB, tj * TILE, row, full_bar(st));
  };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int st = 0; st < kTmaStages; ++st) {
      mbar_init(full_bar(st), 1);
      mbar_init(empty_bar(st), kTmaThreads / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int kc = 0; kc < kTmaStages && kc < nk; ++kc) issue(kc);
  }
  __syncthreads();
  // Before chunk kc is computed the elected thread refills the stage of chunk kc - 1 with chunk
  // kc + kTmaStages - 1 (every warp is done with chunk kc - 1 or about to be: the wait on `empty`
  // is short).
  auto refill = [&](int kc) {
    if (warp == 0) {
      if (lane == 0 && kc >= 1 && kc + kTmaStages - 1 < nk) {
        mbar_wait(empty_bar((kc - 1) % kTmaStages), ((kc - 1) / kTmaStages) & 1u);
        issue(kc + kTmaStages - 1);
      }
      __syncwarp();
    }
  };
  const int kq = lane & 3;
  double* const slot_part = SUB ? part : part + (size_t)blockIdx.x * TILE * TILE;

  if (diag) {
    // Diagonal tile: only the 136 fragments (8 x 8) on or below the diagonal of the 16 x 16
    // fragment grid are needed.  Fragment rows r and 15 - r together hold 17 of them; the pair is
    // shared by two warps, one taking nine fragments (row 15 - r, columns 0..8), the other eight
    // (the rest of row 15 - r and all of row r); which warp of a pair takes nine alternates so
    // that every scheduler partition (warp % 4) carries 34 fragments per k-step.
    const int pr = warp >> 1;
    const bool nine = (((warp & 1) ^ ((warp >> 2) & 1)) == 0);
    const int r_hi = 15 - pr, r_lo = pr;
    const int n_hi = nine ? 9 : 7 - pr;        // fragments this warp takes from row r_hi
    const int c_hi0 = nine ? 0 : 9;            // ... starting at this column
    const int nfr = nine ? 9 : 8;
    const int frag_rows_valid = (n_valid - ti * TILE + 7) / 8;  // ragged last tile
    int boffj[9];
    bool usej[9];
    bool any = false;
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      const bool hi = j < n_hi;
      const int rf = hi ? r_hi : r_lo;
      const int cf = hi ? c_hi0 + j : j - n_hi;
      usej[j] = j < nfr && rf < frag_rows_valid;
      any |= usej[j];
      boffj[j] = kq * LDA + 8 * cf + (lane >> 2);
    }
    const int aoff_hi = kq * LDA + 8 * r_hi + (lane >> 2);
    const int aoff_lo = kq * LDA + 8 * r_lo + (lane >> 2);
    double dacc[9][2];
#pragma unroll
    for (int j = 0; j < 9; ++j) dacc[j][0] = dacc[j][1] = 0.0;
    for (int kc = 0; kc < nk; ++kc) {
      refill(kc);
      const int st = kc % kTmaStages;
      mbar_wait(full_bar(st), (kc / kTmaStages) & 1u);
      const double* a = stages + (size_t)st * kStageDoubles;
      if (any) {
#pragma unroll
        for (int kk = 0; kk < KC; kk += 4) {
          const double fa_hi = a[aoff_hi + kk * LDA], fa_lo = a[aoff_lo + kk * LDA];
          double fb[9];
#pragma unroll
          for (int j = 0; j < 9; ++j) fb[j] = a[boffj[j] + kk * LDA];
#pragma unroll
          for (int j = 0; j < 9; ++j)
            if (usej[j]) dmma884(dacc[j][0], dacc[j][1], j < n_hi ? fa_hi : fa_lo, fb[j]);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty_bar(st));
    }
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      if (!usej[j]) continue;
      const bool hi = j < n_hi;
      syrk_store_pair<TILE, SUB>(dacc[j][0], dacc[j][1], ti, ti, 8 * (hi ? r_hi : r_lo) + (lane >> 2),
                                 8 * (hi ? c_hi0 + j : j - n_hi) + 2 * (lane & 3), ld, n_store, slot_part, sp);
    }
    return;
  }

  // (A column-per-warp mapping for the thin tiles of a ragged last tile row was tried and dropped:
  // with only 2 of 16 fragment rows to compute, the warps outrun the three-stage TMA ring and wait
  // for every chunk -- C3 went from 28.8 to 31.1 ms.  Such rows are folded into tall tiles instead.)
  const int wr = warp / WC, wc = warp % WC;
  int vm = 0, vn = 0;
#pragma unroll
  for (int i = 0; i < FM; ++i) vm += (ti * TILE + wr * WM + 8 * i) < n_valid;
#pragma unroll
  for (int j = 0; j < FN; ++j) vn += (tj * TILE + wc * WN + 8 * j) < n_valid;
  const bool full = vm == FM && vn == FN;
  const int aoff = kq * LDA + wr * WM + (lane >> 2);
  const int boff = kq * LDB + wc * WN + (lane >> 2);
  // tall item: this warp's two extra fragments -- fragment row 16 + (wr & 1) of A against its B
  // fragments 2 (wr >> 1) and 2 (wr >> 1) + 1
  const int xoff = kq * LDA + TILE + 8 * (wr & 1) + (lane >> 2);
  const int xj = 2 * (wr >> 1);
  const bool xvalid = tall && (ti + 1) * TILE + 8 * (wr & 1) < n_valid;

  double acc[FM][FN][2], xacc[2][2];
#pragma unroll
  for (int i = 0; i < FM; ++i)
#pragma unroll
    for (int j = 0; j < FN; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  xacc[0][0] = xacc[0][1] = xacc[1][0] = xacc[1][1] = 0.0;

  for (int kc = 0; kc < nk; ++kc) {
    refill(kc);
    const int st = kc % kTmaStages;
    mbar_wait(full_bar(st), (kc / kTmaStages) & 1u);
    const double* a = stages + (size_t)st * kStageDoubles + aoff;
    const double* b = stages + (size_t)st * kStageDoubles + kTmaADoubles + boff;
    if (full && xvalid) {
      const double* x = stages + (size_t)st * kStageDoubles + xoff;
#pragma unroll
      for (int kk = 0; kk < KC; kk += 4) {
        double fa[FM], fb[FN];
#pragma unroll
        for (int i = 0; i < FM; ++i) fa[i] = a[kk * LDA + 8 * i];
#pragma unroll
        for (int j = 0; j < FN; ++j) fb[j] = b[kk * LDB + 8 * j];
        const double fx = x[kk * LDA];
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
        dmma884(xacc[0][0], xacc[0][1], fx, xj == 0 ? fb[0] : fb[2]);
        dmma884(xacc[1][0], xacc[1][1], fx, xj == 0 ? fb[1] : fb[3]);
      }
    } else if (full) {
#pragma unroll
      for (int kk = 0; kk < KC; kk += 4) {
        double fa[FM], fb[FN];
#pragma unroll
        for (int i = 0; i < FM; ++i) fa[i] = a[kk * LDA + 8 * i];
#pragma unroll
        for (int j = 0; j < FN; ++j) fb[j] = b[kk * LDB + 8 * j];
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
      }
    } else if (vm > 0 && vn > 0) {
#pragma unroll
      for (int kk = 0; kk < KC; kk += 4) {
        double fa[FM], fb[FN];
#pragma unroll
        for (int i = 0; i < FM; ++i) fa[i] = a[kk * LDA + 8 * i];
#pragma unroll
        for (int j = 0; j < FN; ++j) fb[j] = b[kk * LDB + 8 * j];
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j)
            if (i < vm && j < vn) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty_bar(st));  // this warp has read the stage
  }

  const int orow = wr * WM + (lane >> 2);
  const int ocol = wc * WN + 2 * (lane & 3);
#pragma unroll
  for (int i = 0; i < FM; ++i)
#pragma unroll
    for (int j = 0; j < FN; ++j)
      syrk_store_pair<TILE, SUB>(acc[i][j][0], acc[i][j][1], ti, tj, orow + 8 * i, ocol + 8 * j, ld, n_store, slot_part, sp);
  if (xvalid) {
    // the ragged rows below the tile: rows 0.. of the thin tile's partial slot (never with SUB).  The
    // slot is read again here (a volatile load, which is not merged with the first one): kept live
    // through the k-loop it would be spilled at 128 registers.
    const int slot2 = __ldcv(&items[blockIdx.x].slot2);
    double* xp = part + (size_t)slot2 * TILE * TILE + (size_t)(8 * (wr & 1) + (lane >> 2)) * TILE;
#pragma unroll
    for (int e = 0; e < 2; ++e)
      *reinterpret_cast<double2*>(xp + wc * WN + 8 * (xj + e) + 2 * (lane & 3)) = make_double2(xacc[e][0], xacc[e][1]);
  }
}

// P[tile] = sum of the tile's items in a fixed order (ascending k range), restricted to the valid
// part of P and, on diagonal tiles, to the pairs that touch the lower triangle.
template <int TILE>
__global__ void __launch_bounds__(256)
syrk_reduce_kernel(const double* __restrict__ part, const int* __restrict__ tile_first,
                   const int* __restrict__ tile_items, double* __restrict__ P, int ld, int n_valid,
                   const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;
  const int t = blockIdx.x;
  int ti, tj;
  tile_from_linear(t, ti, tj);
  const int first = tile_first[t], cnt = tile_first[t + 1] - first;
  const int* slots = tile_items + first;
  constexpr size_t TT = (size_t)TILE * TILE;
  // blockIdx.y picks a slab of rows of the tile; 4 independent loads in flight per thread
  const int per = TILE * TILE / 2 / gridDim.y;
  for (int q = blockIdx.y * per + threadIdx.x; q < (blockIdx.y + 1) * per; q += blockDim.x) {
    const int r = q / (TILE / 2), c = 2 * (q % (TILE / 2));
    if (ti * TILE + r >= n_valid || tj * TILE + c >= n_valid) continue;
    if (ti == tj && c > r) continue;
    const double* src = part + (size_t)r * TILE + c;
    double2 s = make_double2(0.0, 0.0);
    int sp = 0;
    for (; sp + 4 <= cnt; sp += 4) {
      const double2 v0 = *reinterpret_cast<const double2*>(src + slots[sp] * TT);
      const double2 v1 = *reinterpret_cast<const double2*>(src + slots[sp + 1] * TT);
      const double2 v2 = *reinterpret_cast<const double2*>(src + slots[sp + 2] * TT);
      const double2 v3 = *reinterpret_cast<const double2*>(src + slots[sp + 3] * TT);
      s.x = (((s.x + v0.x) + v1.x) + v2.x) + v3.x;
      s.y = (((s.y + v0.y) + v1.y) + v2.y) + v3.y;
    }
    for (; sp < cnt; ++sp) {
      const double2 v = *reinterpret_cast<const double2*>(src + slots[sp] * TT);
      s.x += v.x;
      s.y += v.y;
    }
    *reinterpret_cast<double2*>(P + (size_t)(ti * TILE + r) * ld + tj * TILE + c) = s;
  }
}

// Local U / dF blocks into the reduce buffer: a sharded run all-reduces one flat buffer.
__global__ void stage_camera_blocks_kernel(int n, const double* __restrict__ src,
                                           double* __restrict__ dst, const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) dst[k] = src[k];
}

// ---- FP64-accurate product on the INT8 tensor cores (Ozaki scheme II) -------------------------------
// P = Yt^T Yt from exact integer products (Ozaki, Uchino, Imamura, "Ozaki Scheme II", 2025):
//  1. every column a is scaled by 2^e_a so that |Yt[k][a]| 2^e_a < 2^b, and rounded to the integer
//     a' = rint(Yt[k][a] 2^e_a) (|a'| <= 2^b <= 2^53: the rounding error is at most 2^-53 of the
//     column's largest entry; a zero column gives a' = 0 and an exactly zero row of P);
//  2. a' is reduced modulo L = 16 pairwise coprime moduli p_i <= 256 into int8 residue planes;
//  3. one int8 SYRK per modulus on tcgen05 (kind::i8, int32 accumulators in tensor memory) gives
//     sum_k a'_k b'_k mod p_i exactly -- int32 is exact over <= 131 071 k-rows, longer k ranges are
//     split into items whose results are reduced mod p_i and summed with integer atomics (exact and
//     order-independent, so P is bit-reproducible);
//  4. Garner's mixed-radix conversion and the symmetric lift recover the integer dot product, exact
//     while k_pad 2^(2b) < prod(p) / 2 (the host picks b accordingly: 53 up to k_pad ~ 2^19.4); it is
//     converted to double by Horner from the most significant digit (16 fused multiply-adds of
//     non-negative terms: relative error <= 16 u = 1.8e-15, exact below 2^53) and scaled by
//     2^-(e_a + e_b), which is exact.
constexpr int kEmuModuli = 16;
constexpr int kEmuTile = 128;     // rows of a residue-sum tile (Pmod) and of one CTA's operand box
constexpr int kEmuPair = 256;     // rows of a work item's tile: M (and full N) of the two-CTA MMA
constexpr int kEmuKB = 128;       // k-rows per pipeline stage: one 128-byte swizzle row of int8
constexpr int kEmuStages = 3;     // x 32 KB (one CTA's half of a pair's operands): the most that leaves room for two CTAs per SM
constexpr int kEmuThreads = 128;  // four warps: one per 32-lane quarter of tensor memory
constexpr unsigned kEmuOpBytes = kEmuTile * kEmuKB;     // 16 384
constexpr unsigned kEmuStageBytes = 2 * kEmuOpBytes;    // 32 768
constexpr size_t kEmuSmemBytes = (size_t)kEmuStages * kEmuStageBytes + 1024 /*alignment*/ + 64 /*barriers*/;
constexpr double kEmuMinWork = 1e11;  // n_pad^2 k_pad from which the emulation is the default
constexpr int kEmuMaxKB = (int)(((1u << 31) - 1) / (128u * 128u) / kEmuKB);  // 1023 k-blocks: |sum| < 2^31
// M = 256, S8 x S8 -> S32, both operands K-major (instruction descriptor of tcgen05.mma); N at bits 17..22
constexpr uint32_t kEmuIdescM256 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kEmuPair >> 4) << 24);

__host__ __device__ constexpr int emu_modulus(int i) {
  constexpr int p[kEmuModuli] = {256, 255, 253, 251, 247, 241, 239, 233, 229, 227, 223, 217, 211, 199, 197, 193};
  return p[i];
}

// Garner's constants: inv[j][i] = p_j^-1 mod p_i (j < i); half[i]: mixed-radix digits of prod(p) / 2
struct EmuConsts {
  int inv[kEmuModuli][kEmuModuli];
  int half[kEmuModuli];
};

// e_a for a column whose largest |entry| has the exponent of the bit pattern `maxbits`: max 2^e_a < 2^b
__device__ __forceinline__ int emu_exponent(unsigned long long maxbits, int b) {
  if (maxbits == 0) return 0;
  return b - 1 - ilogb(__longlong_as_double((long long)maxbits));
}

// Residue planes Yq[i][a][k] (K-major) from Yt[k][a], with the column maxima K2b gathered (colmax).
// A thread converts 16 consecutive k-rows of one column: 16 loads in flight, then for every modulus one
// 16-byte store; the 8 threads of a column in a warp write whole 128-byte lines of a plane row, and its
// loads read 32-byte pieces (4 columns) of 8 k-rows.  Per element, a' = rint(x 2^e_a) is formed once as
// an int64 (two exact power-of-two multiplications: 2^e_a alone is not a normal double for all e_a),
// and biased by 2^55 so that its seven low bytes u_0..u_6 are unsigned digits of a' + 2^55.  Then per
// modulus p, without FP64:
//   f = 2^23 + c_p + sum_k u_k (256^k mod p)   two dp4a; c_p = (-2^23 - 2^55) mod p, so f = a' (mod p),
//                                              and the accumulator starts at the bit pattern of 2^23 + c_p:
//                                              it is f as a float (f < 2^23 + 2^19, exact)
//   q = rint(f / p)                             one FFMA with the float 1 / p and the 1.5 * 2^23 rounding
//                                              constant; exact for every f in range (checked exhaustively
//                                              by tests/test_emu_residue_digits.py) except p = 255,
//                                              which takes q from f - 2^23 (< 2^11) instead
//   r = f - p q                                 one IMAD on the bit patterns; every constant it carries is a
//                                              multiple of 256, so its low byte is that of r in [-127, 127]
// p = 256 is the low byte of a'.  Any representative of a' mod p gives the same residue sums, P is
// unchanged.
constexpr int kResK = 16;                      // k-rows per thread
constexpr int kResTK = 8 * kResK;              // k-rows of a block: one 128-byte line per plane row
constexpr int kResTA = 32;                     // columns of a block: 4 per warp
constexpr int kResThreads = 8 * kResTA;
constexpr float kResRound = 12582912.0f;       // 1.5 * 2^23
constexpr unsigned kResFloat23 = 0x4B000000u;  // bit pattern of 2^23

__host__ __device__ constexpr unsigned emu_pow256_mod(int k, int p) {
  unsigned r = 1;
  for (int i = 0; i < k; ++i) r = r * 256u % (unsigned)p;
  return r;
}
__host__ __device__ constexpr unsigned emu_digit_weights(int k0, int p) {  // bytes 256^(k0 + j) mod p
  return emu_pow256_mod(k0, p) | emu_pow256_mod(k0 + 1, p) << 8 | emu_pow256_mod(k0 + 2, p) << 16 |
         (k0 + 3 < 7 ? emu_pow256_mod(k0 + 3, p) << 24 : 0u);
}
__host__ __device__ constexpr unsigned emu_digit_bias(int p) {  // c_p = (-2^23 - 2^55) mod p
  return (unsigned)((2u * (unsigned)p - emu_pow256_mod(6, p) * 128u % (unsigned)p - (1u << 23) % (unsigned)p) %
                    (unsigned)p);
}

// Low byte: a' mod p_I (lo, hi: the words of a' + 2^55)
template <int I>
__device__ __forceinline__ unsigned emu_residue_byte(unsigned lo, unsigned hi) {
  constexpr int p = emu_modulus(I);
  if constexpr (p == 256) {
    return lo;
  } else {
    constexpr bool small = p == 255;
    const unsigned acc = __dp4a(hi, emu_digit_weights(4, p),
                                __dp4a(lo, emu_digit_weights(0, p), kResFloat23 + emu_digit_bias(p) + (small ? (1u << 23) % p : 0u)));
    float f = __uint_as_float(acc);
    if (small) f = __fadd_rn(f, -8388608.0f);
    const float q = __fmaf_rn(f, 1.0f / (float)p, kResRound);
    return acc - (unsigned)p * __float_as_uint(q);
  }
}

template <int I>
__device__ __forceinline__ uint4 emu_plane_piece(const unsigned (&lo)[kResK], const unsigned (&hi)[kResK]) {
  unsigned w[4];
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const unsigned r0 = emu_residue_byte<I>(lo[4 * g], hi[4 * g]), r1 = emu_residue_byte<I>(lo[4 * g + 1], hi[4 * g + 1]);
    const unsigned r2 = emu_residue_byte<I>(lo[4 * g + 2], hi[4 * g + 2]), r3 = emu_residue_byte<I>(lo[4 * g + 3], hi[4 * g + 3]);
    w[g] = __byte_perm(__byte_perm(r0, r1, 0x0040), __byte_perm(r2, r3, 0x0040), 0x5410);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}
template <int I>
__device__ __forceinline__ void emu_store_planes(int8_t* __restrict__ dst, size_t plane_stride, const unsigned (&lo)[kResK],
                                                 const unsigned (&hi)[kResK]) {
  if constexpr (I < kEmuModuli) {
    *reinterpret_cast<uint4*>(dst + I * plane_stride) = emu_plane_piece<I>(lo, hi);
    emu_store_planes<I + 1>(dst, plane_stride, lo, hi);
  }
}

__global__ void __launch_bounds__(kResThreads, 3)
emu_residue_kernel(const double* __restrict__ Yt, int64_t k_pad, int n_pad, const unsigned long long* __restrict__ colmax,
                   int bits, int8_t* __restrict__ Yq, const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int a = blockIdx.x * kResTA + 4 * warp + (lane & 3);
  if (a >= n_pad) return;
  // 2^e_a = s1 s2, each an exact double (e_a > 1023 only for columns whose maximum is below 2^-971)
  const int e = emu_exponent(colmax[a], bits);
  const int e1 = e < 1023 ? e : 1023;
  const double s1 = ldexp(1.0, e1), s2 = ldexp(1.0, e - e1);
  const size_t plane_stride = (size_t)n_pad * k_pad;
  for (int64_t k0 = (int64_t)blockIdx.y * kResTK + kResK * (lane >> 2); k0 < k_pad; k0 += (int64_t)gridDim.y * kResTK) {
    // k_pad is a multiple of 32: a thread's 16 rows are all in or all out
    const double* src = Yt + k0 * n_pad + a;
    double x[kResK];
#pragma unroll
    for (int j = 0; j < kResK; ++j) x[j] = __ldcs(src + (size_t)j * n_pad);
    unsigned lo[kResK], hi[kResK];
#pragma unroll
    for (int j = 0; j < kResK; ++j) {
      const long long v = __double2ll_rn(__dmul_rn(__dmul_rn(x[j], s1), s2));  // a' = rint(x 2^e_a), |a'| <= 2^53
      lo[j] = (unsigned)v;
      hi[j] = (unsigned)(v >> 32) + (1u << 23);  // + 2^55
    }
    emu_store_planes<0>(Yq + (size_t)a * k_pad + k0, plane_stride, lo, hi);
  }
}

__device__ __forceinline__ void tma_load_3d(unsigned dst, const CUtensorMap* map, int c0, int c1, int c2, unsigned bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
      : "memory");
}
// Shared-memory descriptor of a K-major operand tile written by TMA with SWIZZLE_128B: rows of 128 bytes,
// 8-row groups 1024 bytes apart (tile 1024-byte aligned); layout 2 = 128-byte swizzle, version 1.
__device__ __forceinline__ uint64_t umma_desc_sw128(unsigned saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// 32 consecutive columns of this warp's 32 tensor-memory lanes (one int32 accumulator row per lane)
__device__ __forceinline__ void tmem_ld32(unsigned taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ unsigned cluster_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// address of the same shared-memory object in CTA `rank` of the cluster
__device__ __forceinline__ unsigned mapa_shared(unsigned addr, unsigned rank) {
  unsigned r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Copy into this CTA's shared memory; the bytes complete_tx on `bar`, which may be the peer CTA's mbarrier.
__device__ __forceinline__ void tma_load_3d_pair(unsigned dst, const CUtensorMap* map, int c0, int c1, int c2,
                                                 unsigned bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void umma_i8_pair(unsigned tmem, uint64_t da, uint64_t db, uint32_t idesc, int accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n}\n"
      ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate));
}
// arrive on the mbarrier at this offset in both CTAs of the pair once the MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_pair(unsigned bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((unsigned short)3) : "memory");
}

// One cluster of two CTAs (one per SM) per item: the int8 SYRK of 256-tile (ti, tj) of modulus `mod`
// over its k-blocks, as tcgen05.mma.cta_group::2 with M = 256: CTA r of the pair holds rows
// 128 r .. 128 r + 127 of the A tile and the r-th half of the N rows of B, and its tensor memory
// receives rows 128 r .. of the 256 x N accumulator.  Per k-block an SM thus reads 32 KB for
// 128 x 256 products (128 x 128 with one CTA per MMA).
//   Full tile: A = rows 256 ti.., B = rows 256 tj.., N = 256; on the diagonal the B half of a CTA is
//     its A rows, so it loads one operand (and the MMA also computes the 128 x 128 block above the
//     diagonal, which is not stored).
//   Ragged last tile row (ti = last, rv < 256 valid rows; all of P when n_pad < 256): N = rv rounded up
//     to 16.  Off the diagonal the operands swap (A = tile tj, B = the ragged rows), so the MMA forms
//     the transposed block and the few ragged rows cost a thin N instead of a 256-row A operand.
//     Rows beyond n_pad lie outside the tensor and are zero-filled by the TMA unit.
//   RAGGED selects the ragged row's items, which run as a launch of their own so that their time can be
//   told apart (they reread the 256-row A tiles for a 256 x 16 product at C3).
// Warp 0 lane 0 of each CTA feeds its half of a 3-stage TMA ring; the copies complete on the leader's
// `full` barrier.  Warp 1 lane 0 of the leader issues four 256 x N x 32 MMAs per stage into an int32
// accumulator in tensor memory and frees the stage in both CTAs with a multicast tcgen05.commit.  The
// four warps of each CTA then drain its accumulator rows, reduce them mod p and add them to the residue
// sums of the 128-tiles they belong to (the Pmod layout does not depend on this kernel's tiling).  Two
// CTAs of different clusters share an SM, so one cluster's drain overlaps the other's MMAs.
template <bool RAGGED>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kEmuThreads, 2)
syrk_i8_pair_kernel(const __grid_constant__ CUtensorMap planes, const EmuItem* __restrict__ items,
                    uint32_t* __restrict__ Pmod, int n_tiles, int n_valid, const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;  // uniform over the cluster
  extern __shared__ unsigned char smem_raw[];
  // identical offsets in both CTAs: the leader's MMA descriptors address the peer's stages too
  const unsigned base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const unsigned bars = base + kEmuStages * kEmuStageBytes;
  const unsigned done_bar = bars + 16u * kEmuStages, tmem_slot = done_bar + 8u;
  auto full_bar = [&](int st) { return bars + 8u * st; };
  auto empty_bar = [&](int st) { return bars + 8u * (kEmuStages + st); };
  const unsigned rank = cluster_ctarank();
  const EmuItem it = items[blockIdx.x >> 1];
  const int nkb = it.kb_hi - it.kb_lo;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rv = RAGGED ? n_valid - it.ti * kEmuPair : kEmuPair;  // valid rows of tile row ti
  const int nN = (rv + 15) & ~15;
  const bool swap = nN < kEmuPair && it.ti != it.tj;
  const bool shared_op = nN == kEmuPair && it.ti == it.tj;  // B half of this CTA = its A rows
  const int rowA = (swap ? it.tj : it.ti) * kEmuPair, rowB = (swap ? it.ti : it.tj) * kEmuPair;
  const unsigned op_bytes = shared_op ? kEmuOpBytes : 2 * kEmuOpBytes;

  if (threadIdx.x == 0) {
    for (int st = 0; st < kEmuStages; ++st) {
      mbar_init(full_bar(st), 1);
      mbar_init(empty_bar(st), 1);
    }
    mbar_init(done_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&planes) : "memory");
  }
  if (warp == 0) {  // one warp of each CTA: the pair gets the same columns in both
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kEmuPair)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  cluster_sync();  // barriers of both CTAs initialised before any copy or commit reaches them
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  unsigned tmem;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(tmem_slot) : "memory");

  if (warp == 0 && lane == 0) {
    for (int kb = 0; kb < nkb; ++kb) {
      const int st = kb % kEmuStages;
      if (kb >= kEmuStages) mbar_wait(empty_bar(st), ((unsigned)(kb / kEmuStages) - 1u) & 1u);
      const unsigned dst = base + (unsigned)st * kEmuStageBytes;
      const unsigned full_leader = mapa_shared(full_bar(st), 0);
      const int k0 = (it.kb_lo + kb) * kEmuKB;
      if (rank == 0) mbar_arrive_expect_tx(full_bar(st), 2 * op_bytes);  // both CTAs' copies
      tma_load_3d_pair(dst, &planes, k0, rowA + (int)rank * kEmuTile, it.mod, full_leader);
      if (!shared_op) tma_load_3d_pair(dst + kEmuOpBytes, &planes, k0, rowB + (int)rank * (nN / 2), it.mod, full_leader);
    }
  } else if (warp == 1 && lane == 0 && rank == 0) {
    const uint32_t idesc = kEmuIdescM256 | ((uint32_t)(nN >> 3) << 17);
    for (int kb = 0; kb < nkb; ++kb) {
      const int st = kb % kEmuStages;
      mbar_wait(full_bar(st), (unsigned)(kb / kEmuStages) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const unsigned a = base + (unsigned)st * kEmuStageBytes;
      const uint64_t da = umma_desc_sw128(a), db = shared_op ? da : umma_desc_sw128(a + kEmuOpBytes);
#pragma unroll
      for (int k = 0; k < kEmuKB / 32; ++k)  // 32 bytes of k per MMA: +2 in the 16-byte address field
        umma_i8_pair(tmem, da + 2u * k, db + 2u * k, idesc, (kb | k) != 0);
      umma_commit_pair(empty_bar(st));
    }
    umma_commit_pair(done_bar);
  }
  __syncwarp();
  mbar_wait(done_bar, 0);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

  const int p = emu_modulus(it.mod);
  const int lr = (int)rank * kEmuTile + warp * 32 + lane;  // accumulator row of the pair = A row - rowA
#pragma unroll 1
  for (int c0 = 0; c0 < nN; c0 += 32) {
    // above the diagonal from here on (unswapped: the columns grow with c0)
    if (!swap && rowB + c0 > ((rowA + (int)rank * kEmuTile) | (kEmuTile - 1))) break;
    uint32_t v[32];
    tmem_ld32(tmem + ((unsigned)(warp * 32) << 16) + (unsigned)c0, v);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const int R = swap ? rowB + c0 + j : rowA + lr, C = swap ? rowA + lr : rowB + c0 + j;  // position in P
      const int ti = R / kEmuTile, tj = C / kEmuTile, r = R % kEmuTile, c = C % kEmuTile;
      // valid part of P; on a diagonal 128-tile the pairs the DMMA path's reduce kernel writes
      if (c0 + j >= nN || R >= n_valid || C >= n_valid || tj > ti || (ti == tj && c > (r | 1))) continue;
      int m = (int)v[j] % p;
      if (m < 0) m += p;
      if (m)
        atomicAdd(Pmod + ((size_t)it.mod * n_tiles + ti * (ti + 1) / 2 + tj) * (kEmuTile * kEmuTile) +
                      (size_t)c * kEmuTile + r,
                  (uint32_t)m);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  cluster_sync();  // both CTAs done with the accumulator columns before they are freed
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kEmuPair) : "memory");
  }
}

// The integer sum_k a'_k b'_k from its residue sums (Garner, symmetric lift) as a double (Horner from
// the most significant digit; see the bound above).
__device__ __forceinline__ double emu_lift(const uint32_t (&x)[kEmuModuli], const EmuConsts& C) {
  int v[kEmuModuli];
#pragma unroll
  for (int i = 0; i < kEmuModuli; ++i) {
    const unsigned p = (unsigned)emu_modulus(i);
    unsigned t = x[i] % p;
#pragma unroll
    for (int j = 0; j < i; ++j) t = (t + 2u * p - (unsigned)v[j]) * (unsigned)C.inv[j][i] % p;
    v[i] = (int)t;
  }
  // value >= prod(p) / 2: negative, -(prod(p) - value); prod(p) - 1 - value has the digits p_i - 1 - v_i
  int cmp = 0;
#pragma unroll
  for (int i = kEmuModuli - 1; i >= 0; --i)
    if (cmp == 0) cmp = v[i] > C.half[i] ? 1 : (v[i] < C.half[i] ? -1 : 0);
  const bool neg = cmp >= 0;
  double acc = 0.0;
#pragma unroll
  for (int i = kEmuModuli - 1; i >= 0; --i) {
    const int d = neg ? emu_modulus(i) - 1 - v[i] + (i == 0 ? 1 : 0) : v[i];
    acc = __fma_rn(acc, (double)emu_modulus(i), (double)d);
  }
  return neg ? -acc : acc;
}

// P[lower] from the residue sums: a block converts a 32 x 32 piece of a tile (read along the columns
// of the column-major sums, written along the rows of P through shared memory).
__global__ void __launch_bounds__(256)
emu_reconstruct_kernel(const uint32_t* __restrict__ Pmod, int n_tiles, const unsigned long long* __restrict__ colmax,
                       int bits, double* __restrict__ P, int ld, int n_valid, const EmuConsts C, const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;
  __shared__ double s[32][33];
  const int t = blockIdx.x;
  int ti, tj;
  tile_from_linear(t, ti, tj);
  const int rb = blockIdx.y & 3, cb = blockIdx.y >> 2;
  if (ti == tj && cb > rb) return;  // above the diagonal
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int R = ti * kEmuTile + rb * 32 + tx;
  const int er = R < n_valid ? emu_exponent(colmax[R], bits) : 0;
  for (int cc = ty; cc < 32; cc += 8) {
    const int c = cb * 32 + cc, Cg = tj * kEmuTile + c;
    double val = 0.0;
    if (R < n_valid && Cg < n_valid) {
      uint32_t x[kEmuModuli];
#pragma unroll
      for (int i = 0; i < kEmuModuli; ++i)
        x[i] = Pmod[((size_t)i * n_tiles + t) * (kEmuTile * kEmuTile) + (size_t)c * kEmuTile + rb * 32 + tx];
      val = ldexp(emu_lift(x, C), -(er + emu_exponent(colmax[Cg], bits)));
    }
    s[cc][tx] = val;
  }
  __syncthreads();
  for (int rr = ty; rr < 32; rr += 8) {
    const int r = rb * 32 + rr, c = cb * 32 + tx;
    const int Rg = ti * kEmuTile + r, Cg = tj * kEmuTile + c;
    if (Rg >= n_valid || Cg >= n_valid || (ti == tj && c > (r | 1))) continue;
    P[(size_t)Rg * ld + Cg] = s[tx][rr];
  }
}

// ---- host side --------------------------------------------------------------------------------
static inline int syrk_kc(int tile) { return tile == kTmaTile ? kTmaKC : kDmmaKC; }
static inline int syrk_occupancy(int tile) { return tile == kTmaTile ? 1 : 4; }

// Relative duration of a tile per k-row (1 = full tile), mirroring the kernel's warp mapping:
// edge tiles skip the 8x8 fragments beyond n_valid, diagonal tiles the sub-tiles above the
// diagonal.  A warp sits on scheduler partition (warp % 4) with its own FP64 pipe: a CTA that has
// an SM to itself takes as long as its busiest partition; with several CTAs per SM the partitions
// even out and the mean counts.
static double tile_weight(int TILE, int ti, int tj, int n_valid, int64_t k_pad = 0, double floor_override = -1.0) {
  const int WR = TILE == kTmaTile ? 4 : kDmmaWR, WC = TILE == kTmaTile ? 4 : kDmmaWC;  // syrk_tma_kernel: 4 x 4 warps
  const int occ = syrk_occupancy(TILE);
  const int WM = TILE / WR, WN = TILE / WC, FM = WM / 8, FN = WN / 8;
  double load[4] = {0, 0, 0, 0};
  const bool folded_diag = ti == tj && TILE == kTmaTile;

  if (folded_diag) {
    // the TMA kernel's diagonal mapping: fragment rows r and 15 - r shared by two warps (9 + 8)
    const int rows_valid = std::min(16, (n_valid - ti * TILE + 7) / 8);
    for (int warp = 0; warp < 16; ++warp) {
      const int pr = warp >> 1;
      const bool nine = (((warp & 1) ^ ((warp >> 2) & 1)) == 0);
      const int r_hi = 15 - pr, r_lo = pr, n_hi = nine ? 9 : 7 - pr, nfr = nine ? 9 : 8;
      for (int j = 0; j < nfr; ++j) load[warp % 4] += ((j < n_hi ? r_hi : r_lo) < rows_valid) ? 1.0 : 0.0;
    }
  }
  for (int warp = 0; warp < WR * WC && !folded_diag; ++warp) {
    int wr = warp / WC, wc = warp % WC;
    bool live = true;
    if (ti == tj && WR == WC) {
      live = warp < WR * (WR + 1) / 2;
      if (live) {
        wr = 0;
        while ((wr + 1) * (wr + 2) / 2 <= warp) ++wr;
        wc = warp - wr * (wr + 1) / 2;
      }
    }
    int vm = 0, vn = 0;
    for (int i = 0; i < FM; ++i) vm += (ti * TILE + wr * WM + 8 * i) < n_valid;
    for (int j = 0; j < FN; ++j) vn += (tj * TILE + wc * WN + 8 * j) < n_valid;
    if (live) load[warp % 4] += (double)vm * vn;
  }
  const double per_part = (double)FM * FN * ((WR * WC + 3) / 4);
  const double mx = std::max(std::max(load[0], load[1]), std::max(load[2], load[3]));
  const double mean = (load[0] + load[1] + load[2] + load[3]) / 4.0;
  const double w = (occ == 1 ? mx : mean) / per_part;
  // A CTA pays for every k-row it streams whatever it computes on it (copies, barrier, pipeline
  // bookkeeping): tiles with little tensor work are bounded by that floor, not by their DMMA count.
  // Measured at C2 (50 x 10k): the 64-tile kernel (four CTAs per SM) is fastest with uniform cuts
  // (floor 1.0: 0.302 ms per iteration, 0.75: 0.309, 0.5: 0.344, 0.35: 0.430).
  // The TMA-fed 128-tile kernel has no per-row copy instructions to pay for: a thin tile costs what its
  // fragments cost, down to the rate at which the TMA unit streams the rows (measured floor ~0.3).
  // Measured with the TMA kernel (B200): C3 (4.3 GB operand, ~3300-row pieces) floor 0.5: 28.79 ms,
  // 0.3: 28.86, 0.15: 28.86, 0.75: 29.42; C2 (108 MB operand, two waves of ~730-row pieces) floor
  // 1.0: 0.286 ms, 0.5: 0.298, 0.3: 0.311 -- with two waves the schedule is decided by whole items,
  // and uniform cuts pack them best.
  const bool small_operand = k_pad > 0 && (double)k_pad * n_valid * 8.0 <= 256.0 * 1024 * 1024;
  double floor_w = occ == 1 && !small_operand ? 0.5 : 1.0;
  if (floor_override >= 0.0) floor_w = floor_override;
  return w > floor_w ? w : floor_w;
}

struct SyrkPlan {
  std::vector<SyrkItem> items;       // launch order: ascending k range, then tile
  std::vector<int> tile_first;       // [n_tiles + 1]
  std::vector<int> tile_items;       // partial-tile slot per (tile, piece), pieces in ascending k order
  int n_slots = 0;                   // partial tiles: one per item + one per tall item (its thin tile below)
  int tall_row = -1;                 // tile row whose off-diagonal tiles also compute the ragged rows below
  double makespan = 0.0;             // modelled duration in k-rows of a full tile on one SM slot
};

// The ragged last tile row of 128-tiles is folded into the row above (see kTmaTallRows) when at most
// kTmaTallRows rows are left over: returns that row (nt1 - 2), else -1.
static int tall_tile_row(int n_pad, int TILE) {
  const int nt1 = (n_pad + TILE - 1) / TILE;
  const int left = n_pad - (nt1 - 1) * TILE;
  if (TILE != kTmaTile || nt1 < 3 || left > kTmaTallRows) return -1;
  return nt1 - 2;
}

// Cut every tile's K range into pieces so that all CTAs take about the same time and their number
// fills whole waves of SM slots: pieces(t) ~ weight(t) x S.  S is chosen by simulating the block
// scheduler (CTAs start in launch order on the first free slot) for every admissible S and
// keeping the shortest schedule.  Constraints: a piece streams >= 512 k-rows (prologue, epilogue
// and the partial-tile write stay small against it), and -- L2 residency -- the k-slab that the
// CTAs of one "column" of the schedule share should stay below 48 MB: ncu showed 18.6 GB of DRAM
// reads for the 4.3 GB operand of C3 when 271 MB slabs were streamed by tiles drifting apart.
static SyrkPlan plan_syrk(int n_pad, int TILE, int64_t k_pad, int num_sms) {
  const int KC = syrk_kc(TILE), occ = syrk_occupancy(TILE);
  const int nt1 = (n_pad + TILE - 1) / TILE;
  const int n_tiles = nt1 * (nt1 + 1) / 2;
  const int64_t n_chunks = k_pad / KC;
  const int slots = num_sms * occ;
  std::vector<double> w(n_tiles), w_run(n_tiles);  // w: decides the cuts; w_run: the modelled duration per k-row
  const bool lpt = (double)k_pad * n_pad * 8.0 <= 116.0 * 1024 * 1024;
  const double run_floor = 0.5;
  const int tall_row = tall_tile_row(n_pad, TILE);
  // absorbed[t]: thin tile (nt1 - 1, tj), tj < tall_row: computed by the tall tile (tall_row, tj)
  std::vector<char> absorbed(n_tiles, 0), is_tall(n_tiles, 0);
  for (int t = 0, ti = 0; ti < nt1; ++ti)
    for (int tj = 0; tj <= ti; ++tj, ++t) {
      w[t] = tile_weight(TILE, ti, tj, n_pad, k_pad);
      // longest-first schedules are simulated with what a tile really costs (its fragments, down to
      // the rate of the TMA ring), not with the weight that decides the cuts
      w_run[t] = lpt ? tile_weight(TILE, ti, tj, n_pad, k_pad, run_floor) : w[t];
      if (tall_row >= 0 && tj < tall_row) {
        if (ti == tall_row) { is_tall[t] = 1; w[t] *= 1.0 + 2.0 / 16.0; w_run[t] *= 1.0 + 2.0 / 16.0; }  // two more fragments per warp
        if (ti == nt1 - 1) absorbed[t] = 1;
      }
    }
  const int64_t min_chunks = std::max<int64_t>(1, 512 / KC);
  const int64_t s_max = std::max<int64_t>(1, n_chunks / min_chunks);
  const int64_t slab_cap = (int64_t)48 << 20;
  const int64_t s_l2 = std::min<int64_t>(s_max, (k_pad * (int64_t)n_pad * 8 + slab_cap - 1) / slab_cap);
  const int64_t s_cap = std::min<int64_t>(s_max, std::max<int64_t>(s_l2, std::max<int64_t>(1, (int64_t)24 * slots / n_tiles)));
  const int64_t s_lo = std::max<int64_t>(1, std::min<int64_t>(s_l2, s_cap));
  const double overhead = 48.0;  // k-rows of a full tile: pipeline fill + partial-tile write

  auto build = [&](int64_t S, SyrkPlan* out) -> double {
    struct Piece { int t; int64_t lo, hi; int kidx; };  // kidx: position among its tile's pieces (ascending k)
    std::vector<Piece> pieces;
    std::vector<int> count(n_tiles);
    for (int t = 0; t < n_tiles; ++t) {
      if (absorbed[t]) { count[t] = 0; continue; }
      int64_t p = (int64_t)std::llround(w[t] * (double)S);
      p = std::max<int64_t>(1, std::min<int64_t>(p, s_max));
      const int64_t cps = (n_chunks + p - 1) / p;
      p = (n_chunks + cps - 1) / cps;
      count[t] = (int)p;
      for (int64_t k = 0; k < p; ++k) pieces.push_back({t, k * cps, std::min<int64_t>(n_chunks, (k + 1) * cps), (int)k});
    }
    std::stable_sort(pieces.begin(), pieces.end(), [](const Piece& a, const Piece& b) {
      return a.lo != b.lo ? a.lo < b.lo : a.t < b.t;
    });
    // An operand that stays in the L2 whatever the order (C2: 110 MB) is scheduled longest item first:
    // with ~2 waves of items of unequal duration (full tiles 1.0, diagonal / ragged ones ~0.55 per
    // k-row) the k-major order leaves SMs with two long items next to SMs with two short ones.
    if (lpt)
      std::stable_sort(pieces.begin(), pieces.end(), [&](const Piece& a, const Piece& b) {
        return w_run[a.t] * (double)(a.hi - a.lo) > w_run[b.t] * (double)(b.hi - b.lo);
      });
    // list scheduling on `slots` slots, each running at 1/occ of an SM
    std::priority_queue<double, std::vector<double>, std::greater<double>> free_at;
    for (int k = 0; k < slots; ++k) free_at.push(0.0);
    double makespan = 0.0;
    for (const Piece& pc : pieces) {
      const double start = free_at.top();
      free_at.pop();
      const double end = start + (w_run[pc.t] * (double)(pc.hi - pc.lo) * KC + overhead) * occ;
      free_at.push(end);
      makespan = std::max(makespan, end);
    }
    if (out) {
      out->items.clear();
      out->tile_first.assign(n_tiles + 1, 0);
      std::vector<int> ti_of(n_tiles), tj_of(n_tiles);
      for (int t = 0, ti = 0; ti < nt1; ++ti)
        for (int tj = 0; tj <= ti; ++tj, ++t) { ti_of[t] = ti; tj_of[t] = tj; }
      auto tile_index = [](int ti, int tj) { return ti * (ti + 1) / 2 + tj; };
      // a thin tile absorbed by a tall one has as many partial tiles as that tile has pieces
      for (int t = 0; t < n_tiles; ++t)
        out->tile_first[t + 1] = out->tile_first[t] + (absorbed[t] ? count[tile_index(tall_row, tj_of[t])] : count[t]);
      out->tile_items.assign(out->tile_first[n_tiles], 0);
      int n_slots = (int)pieces.size();  // slot of an item = its index; the second slots follow
      for (const Piece& pc : pieces) {  // launch order; a tile's partial tiles are listed in ascending k order
        const int item = (int)out->items.size();
        out->tile_items[out->tile_first[pc.t] + pc.kidx] = item;
        int slot2 = -1;
        if (is_tall[pc.t]) {
          slot2 = n_slots++;
          const int thin = tile_index(nt1 - 1, tj_of[pc.t]);
          out->tile_items[out->tile_first[thin] + pc.kidx] = slot2;
        }
        out->items.push_back({ti_of[pc.t], tj_of[pc.t], (int)pc.lo, (int)pc.hi, slot2});
      }
      out->n_slots = n_slots;
      out->tall_row = tall_row;
      out->makespan = makespan;
    }
    return makespan;
  };

  int64_t best_S = s_lo;
  double best = 1e300;
  for (int64_t S = s_lo; S <= s_cap; ++S) {
    const double m = build(S, nullptr);
    if (m < best * (1.0 - 1e-9)) { best = m; best_S = S; }
  }
  SyrkPlan plan;
  build(best_S, &plan);
  return plan;
}

// Plans are kept for the life of the process: the schedule search costs milliseconds of host
// time, more than a small adjustment, and callers adjust scene after scene of the same shape.
static const SyrkPlan& cached_plan(int n_pad, int tile, int64_t k_pad, int num_sms) {
  struct Key { int n_pad, tile; int64_t k_pad; int sms; };
  static std::mutex mu;
  static std::vector<std::pair<Key, SyrkPlan*>> cache;
  std::lock_guard<std::mutex> lock(mu);
  for (auto& kv : cache)
    if (kv.first.n_pad == n_pad && kv.first.tile == tile && kv.first.k_pad == k_pad && kv.first.sms == num_sms)
      return *kv.second;
  SyrkPlan* p = new SyrkPlan(plan_syrk(n_pad, tile, k_pad, num_sms));
  cache.push_back({Key{n_pad, tile, k_pad, num_sms}, p});
  return *p;
}

// ---- tensor maps (host) ---------------------------------------------------------------------------
// cuTensorMapEncodeTiled comes from the driver; it is fetched through the runtime so that the
// library does not link against libcuda (the build container has no driver).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn tensor_map_encoder() {
  static EncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      f = nullptr;
    cudaGetLastError();
    return reinterpret_cast<EncodeTiledFn>(f);
  }();
  return fn;
}

// k-major operand `base` [rows][ld] doubles, `cols` valid columns: boxes of `box_cols` columns (kTmaLda
// = 148 for the row operand, kTmaLdb = 132 for the column operand) x kTmaKC rows.
static int make_operand_map(CUtensorMap* map, const double* base, int cols, int64_t rows, int ld, int box_cols) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) { set_error("cuTensorMapEncodeTiled is not available from this driver"); return BA_ERR_CUDA; }
  const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(double)};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)kTmaKC};
  const cuuint32_t estride[2] = {1, 1};
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), gdim, gstride, box,
                         estride, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for a %d x %lld operand, ld %d", (int)r, cols, (long long)rows, ld);
    return BA_ERR_CUDA;
  }
  return BA_OK;
}

// The 128-tile product, the wide Cholesky updates and the INT8 emulation are all fed by TMA; every
// driver that runs sm_100a code offers the encoder, so an engine checks for it once when created.
int require_tensor_map_encoder() {
  if (tensor_map_encoder()) return BA_OK;
  set_error("cuTensorMapEncodeTiled is not available from this driver (the TMA-fed kernels need it)");
  return BA_ERR_CUDA;
}

// ---- emulated product: host side ------------------------------------------------------------------
static const EmuConsts& emu_consts() {
  static const EmuConsts c = [] {
    EmuConsts k{};
    for (int i = 0; i < kEmuModuli; ++i)
      for (int j = 0; j < i; ++j) {
        const int p = emu_modulus(i), a = emu_modulus(j) % p;
        int x = 1;
        while (a * x % p != 1) ++x;  // p < 257: a search is enough
        k.inv[j][i] = x;
      }
    unsigned __int128 h = 1;
    for (int i = 0; i < kEmuModuli; ++i) h *= (unsigned)emu_modulus(i);
    h /= 2;
    for (int i = 0; i < kEmuModuli; ++i) {
      k.half[i] = (int)(h % (unsigned)emu_modulus(i));
      h /= (unsigned)emu_modulus(i);
    }
    return k;
  }();
  return c;
}

// Largest b <= 53 with k_pad 2^(2b) < prod(p) / 2: the CRT lift of a dot product of k_pad terms of
// magnitude <= 2^b each is then exact.  0 if there is none.
static int emu_bits_for(int64_t k_pad) {
  unsigned __int128 half = 1;
  for (int i = 0; i < kEmuModuli; ++i) half *= (unsigned)emu_modulus(i);
  half /= 2;
  for (int b = 53; b > 0; --b)
    if ((unsigned __int128)k_pad < (half >> (2 * b))) return b;  // k_pad 2^(2b) < half, whole multiples of 2^(2b)
  return 0;
}

int syrk_emu_info(int64_t k_pad, int32_t* moduli, int* n_moduli, int* bits) {
  if (k_pad < 1) { set_error("k_pad must be positive"); return BA_ERR_INVALID; }
  if (moduli)
    for (int i = 0; i < kEmuModuli; ++i) moduli[i] = emu_modulus(i);
  if (n_moduli) *n_moduli = kEmuModuli;
  if (bits) *bits = emu_bits_for(k_pad);
  return BA_OK;
}

// Work items: every (modulus, lower 256-tile) over P equal k pieces of <= kEmuMaxKB blocks, in two
// lists: the tiles of whole 256-row tile rows, and those of a ragged last tile row (launched apart).
// Every item of a list costs about the same per k-block, so the plan only picks P for whole waves of
// two clusters per pair of SMs, and orders the items k-piece first (as plan_syrk does: the clusters in
// flight share one k-slab in the L2).
struct EmuPlan {
  std::vector<EmuItem> full, ragged;
};
static std::vector<EmuItem> plan_emu_list(int row_lo, int row_hi, int64_t nkb, int num_sms) {
  int64_t n_tiles = 0;
  for (int ti = row_lo; ti < row_hi; ++ti) n_tiles += ti + 1;
  std::vector<EmuItem> items;
  if (n_tiles == 0) return items;
  const int64_t slots = num_sms;
  const int64_t p_min = (nkb + kEmuMaxKB - 1) / kEmuMaxKB;
  const double overhead = 16.0;  // k-blocks: pipeline fill and the accumulator drain
  int64_t best_p = p_min;
  double best = 1e300;
  for (int64_t p = p_min; p <= std::min<int64_t>(nkb, p_min + 8); ++p) {
    const int64_t n = kEmuModuli * n_tiles * p, waves = (n + slots - 1) / slots;
    const double t = (double)waves * ((double)((nkb + p - 1) / p) + overhead);
    if (t < best * (1.0 - 1e-9)) { best = t; best_p = p; }
  }
  const int64_t per = (nkb + best_p - 1) / best_p;
  for (int64_t lo = 0; lo < nkb; lo += per)
    for (int m = 0; m < kEmuModuli; ++m)
      for (int ti = row_lo; ti < row_hi; ++ti)
        for (int tj = 0; tj <= ti; ++tj) items.push_back({m, ti, tj, (int)lo, (int)std::min<int64_t>(nkb, lo + per)});
  return items;
}
static EmuPlan plan_emu(int n_pad, int64_t k_pad, int num_sms) {
  const int full_rows = n_pad / kEmuPair, nt1 = (n_pad + kEmuPair - 1) / kEmuPair;
  const int64_t nkb = (k_pad + kEmuKB - 1) / kEmuKB;
  return {plan_emu_list(0, full_rows, nkb, num_sms), plan_emu_list(full_rows, nt1, nkb, num_sms)};
}

// ---- the planned product: choice, upload, launch ---------------------------------------------------
template <typename T>
static int dev_upload(T** dst, const std::vector<T>& src, cudaStream_t s) {
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(dst), src.size() * sizeof(T), s));
  BA_CUDA(cudaMemcpyAsync(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, s));
  return BA_OK;
}

int syrk_prepare(SyrkProduct* p, SyrkKind kind, int n_pad, int64_t k_pad, int num_sms, cudaStream_t s) {
  *p = SyrkProduct();
  p->n_pad = n_pad;
  p->k_pad = k_pad;
  p->num_sms = num_sms;
  p->emu_bits = emu_bits_for(k_pad);
  if (kind == SYRK_AUTO) {
    // The emulation is chosen when it is exact to (nearly) full FP64 input precision and the product
    // is large enough for the INT8 tensor cores to pay for the conversion passes; BA_SYRK_EMU=0|1
    // overrides the size rule (A/B timing and tests).  FP64 64-tiles up to n_pad = 384 (C2, n = 451:
    // 128-tiles 0.283 ms vs 64-tiles 0.302 ms per iteration).
    const char* v = std::getenv("BA_SYRK_EMU");
    const bool emu = v ? std::atoi(v) != 0 : p->emu_bits >= 50 && (double)n_pad * n_pad * (double)k_pad >= kEmuMinWork;
    kind = emu ? SYRK_EMULATED : n_pad <= 384 ? SYRK_TILE64 : SYRK_TILE128;
  }
  p->kind = kind;
  const bool timing = std::getenv("BA_TIMING") != nullptr;
  if (kind == SYRK_EMULATED) {
    const EmuPlan plan = plan_emu(n_pad, k_pad, num_sms);
    std::vector<EmuItem> items = plan.full;
    items.insert(items.end(), plan.ragged.begin(), plan.ragged.end());
    const int nt1 = (n_pad + kEmuTile - 1) / kEmuTile;
    p->n_tiles = nt1 * (nt1 + 1) / 2;
    p->emu_n_items = (int)items.size();
    p->emu_n_ragged = (int)plan.ragged.size();
    BA_TRY(dev_upload(&p->emu_items, items, s));
    BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&p->Yq), (size_t)kEmuModuli * n_pad * k_pad, s));
    BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&p->Pmod),
                            (size_t)kEmuModuli * p->n_tiles * kEmuTile * kEmuTile * sizeof(uint32_t), s));
    BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&p->colmax), (size_t)n_pad * sizeof(unsigned long long), s));
    if (timing)
      std::fprintf(stderr, "[ba syrk plan] int8 emulation: b = %d, %d tiles x %d moduli, %d items\n", p->emu_bits,
                   p->n_tiles, kEmuModuli, p->emu_n_items);
  } else {
    const int tile = kind == SYRK_TILE128 ? kTmaTile : kDmmaTile;
    const SyrkPlan& plan = cached_plan(n_pad, tile, k_pad, num_sms);
    const int nt1 = (n_pad + tile - 1) / tile;
    p->n_tiles = nt1 * (nt1 + 1) / 2;
    p->n_items = (int)plan.items.size();
    BA_TRY(dev_upload(&p->items, plan.items, s));
    BA_TRY(dev_upload(&p->tile_first, plan.tile_first, s));
    BA_TRY(dev_upload(&p->tile_items, plan.tile_items, s));
    BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&p->part), (size_t)plan.n_slots * tile * tile * sizeof(double), s));
    if (timing)
      std::fprintf(stderr, "[ba syrk plan] tile %d: %d tiles, %d items on %d slots, modelled %.0f k-rows (ideal %.0f)\n",
                   tile, p->n_tiles, p->n_items, num_sms * syrk_occupancy(tile), plan.makespan, 0.0);
  }
  BA_CUDA(cudaStreamSynchronize(s));  // allocated and filled on s, used on whatever stream launches the product
  return BA_OK;
}

void syrk_release(SyrkProduct* p, cudaStream_t s) {
  void* ptrs[] = {p->items, p->tile_first, p->tile_items, p->part, p->emu_items, p->Yq, p->Pmod, p->colmax};
  for (void* q : ptrs)
    if (q) cudaFreeAsync(q, s);
  *p = SyrkProduct();
}

// The residue planes as one 3D tensor {k, row, plane} of bytes; boxes of 128 k x 128 rows of one plane
// (rows beyond n_pad are zero-filled), 128-byte swizzle: the canonical K-major operand of tcgen05.mma.
static int make_plane_map(CUtensorMap* map, const int8_t* Yq, int n_pad, int64_t k_pad) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) { set_error("cuTensorMapEncodeTiled is not available from this driver"); return BA_ERR_CUDA; }
  const cuuint64_t gdim[3] = {(cuuint64_t)k_pad, (cuuint64_t)n_pad, (cuuint64_t)kEmuModuli};
  const cuuint64_t gstride[2] = {(cuuint64_t)k_pad, (cuuint64_t)k_pad * n_pad};
  const cuuint32_t box[3] = {(cuuint32_t)kEmuKB, (cuuint32_t)kEmuTile, 1};
  const cuuint32_t estride[3] = {1, 1, 1};
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<int8_t*>(Yq), gdim, gstride, box, estride,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for %d residue planes of %d x %lld", (int)r, kEmuModuli, n_pad,
              (long long)k_pad);
    return BA_ERR_CUDA;
  }
  return BA_OK;
}

// Emulated product: residue planes of Yt, one int8 SYRK per modulus into the residue sums, P from them.
static int launch_emulated(const SyrkProduct* p, const double* Yt, double* P, const ba_lm_state* ctl, cudaStream_t s,
                           ba_engine* prof) {
  CUtensorMap map;
  BA_TRY(make_plane_map(&map, p->Yq, p->n_pad, p->k_pad));
  BA_CUDA(cudaFuncSetAttribute(syrk_i8_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEmuSmemBytes));
  BA_CUDA(cudaFuncSetAttribute(syrk_i8_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEmuSmemBytes));
  const int n_tiles = p->n_tiles;
  std::optional<ProfScope> ps;
  if (prof) ps.emplace(prof, PG_SYRK, s);
  // colmax was gathered by K2b (launch_k2b resets it before every launch)
  BA_CUDA(cudaMemsetAsync(p->Pmod, 0, (size_t)kEmuModuli * n_tiles * kEmuTile * kEmuTile * sizeof(uint32_t), s));
  {
    const int64_t k_tiles = (p->k_pad + kResTK - 1) / kResTK;
    emu_residue_kernel<<<dim3((p->n_pad + kResTA - 1) / kResTA, (unsigned)std::min<int64_t>(k_tiles, 65535)),
                         kResThreads, 0, s>>>(Yt, p->k_pad, p->n_pad, p->colmax, p->emu_bits, p->Yq, ctl);
    BA_LAUNCH_CHECK();
  }
  const int n_full = p->emu_n_items - p->emu_n_ragged;
  if (n_full > 0) {
    syrk_i8_pair_kernel<false><<<2 * n_full, kEmuThreads, kEmuSmemBytes, s>>>(map, p->emu_items, p->Pmod, n_tiles,
                                                                              p->n_pad, ctl);
    BA_LAUNCH_CHECK();
  }
  if (p->emu_n_ragged > 0) {
    syrk_i8_pair_kernel<true><<<2 * p->emu_n_ragged, kEmuThreads, kEmuSmemBytes, s>>>(
        map, p->emu_items + n_full, p->Pmod, n_tiles, p->n_pad, ctl);
    BA_LAUNCH_CHECK();
  }
  emu_reconstruct_kernel<<<dim3(n_tiles, 16), 256, 0, s>>>(p->Pmod, n_tiles, p->colmax, p->emu_bits, P, p->n_pad,
                                                          p->n_pad, emu_consts(), ctl);
  BA_LAUNCH_CHECK();
  return BA_OK;
}

int syrk_launch(const SyrkProduct* p, const double* Yt, double* P, const ba_lm_state* ctl, cudaStream_t s,
                ba_engine* prof) {
  if (p->kind == SYRK_EMULATED) return launch_emulated(p, Yt, P, ctl, s, prof);
  const bool tma = p->kind == SYRK_TILE128;
  const int tile = tma ? kTmaTile : kDmmaTile;
  const int64_t n_chunks = p->k_pad / syrk_kc(tile);
  const SubSplit none{0, 1, 0, 0, {}};
  CUtensorMap mapA, mapB;
  if (tma) {
    BA_TRY(make_operand_map(&mapA, Yt, p->n_pad, p->k_pad, p->n_pad, kTmaLda));
    BA_TRY(make_operand_map(&mapB, Yt, p->n_pad, p->k_pad, p->n_pad, kTmaLdb));
    BA_CUDA(cudaFuncSetAttribute(syrk_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)kTmaSmemBytes));
  } else {
    BA_CUDA(cudaFuncSetAttribute(syrk_dmma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)kDmmaSmemBytes));
  }
  std::optional<ProfScope> ps;  // the "syrk" scope: the tile kernel, not the sums of its partial tiles
  if (prof) ps.emplace(prof, PG_SYRK, s);
  if (tma)
    syrk_tma_kernel<false><<<p->n_items, kTmaThreads, kTmaSmemBytes, s>>>(mapA, mapB, p->n_pad, p->n_pad, n_chunks,
                                                                          p->items, p->part, ctl, 0, none);
  else
    syrk_dmma_kernel<false><<<p->n_items, kDmmaThreads, kDmmaSmemBytes, s>>>(Yt, p->n_pad, p->n_pad, n_chunks,
                                                                             p->items, p->part, ctl, 0, none);
  BA_LAUNCH_CHECK();
  ps.reset();
  // enough blocks to fill the GPU (C2: 10 tiles x 8 slabs = 80 blocks took 33 us for 38 MB), at
  // least one pair of doubles per thread
  const int slabs_max = tile * tile / 2 / 256;
  int slabs = 1;
  while (slabs < slabs_max && p->n_tiles * slabs < 4 * p->num_sms) slabs *= 2;
  const dim3 grid(p->n_tiles, slabs);
  if (tma)
    syrk_reduce_kernel<kTmaTile><<<grid, 256, 0, s>>>(p->part, p->tile_first, p->tile_items, P, p->n_pad, p->n_pad, ctl);
  else
    syrk_reduce_kernel<kDmmaTile><<<grid, 256, 0, s>>>(p->part, p->tile_first, p->tile_items, P, p->n_pad, p->n_pad, ctl);
  BA_LAUNCH_CHECK();
  return BA_OK;
}

// S[t0:, t0:] -= Lt[:, t0:]^T Lt[:, t0:]  (lower triangle, rows < n_rows) with Lt k-major
// [depth][ld]: the wide trailing update of the two-level blocked Cholesky.  128-tiles (one CTA per
// SM) once there are enough of them, 64-tiles (four per SM) below.  Only the 128-tile form is
// divided over the ranks of a sharded run.
int launch_chol_wide_update(double* S, int ld, int n_rows, int t0, const double* Lt, int depth,
                            const ba_lm_state* ctl, cudaStream_t s, const CholSplit* split) {
  const bool tma = n_rows - t0 >= kCholSplitMinRows;
  const int tile = tma ? kTmaTile : kDmmaTile;
  const int n_store = n_rows - t0;
  const int n_valid = (n_store + 7) / 8 * 8;  // <= ld - t0: ld is a multiple of 8, t0 of 64
  const int nt1 = (n_valid + tile - 1) / tile;
  const int n_tiles = nt1 * (nt1 + 1) / 2;
  const int n_chunks = depth / syrk_kc(tile);
  const size_t origin = (size_t)t0 * ld + t0;
  SubSplit sp{0, 1, 0, 0, {}};
  if (tma && split && split->world > 1) {
    sp.rank = split->rank;
    sp.world = split->world;
    sp.tile_row0 = t0 / tile;
    sp.push_cols = split->push_cols;
    for (int q = 0; q < split->world; ++q) sp.peer[q] = split->S_peer[q] + origin;
  }
  if (tma) {
    CUtensorMap mapA, mapB;
    BA_TRY(make_operand_map(&mapA, Lt + t0, n_valid, depth, ld, kTmaLda));
    BA_TRY(make_operand_map(&mapB, Lt + t0, n_valid, depth, ld, kTmaLdb));
    BA_CUDA(cudaFuncSetAttribute(syrk_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)kTmaSmemBytes));
    syrk_tma_kernel<true><<<n_tiles, kTmaThreads, kTmaSmemBytes, s>>>(mapA, mapB, ld, n_valid, n_chunks, nullptr,
                                                                      S + origin, ctl, n_store, sp);
  } else {
    BA_CUDA(cudaFuncSetAttribute(syrk_dmma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)kDmmaSmemBytes));
    syrk_dmma_kernel<true><<<n_tiles, kDmmaThreads, kDmmaSmemBytes, s>>>(Lt + t0, ld, n_valid, n_chunks, nullptr,
                                                                         S + origin, ctl, n_store, sp);
  }
  BA_LAUNCH_CHECK();
  return BA_OK;
}

int launch_k3(ba_engine* e, bool conditional, cudaStream_t s) {
  const ba_lm_state* ctl = conditional ? e->ctl : nullptr;
  {
    const int n = e->M * 90;
    stage_camera_blocks_kernel<<<(n + 255) / 256, 256, 0, s>>>(n, e->Uloc, e->U(), ctl);
    BA_LAUNCH_CHECK();
  }
  if (e->dense) return syrk_launch(&e->syrk, e->Yt, e->P(), ctl, s, e);
  return launch_schur_sparse(e, ctl, s);
}

// Host-only check of the planner (no device needed): every tile's pieces must tile [0, n_chunks)
// exactly once, in ascending order.
int syrk_plan_selftest(int n_cams, int64_t n_points, int tile, int num_sms, int* n_items, int* n_tiles,
                       double* makespan_rows, double* ideal_rows) {
  const int n_pad = (9 * n_cams + 1 + 7) / 8 * 8;
  const int64_t k_pad = (3 * n_points + 31) / 32 * 32;
  if (tile != 64 && tile != 128) { set_error("tile must be 64 or 128"); return BA_ERR_INVALID; }
  const SyrkPlan& plan = cached_plan(n_pad, tile, k_pad, num_sms);
  const int64_t n_chunks = k_pad / syrk_kc(tile);
  const int nt = (int)plan.tile_first.size() - 1;
  double work = 0.0;
  const int nt1_all = (n_pad + tile - 1) / tile;
  for (int t = 0; t < nt; ++t) {
    int64_t pos = 0;
    {
      // a thin tile folded into the tall tile above it: as many second slots as that tile has pieces
      int ti = 0;
      while ((ti + 1) * (ti + 2) / 2 <= t) ++ti;
      const int tj = t - ti * (ti + 1) / 2;
      if (plan.tall_row >= 0 && ti == nt1_all - 1 && tj < plan.tall_row) {
        const int tt = plan.tall_row * (plan.tall_row + 1) / 2 + tj;
        const int cnt = plan.tile_first[t + 1] - plan.tile_first[t];
        if (cnt != plan.tile_first[tt + 1] - plan.tile_first[tt]) { set_error("plan: thin tile %d has %d slots", t, cnt); return BA_ERR_STATE; }
        for (int k = 0; k < cnt; ++k) {
          const int slot = plan.tile_items[plan.tile_first[t] + k];
          const SyrkItem& it = plan.items[plan.tile_items[plan.tile_first[tt] + k]];
          if (slot < (int)plan.items.size() || slot >= plan.n_slots || it.slot2 != slot) { set_error("plan: thin tile %d slot %d", t, slot); return BA_ERR_STATE; }
        }
        continue;
      }
    }
    for (int k = plan.tile_first[t]; k < plan.tile_first[t + 1]; ++k) {
      const SyrkItem& it = plan.items[plan.tile_items[k]];
      int ti = 0;
      while ((ti + 1) * (ti + 2) / 2 <= t) ++ti;
      if (it.ti != ti || it.tj != t - ti * (ti + 1) / 2 || it.c_lo != pos || it.c_hi <= it.c_lo) {
        set_error("plan: tile %d piece %d covers [%d, %d), expected to start at %lld", t, k, it.c_lo, it.c_hi, (long long)pos);
        return BA_ERR_STATE;
      }
      pos = it.c_hi;
    }
    if (pos != n_chunks) { set_error("plan: tile %d ends at chunk %lld of %lld", t, (long long)pos, (long long)n_chunks); return BA_ERR_STATE; }
    int ti = 0;
    while ((ti + 1) * (ti + 2) / 2 <= t) ++ti;
    work += tile_weight(tile, ti, t - ti * (ti + 1) / 2, n_pad, k_pad) * (double)k_pad;
  }
  if (n_items) *n_items = (int)plan.items.size();
  if (n_tiles) *n_tiles = nt;
  if (makespan_rows) *makespan_rows = plan.makespan;
  if (ideal_rows) *ideal_rows = work / num_sms;
  return BA_OK;
}

}  // namespace ba
