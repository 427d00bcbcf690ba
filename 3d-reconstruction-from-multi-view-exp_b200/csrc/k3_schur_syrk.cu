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
// Pipeline: cp.async (LDGSTS) 16-byte copies, 3 stages of KC k-rows, shared-memory rows padded
// to TILE+4 doubles (stride = 4 mod 16: the 8-byte fragment loads of a half-warp hit 16
// distinct bank pairs -- ncu: 0 bank conflicts).
//
// Compute roofline (FP64 tensor): algorithmic flops = 3N * n (n + 1), n = 9M - 7.
//
// Large dense products (C3: n_pad^2 k_pad = 9.8e11) run instead on the INT8 tensor cores, FP64-accurate
// through the modular Ozaki scheme (see "FP64-accurate product on the INT8 tensor cores" below):
// emu_colmax_kernel and emu_residue_kernel turn Yt into 16 int8 residue planes, syrk_i8_pair_kernel
// (tcgen05.mma kind::i8 on pairs of SMs) forms one SYRK per modulus, emu_reconstruct_kernel lifts the exact integer
// products back to FP64 into P.  The DMMA kernels stay for smaller products (C2), the Cholesky's
// trailing updates and the projective-depth Gram matrix.  BA_SYRK_EMU=0|1 overrides the size rule.
//
// Sparse visibility: see k3_schur_sparse.cu (output-stationary, no atomics).
#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <functional>
#include <mutex>
#include <queue>
#include <vector>

#include "ba_common.cuh"

namespace ba {

constexpr int kStages = 3;

__device__ __forceinline__ void cp_async16_zfill(void* smem, const void* gmem, int src_bytes) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(sa), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

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

// TILE x TILE output tile per CTA; WR x WC warps, each owning a (TILE/WR) x (TILE/WC) sub-tile.
// SUB = false: the tile of this split is written to part[split][tile] (Schur product).
// SUB = true:  one split; the tile is subtracted in place from the lower triangle of the n_store x
//              n_store matrix `part` (leading dimension ld) -- the rank-k trailing update of the
//              blocked Cholesky (k4_cholesky.cu), where Yt is the k-major copy of a block column.
template <int TILE, int WR, int WC, int KC, bool SUB>
__global__ void __launch_bounds__(WR* WC * 32)
syrk_dmma_kernel(const double* __restrict__ Yt, int ld, int n_valid, int64_t n_chunks,
                 const SyrkItem* __restrict__ items, double* __restrict__ part,
                 const ba_lm_state* ctl, int n_store, SubSplit sp) {
  if (ctl && ctl->done) return;
  constexpr int NT = WR * WC * 32;
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
  // on different scheduler partitions, so the 10 (of 16) live warps of a 128-tile load the four
  // FP64 pipes 3/3/2/2 instead of 4/3/2/1 -- and the remaining warps only help with the copies.
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
  if (SUB) {
    // S -= acc on the lower triangle; an accumulator pair sits at (r, c), (r, c + 1), c even
#pragma unroll
    for (int i = 0; i < FM; ++i)
#pragma unroll
      for (int j = 0; j < FN; ++j) {
        const int r = ti * TILE + orow + 8 * i, c = tj * TILE + ocol + 8 * j;
        if (r >= n_store || c > r) continue;
        const size_t off = (size_t)r * ld + c;
        double* p = part + off;
        const bool push = sp.world > 1 && tj * TILE < sp.push_cols;
        if (c + 1 <= r) {
          double2 v = *reinterpret_cast<double2*>(p);
          v.x -= acc[i][j][0];
          v.y -= acc[i][j][1];
          *reinterpret_cast<double2*>(p) = v;
          if (push)
            for (int q = 0; q < sp.world; ++q)
              if (q != sp.rank) *reinterpret_cast<double2*>(sp.peer[q] + off) = v;
        } else {
          const double v = *p - acc[i][j][0];
          *p = v;
          if (push)
            for (int q = 0; q < sp.world; ++q)
              if (q != sp.rank) sp.peer[q][off] = v;
        }
      }
    return;
  }
  // partial tile of this item: part[item][TILE][TILE]
  double* out = part + (size_t)blockIdx.x * TILE * TILE;
#pragma unroll
  for (int i = 0; i < FM; ++i)
#pragma unroll
    for (int j = 0; j < FN; ++j)
      *reinterpret_cast<double2*>(out + (size_t)(orow + 8 * i) * TILE + ocol + 8 * j) =
          make_double2(acc[i][j][0], acc[i][j][1]);
}

// ---- 128-tiles fed by TMA ------------------------------------------------------------------------
// The same product with a Blackwell-native operand feed.  ncu on the cp.async kernel at C3: every
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

// Epilogue of one accumulator pair at tile-local (rl, cl), cl even: into the item's partial tile
// (`part` points at it), or (SUB) subtracted in place from the lower triangle of S (`part`), with
// the peer stores of a divided update.
template <bool SUB>
__device__ __forceinline__ void syrk_store_pair(double v0, double v1, int ti, int tj, int rl, int cl, int ld,
                                                int n_store, double* __restrict__ part, const SubSplit& sp) {
  constexpr int TILE = kTmaTile;
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

// One CTA runs a list of SEGMENTS (work items: tile x k-range), items[cta_first[b] .. cta_first[b + 1])
// -- one item per CTA when cta_first is null (large operands: the planner cuts whole waves of items
// in k-major order so that a k-slab stays in the L2), several for small operands (stream-K: every
// CTA gets the same modelled work, crossing tile boundaries).  The TMA ring runs across segment
// boundaries: the elected thread keeps its own cursor two to three chunks ahead of the warps, so the
// pipeline is filled once per CTA, not once per item.  The slot of an item's partial tile is its
// index in `items`.
template <bool SUB>
__global__ void __launch_bounds__(kTmaThreads, 1)
syrk_tma_kernel(const __grid_constant__ CUtensorMap tmapA, const __grid_constant__ CUtensorMap tmapB, int ld,
                int n_valid, int64_t n_chunks, const SyrkItem* __restrict__ items, const int* __restrict__ cta_first,
                double* __restrict__ part, const ba_lm_state* ctl, int n_store, SubSplit sp) {
  if (ctl && ctl->done) return;
  constexpr int TILE = kTmaTile, KC = kTmaKC, LDA = kTmaLda, LDB = kTmaLdb, WR = 4, WC = 4;
  constexpr int WM = TILE / WR, WN = TILE / WC, FM = WM / 8, FN = WN / 8;
  extern __shared__ unsigned char smem_raw[];

  int seg_lo = blockIdx.x, seg_hi = blockIdx.x + 1;
  if (!SUB && cta_first) { seg_lo = cta_first[blockIdx.x]; seg_hi = cta_first[blockIdx.x + 1]; }
  // segment `seg` -> tile, first chunk, chunks, second slot
  auto segment = [&](int seg, int& ti, int& tj, int& c_lo, int& nk, int& slot2) {
    if (SUB) {
      tile_from_linear(seg, ti, tj);
      c_lo = 0;
      nk = (int)n_chunks;
      slot2 = -1;
    } else {
      const SyrkItem it = items[seg];
      ti = it.ti; tj = it.tj; c_lo = it.c_lo; nk = it.c_hi > it.c_lo ? it.c_hi - it.c_lo : 0; slot2 = it.slot2;
    }
  };
  if (SUB) {
    int ti, tj;
    tile_from_linear(blockIdx.x, ti, tj);
    if (sp.world > 1 && (sp.tile_row0 + ti) % sp.world != sp.rank) return;  // another rank's tile row
  }

  // carve shared memory: operand stages (128-byte aligned for the TMA unit), then the mbarriers
  const unsigned base = (smem_u32(smem_raw) + 127u) & ~127u;
  const double* stages = reinterpret_cast<const double*>(smem_raw + (base - smem_u32(smem_raw)));
  constexpr int kStageDoubles = kTmaADoubles + kTmaBDoubles;
  const unsigned bars = base + kTmaStages * kTmaStageBytes;
  auto full_bar = [&](int st) { return bars + 8u * st; };
  auto empty_bar = [&](int st) { return bars + 8u * (kTmaStages + st); };

  // ---- the elected thread's side of the ring: a cursor over the chunks of all segments ----------
  int pseg = seg_lo - 1, pkc = 0, pnk = 0;   // cursor: segment, next chunk in it, its chunk count
  int pti = 0, ptj = 0, pclo = 0;            // ... and its tile / first chunk (kept in registers:
                                             // the item is read from global memory once per segment)
  unsigned issued = 0;                       // chunks issued so far = global index of the next one
  auto issue_next = [&]() {                  // thread 0 only
    while (pkc >= pnk) {
      if (++pseg >= seg_hi) { pseg = seg_hi; return; }
      int slot2;
      segment(pseg, pti, ptj, pclo, pnk, slot2);
      pkc = 0;
    }
    const int st = (int)(issued % kTmaStages);
    const unsigned dst = base + (unsigned)st * kTmaStageBytes;
    const int row = (pclo + pkc) * KC;
    const bool dg = pti == ptj;
    mbar_arrive_expect_tx(full_bar(st), kTmaABytes + (dg ? 0u : kTmaBBytes));
    tma_load_2d(dst, &tmapA, pti * TILE, row, full_bar(st));
    if (!dg) tma_load_2d(dst + kTmaABytes, &tmapB, ptj * TILE, row, full_bar(st));
    ++issued;
    ++pkc;
  };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int st = 0; st < kTmaStages; ++st) {
      mbar_init(full_bar(st), 1);
      mbar_init(empty_bar(st), kTmaThreads / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int k = 0; k < kTmaStages; ++k) issue_next();
  }
  __syncthreads();
  // Before global chunk g is computed the elected thread refills the stage of chunk g - 1 with the
  // next chunk not yet issued (every warp is done with chunk g - 1 or about to be: the wait on
  // `empty` is short).
  auto refill = [&](unsigned g) {
    if (warp == 0) {
      if (lane == 0 && g >= 1 && issued == g + kTmaStages - 1) {
        mbar_wait(empty_bar((int)((g - 1) % kTmaStages)), ((g - 1) / kTmaStages) & 1u);
        issue_next();
      }
      __syncwarp();
    }
  };
  const int kq = lane & 3;
  unsigned g = 0;  // global chunk counter of this CTA

  for (int seg = seg_lo; seg < seg_hi; ++seg) {
    int ti, tj, c_lo_unused, nk, slot2;
    segment(seg, ti, tj, c_lo_unused, nk, slot2);
    const bool diag = ti == tj;
    const bool tall = slot2 >= 0;
    double* const slot_part = SUB ? part : part + (size_t)seg * TILE * TILE;

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
      for (int kc = 0; kc < nk; ++kc, ++g) {
        refill(g);
        const int st = (int)(g % kTmaStages);
        mbar_wait(full_bar(st), (g / kTmaStages) & 1u);
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
        syrk_store_pair<SUB>(dacc[j][0], dacc[j][1], ti, ti, 8 * (hi ? r_hi : r_lo) + (lane >> 2),
                             8 * (hi ? c_hi0 + j : j - n_hi) + 2 * (lane & 3), ld, n_store, slot_part, sp);
      }
      continue;
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

    for (int kc = 0; kc < nk; ++kc, ++g) {
      refill(g);
      const int st = (int)(g % kTmaStages);
      mbar_wait(full_bar(st), (g / kTmaStages) & 1u);
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
        syrk_store_pair<SUB>(acc[i][j][0], acc[i][j][1], ti, tj, orow + 8 * i, ocol + 8 * j, ld, n_store, slot_part, sp);
    if (xvalid) {
      // the ragged rows below the tile: rows 0.. of the thin tile's partial slot (never with SUB)
      double* xp = part + (size_t)slot2 * TILE * TILE + (size_t)(8 * (wr & 1) + (lane >> 2)) * TILE;
#pragma unroll
      for (int e = 0; e < 2; ++e)
        *reinterpret_cast<double2*>(xp + wc * WN + 8 * (xj + e) + 2 * (lane & 3)) = make_double2(xacc[e][0], xacc[e][1]);
    }
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

// e_a for a column whose largest |entry| has the bit pattern `maxbits`: max 2^e_a < 2^b
__device__ __forceinline__ int emu_exponent(unsigned long long maxbits, int b) {
  if (maxbits == 0) return 0;
  return b - 1 - ilogb(__longlong_as_double((long long)maxbits));
}

// Column maxima of |Yt| as bit patterns (the order of an integer max does not matter).
__global__ void __launch_bounds__(128)
emu_colmax_kernel(const double* __restrict__ Yt, int64_t k_pad, int n_pad, unsigned long long* __restrict__ colmax,
                  const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;
  const int a = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
  if (a >= n_pad) return;
  const int64_t rows = (k_pad + gridDim.y - 1) / gridDim.y;
  const int64_t k0 = (int64_t)blockIdx.y * rows, k1 = k0 + rows < k_pad ? k0 + rows : k_pad;
  constexpr unsigned long long kAbs = 0x7FFFFFFFFFFFFFFFull;
  unsigned long long m0 = 0, m1 = 0;
#pragma unroll 8
  for (int64_t k = k0; k < k1; ++k) {
    const double2 v = __ldg(reinterpret_cast<const double2*>(Yt + k * n_pad + a));
    m0 = max(m0, (unsigned long long)__double_as_longlong(v.x) & kAbs);
    m1 = max(m1, (unsigned long long)__double_as_longlong(v.y) & kAbs);
  }
  if (m0) atomicMax(colmax + a, m0);
  if (m1) atomicMax(colmax + a + 1, m1);
}

// Symmetric residue of the integer v (|v| <= 2^53) modulo p_I as an int in [-128, 127]: q = rint(v / p)
// through the 1.5 * 2^52 rounding constant (|v / p| < 2^46), r = v - p q exact.  1 / p is rounded, so
// q can miss the nearest integer by one when v / p lies within 0.0052 of a half: |r| <= 128.8.
// (Called from fully unrolled loops: p and 1 / p are compile-time constants.)
__device__ __forceinline__ int emu_residue(double v, int i) {
  const double p = (double)emu_modulus(i), inv = 1.0 / p, magic = 6755399441055744.0;
  const double q = __dadd_rn(__fma_rn(v, inv, magic), -magic);
  const double r = __fma_rn(-p, q, v);
  const int ri = __double2loint(__dadd_rn(r, magic));
  return ri > 127 ? ri - (int)p : ri;
}

// Residue planes Yq[i][a][k] (K-major) from Yt[k][a]: a block converts 64 k-rows x 32 columns,
// transposing through shared memory -- rows are read as 256-byte segments, plane rows written as
// 64-byte segments.  48 KB of shared memory and <= 64 registers: four blocks (32 warps) per SM.
constexpr int kResTK = 64, kResTA = 32, kResThreads = 256;
constexpr size_t kResSmemBytes = (size_t)kResTK * kResTA * sizeof(double) + (size_t)kEmuModuli * kResTA * kResTK;

__global__ void __launch_bounds__(kResThreads, 4)
emu_residue_kernel(const double* __restrict__ Yt, int64_t k_pad, int n_pad, const unsigned long long* __restrict__ colmax,
                   int bits, int8_t* __restrict__ Yq, const ba_lm_state* ctl) {
  if (ctl && ctl->done) return;
  extern __shared__ __align__(16) unsigned char res_smem[];
  double* sIn = reinterpret_cast<double*>(res_smem);  // [64 k][32 a]
  uint2* sOut = reinterpret_cast<uint2*>(res_smem + kResTK * kResTA * sizeof(double));  // [16][32 a][8 x 8 bytes]
  const int64_t k0 = (int64_t)blockIdx.x * kResTK;
  const int a0 = blockIdx.y * kResTA;
  const int t = threadIdx.x;
  for (int q = t; q < kResTK * kResTA / 2; q += kResThreads) {
    const int row = q / (kResTA / 2), cp = q % (kResTA / 2);
    const int a = a0 + 2 * cp;
    const int64_t k = k0 + row;
    double2 v = make_double2(0.0, 0.0);
    if (k < k_pad && a < n_pad) v = __ldg(reinterpret_cast<const double2*>(Yt + k * n_pad + a));
    reinterpret_cast<double2*>(sIn)[q] = v;
  }
  __syncthreads();
  // thread: column a0 + lane, k-rows 8 w .. 8 w + 7; its 8 residues of a plane are one 8-byte piece,
  // stored at piece w ^ (lane & 6) of the column's 64-byte row (the XOR keeps the two pieces of every
  // 16-byte chunk adjacent and in order, and spreads the stores over the banks)
  const int lane = t & 31, w = t >> 5;
  const int e = a0 + lane < n_pad ? emu_exponent(colmax[a0 + lane], bits) : 0;
  double v[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] = rint(ldexp(sIn[(8 * w + j) * kResTA + lane], e));
#pragma unroll
  for (int i = 0; i < kEmuModuli; ++i) {
    uint32_t word[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int r0 = emu_residue(v[4 * u], i), r1 = emu_residue(v[4 * u + 1], i);
      const int r2 = emu_residue(v[4 * u + 2], i), r3 = emu_residue(v[4 * u + 3], i);
      word[u] = __byte_perm(__byte_perm(r0, r1, 0x0040), __byte_perm(r2, r3, 0x0040), 0x5410);
    }
    sOut[(i * kResTA + lane) * 8 + (w ^ (lane & 6))] = make_uint2(word[0], word[1]);
  }
  __syncthreads();
  // 16-byte chunks: 16 planes x 32 columns x 4 chunks, two planes per pass of the block
  const int sa = (t >> 2) & 31, c = t & 3, ih = t >> 7;
  const int ga = a0 + sa;
  const int64_t gk = k0 + 16 * c;  // k_pad is a multiple of 32: a chunk is all in or all out
  if (ga >= n_pad || gk >= k_pad) return;
#pragma unroll
  for (int i = ih; i < kEmuModuli; i += 2)
    *reinterpret_cast<uint4*>(Yq + ((size_t)i * n_pad + ga) * k_pad + gk) =
        *reinterpret_cast<const uint4*>(sOut + (i * kResTA + sa) * 8 + ((2 * c) ^ (sa & 6)));
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
static inline int syrk_kc(int tile) { return tile == 128 ? 32 : 16; }
static inline int syrk_occupancy(int tile) { return tile == 128 ? 1 : 4; }

int syrk_feed_is_tma();
// The planner's view of the feed: BA_SYRK_PLAN_ASSUME_TMA=1 lets the host-only self-check of the
// plan (ba_syrk_plan_info, run on CPU boxes) exercise the TMA kernel's tile shapes.
static bool plan_for_tma() {
  static const bool assume = std::getenv("BA_SYRK_PLAN_ASSUME_TMA") != nullptr;
  return assume || syrk_feed_is_tma();
}

// Relative duration of a tile per k-row (1 = full tile), mirroring the kernel's warp mapping:
// edge tiles skip the 8x8 fragments beyond n_valid, diagonal tiles the sub-tiles above the
// diagonal.  A warp sits on scheduler partition (warp % 4) with its own FP64 pipe: a CTA that has
// an SM to itself takes as long as its busiest partition; with several CTAs per SM the partitions
// even out and the mean counts.
static double tile_weight(int TILE, int WR, int WC, int occ, int ti, int tj, int n_valid, int64_t k_pad = 0,
                          double floor_override = -1.0) {
  const int WM = TILE / WR, WN = TILE / WC, FM = WM / 8, FN = WN / 8;
  double load[4] = {0, 0, 0, 0};
  const bool tma_tile = TILE == kTmaTile && occ == 1 && plan_for_tma();
  const bool folded_diag = ti == tj && tma_tile;

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
  // (floor 1.0: 0.302 ms per iteration, 0.75: 0.309, 0.5: 0.344, 0.35: 0.430); the 128-tile
  // kernel with floor 0.75 (1.0: 0.326, 0.75: 0.283, 0.5: 0.343, 0.35: 0.355).
  // The TMA-fed kernel has no per-row copy instructions to pay for: a thin tile costs what its
  // fragments cost, down to the rate at which the TMA unit streams the rows (measured floor ~0.3).
  // Measured with the TMA kernel (B200): C3 (4.3 GB operand, ~3300-row pieces) floor 0.5: 28.79 ms,
  // 0.3: 28.86, 0.15: 28.86, 0.75: 29.42; C2 (108 MB operand, two waves of ~730-row pieces) floor
  // 1.0: 0.286 ms, 0.5: 0.298, 0.3: 0.311 -- with two waves the schedule is decided by whole items,
  // and uniform cuts pack them best.
  const bool small_operand = k_pad > 0 && (double)k_pad * n_valid * 8.0 <= 256.0 * 1024 * 1024;
  double floor_w = occ == 1 ? (plan_for_tma() ? (small_operand ? 1.0 : 0.5) : 0.75) : 1.0;
  if (const char* f = std::getenv("BA_SYRK_FLOOR")) floor_w = std::atof(f);  // tuning experiments only
  if (floor_override >= 0.0) floor_w = floor_override;
  return w > floor_w ? w : floor_w;
}

struct SyrkPlan {
  std::vector<SyrkItem> items;       // launch order: ascending k range, then tile
  std::vector<int> tile_first;       // [n_tiles + 1]
  std::vector<int> tile_items;       // partial-tile slot per (tile, piece), pieces in ascending k order
  std::vector<int> cta_first;        // stream-K plans: [n_ctas + 1] first item of every CTA (else empty)
  int n_slots = 0;                   // partial tiles: one per item + one per tall item (its thin tile below)
  int tall_row = -1;                 // tile row whose off-diagonal tiles also compute the ragged rows below
  double makespan = 0.0;             // modelled duration in k-rows of a full tile on one SM slot
};

// The ragged last tile row is folded into the row above (see kTmaTallRows) when the TMA kernel runs
// and at most kTmaTallRows rows are left over: returns that row (nt1 - 2), else -1.
static int tall_tile_row(int n_pad, int TILE, int occ) {
  static const bool off = std::getenv("BA_SYRK_NO_TALL") != nullptr;  // A/B timing only
  const int nt1 = (n_pad + TILE - 1) / TILE;
  const int left = n_pad - (nt1 - 1) * TILE;
  if (off || TILE != kTmaTile || occ != 1 || !plan_for_tma() || nt1 < 3 || left > kTmaTallRows) return -1;
  return nt1 - 2;
}

// Cut every tile's K range into pieces so that all CTAs take about the same time and their number
// fills whole waves of SM slots: pieces(t) ~ weight(t) x S.  S is chosen by simulating the block
// scheduler (CTAs start in launch order on the first free slot) for every admissible S and
// keeping the shortest schedule.  Constraints: a piece streams >= 512 k-rows (prologue, epilogue
// and the partial-tile write stay small against it), and -- L2 residency -- the k-slab that the
// CTAs of one "column" of the schedule share should stay below 48 MB: ncu showed 18.6 GB of DRAM
// reads for the 4.3 GB operand of C3 when 271 MB slabs were streamed by tiles drifting apart.
static SyrkPlan plan_syrk(int n_pad, int TILE, int WR, int WC, int64_t k_pad, int num_sms) {
  const int KC = syrk_kc(TILE), occ = syrk_occupancy(TILE);
  const int nt1 = (n_pad + TILE - 1) / TILE;
  const int n_tiles = nt1 * (nt1 + 1) / 2;
  const int64_t n_chunks = k_pad / KC;
  const int slots = num_sms * occ;
  std::vector<double> w(n_tiles), w_run(n_tiles);  // w: decides the cuts; w_run: the modelled duration per k-row
  static const char* lpt_env = std::getenv("BA_SYRK_LPT");  // "0" / "1": A/B timing
  const bool lpt = lpt_env ? std::atoi(lpt_env) != 0 : (double)k_pad * n_pad * 8.0 <= 116.0 * 1024 * 1024;
  static const double run_floor = std::getenv("BA_SYRK_RUN_FLOOR") ? std::atof(std::getenv("BA_SYRK_RUN_FLOOR")) : 0.5;
  const int tall_row = tall_tile_row(n_pad, TILE, occ);
  // absorbed[t]: thin tile (nt1 - 1, tj), tj < tall_row: computed by the tall tile (tall_row, tj)
  std::vector<char> absorbed(n_tiles, 0), is_tall(n_tiles, 0);
  for (int t = 0, ti = 0; ti < nt1; ++ti)
    for (int tj = 0; tj <= ti; ++tj, ++t) {
      w[t] = tile_weight(TILE, WR, WC, occ, ti, tj, n_pad, k_pad);
      // longest-first schedules are simulated with what a tile really costs (its fragments, down to
      // the rate of the TMA ring), not with the weight that decides the cuts
      w_run[t] = lpt ? tile_weight(TILE, WR, WC, occ, ti, tj, n_pad, k_pad, run_floor) : w[t];
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

// Small operands (the whole of Y^T stays in the 126 MB L2, so the order in which k-ranges are
// visited does not matter): stream-K.  With whole items the C2 product is two waves of ~1000-row
// items on 148 SMs -- the schedule, not the kernel, bounds it at 0.55 of the DMMA peak.  Here the
// modelled work (tile weight x chunks, tile by tile) is dealt to one CTA per SM in equal shares,
// crossing tile boundaries; a CTA's segments run through one TMA ring (syrk_tma_kernel), so the
// pipeline is filled once per CTA.  Every segment still writes its own partial tile, and the tiles
// are summed in ascending k order as before: deterministic.
static SyrkPlan plan_streamk(int n_pad, int64_t k_pad, int num_sms) {
  constexpr int TILE = kTmaTile, KC = kTmaKC;
  const int nt1 = (n_pad + TILE - 1) / TILE;
  const int n_tiles = nt1 * (nt1 + 1) / 2;
  const int64_t n_chunks = k_pad / KC;
  std::vector<double> w(n_tiles);
  for (int t = 0, ti = 0; ti < nt1; ++ti)
    for (int tj = 0; tj <= ti; ++tj, ++t) {
      // executed 8 x 8 fragments per k-step against the 256 of a full tile; a thin tile is bound by
      // the ring's latency instead (measured ~0.3)
      const int rows = std::min(16, (n_pad - ti * TILE + 7) / 8);
      const double frags = ti == tj ? rows * (rows + 1) / 2.0 : rows * 16.0;
      w[t] = std::max(0.3, frags / 256.0);
    }
  const int64_t min_seg = 4;       // chunks
  const double seg_cost = 1.5;     // chunks of a full tile: accumulator hand-over and the partial-tile store
  double total = 0.0;
  for (int t = 0; t < n_tiles; ++t) total += w[t] * (double)n_chunks + seg_cost;
  const int G = num_sms;
  const double budget = total / G + seg_cost;
  SyrkPlan plan;
  plan.tile_first.assign(n_tiles + 1, 0);
  plan.cta_first.assign(1, 0);
  int cta = 0;
  double left = budget;
  auto next_cta = [&]() {
    plan.cta_first.push_back((int)plan.items.size());
    ++cta;
    left = budget;
  };
  for (int t = 0, ti = 0; ti < nt1; ++ti)
    for (int tj = 0; tj <= ti; ++tj, ++t) {
      int64_t pos = 0;
      while (pos < n_chunks) {
        const int64_t rem = n_chunks - pos;
        int64_t can = (int64_t)std::floor((left - seg_cost) / w[t]);
        if (cta == G - 1) can = rem;  // the last CTA takes whatever is left
        if (can < min_seg && cta < G - 1) { next_cta(); continue; }
        int64_t take = std::min<int64_t>(rem, std::max<int64_t>(can, min_seg));
        if (rem - take < min_seg) take = rem;  // no crumbs
        plan.tile_items.push_back((int)plan.items.size());
        plan.items.push_back({ti, tj, (int)pos, (int)(pos + take), -1});
        pos += take;
        left -= (double)take * w[t] + seg_cost;
      }
      plan.tile_first[t + 1] = (int)plan.items.size();
    }
  while ((int)plan.cta_first.size() < G + 1) plan.cta_first.push_back((int)plan.items.size());
  plan.n_slots = (int)plan.items.size();
  plan.makespan = budget * KC;
  return plan;
}

// Measured on B200 (C2, 50 cameras x 10k points): 0.82 ms against 0.29 ms with whole items in k-major
// order -- with every CTA streaming its own (tile, k-range) nothing is shared between the SMs any
// more and the thin tiles' long k-ranges become the makespan.  The plan and the multi-segment kernel
// are kept behind BA_SYRK_STREAMK=1 for the next attempt (k-major dealing of equal shares).
static bool use_streamk(int n_pad, int tile, int64_t k_pad) {
  static const bool on = std::getenv("BA_SYRK_STREAMK") != nullptr;
  return on && tile == kTmaTile && plan_for_tma() && (double)k_pad * n_pad * 8.0 <= 128.0 * 1024 * 1024;
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
  SyrkPlan* p = new SyrkPlan(use_streamk(n_pad, tile, k_pad) ? plan_streamk(n_pad, k_pad, num_sms)
                             : tile == 128 ? plan_syrk(n_pad, 128, 4, 4, k_pad, num_sms)
                                           : plan_syrk(n_pad, 64, 2, 2, k_pad, num_sms));
  cache.push_back({Key{n_pad, tile, k_pad, num_sms}, p});
  return *p;
}

// Plans the dense Schur product of this engine and uploads the work items.
static int emu_plan_engine(ba_engine* e);
int emu_bits_for(int64_t k_pad);
static bool emu_select(const ba_engine* e);

int syrk_plan_engine(ba_engine* e) {
  if (!e->dense) return BA_OK;
  e->emu_bits = emu_bits_for(e->k_pad);
  e->syrk_emu = emu_select(e) ? 1 : 0;
  if (e->syrk_emu) return emu_plan_engine(e);
  const SyrkPlan& plan = cached_plan(e->n_pad, e->syrk_tile, e->k_pad, e->num_sms);
  e->syrk_n_items = (int)plan.items.size();
  e->syrk_n_ctas = plan.cta_first.empty() ? e->syrk_n_items : (int)plan.cta_first.size() - 1;
  if (!plan.cta_first.empty()) {
    BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&e->syrk_cta_first), plan.cta_first.size() * sizeof(int), (cudaStream_t)0));
    BA_CUDA(cudaMemcpy(e->syrk_cta_first, plan.cta_first.data(), plan.cta_first.size() * sizeof(int), cudaMemcpyHostToDevice));
  }
  const int nt1 = (e->n_pad + e->syrk_tile - 1) / e->syrk_tile;
  e->syrk_n_tiles = nt1 * (nt1 + 1) / 2;
  const size_t tt = (size_t)e->syrk_tile * e->syrk_tile;
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&e->syrk_items), plan.items.size() * sizeof(SyrkItem), (cudaStream_t)0));
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&e->syrk_tile_first), plan.tile_first.size() * sizeof(int), (cudaStream_t)0));
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&e->syrk_tile_items), plan.tile_items.size() * sizeof(int), (cudaStream_t)0));
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&e->Spart), (size_t)plan.n_slots * tt * sizeof(double), (cudaStream_t)0));
  BA_CUDA(cudaMemcpy(e->syrk_items, plan.items.data(), plan.items.size() * sizeof(SyrkItem), cudaMemcpyHostToDevice));
  BA_CUDA(cudaMemcpy(e->syrk_tile_first, plan.tile_first.data(), plan.tile_first.size() * sizeof(int), cudaMemcpyHostToDevice));
  BA_CUDA(cudaMemcpy(e->syrk_tile_items, plan.tile_items.data(), plan.tile_items.size() * sizeof(int), cudaMemcpyHostToDevice));
  if (std::getenv("BA_TIMING"))
    std::fprintf(stderr, "[ba syrk plan] tile %d: %d tiles, %d items on %d slots, modelled %.0f k-rows (ideal %.0f)\n",
                 e->syrk_tile, e->syrk_n_tiles, e->syrk_n_items, e->num_sms * syrk_occupancy(e->syrk_tile),
                 plan.makespan, 0.0);
  return BA_OK;
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

// BA_SYRK_NO_TMA=1 keeps the cp.async kernel (A/B timing).
static bool syrk_use_tma() {
  static const bool on = std::getenv("BA_SYRK_NO_TMA") == nullptr;
  return on;
}

int syrk_feed_is_tma() { return syrk_use_tma() && tensor_map_encoder() != nullptr; }

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
int emu_bits_for(int64_t k_pad) {
  unsigned __int128 half = 1;
  for (int i = 0; i < kEmuModuli; ++i) half *= (unsigned)emu_modulus(i);
  half /= 2;
  for (int b = 53; b > 0; --b)
    if ((unsigned __int128)k_pad < (half >> (2 * b))) return b;  // k_pad 2^(2b) < half, whole multiples of 2^(2b)
  return 0;
}

// The emulation is chosen when it is exact to (nearly) full FP64 input precision and the product is
// large enough for the INT8 tensor cores to pay for the conversion passes.  BA_SYRK_EMU=0|1 overrides
// the size rule (A/B timing and tests); it is read when an engine is created.
int syrk_emu_info(int64_t k_pad, int32_t* moduli, int* n_moduli, int* bits) {
  if (k_pad < 1) { set_error("k_pad must be positive"); return BA_ERR_INVALID; }
  if (moduli)
    for (int i = 0; i < kEmuModuli; ++i) moduli[i] = emu_modulus(i);
  if (n_moduli) *n_moduli = kEmuModuli;
  if (bits) *bits = emu_bits_for(k_pad);
  return BA_OK;
}

static bool emu_select(const ba_engine* e) {
  if (const char* v = std::getenv("BA_SYRK_EMU")) return std::atoi(v) != 0;
  return e->emu_bits >= 50 && tensor_map_encoder() != nullptr &&
         (double)e->n_pad * e->n_pad * (double)e->k_pad >= kEmuMinWork;
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

static int emu_plan_engine(ba_engine* e) {
  const EmuPlan plan = plan_emu(e->n_pad, e->k_pad, e->num_sms);
  std::vector<EmuItem> items = plan.full;
  items.insert(items.end(), plan.ragged.begin(), plan.ragged.end());
  const int nt1 = (e->n_pad + kEmuTile - 1) / kEmuTile;
  e->syrk_n_tiles = nt1 * (nt1 + 1) / 2;
  e->emu_n_items = (int)items.size();
  e->emu_n_full = (int)plan.full.size();
  const cudaStream_t s0 = (cudaStream_t)0;
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&e->emu_items), items.size() * sizeof(EmuItem), s0));
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&e->Yq), (size_t)kEmuModuli * e->n_pad * e->k_pad, s0));
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&e->Pmod),
                          (size_t)kEmuModuli * e->syrk_n_tiles * kEmuTile * kEmuTile * sizeof(uint32_t), s0));
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&e->colmax), (size_t)e->n_pad * sizeof(unsigned long long), s0));
  BA_CUDA(cudaMemcpy(e->emu_items, items.data(), items.size() * sizeof(EmuItem), cudaMemcpyHostToDevice));
  if (std::getenv("BA_TIMING"))
    std::fprintf(stderr, "[ba syrk plan] int8 emulation: b = %d, %d tiles x %d moduli, %d items\n", e->emu_bits,
                 e->syrk_n_tiles, kEmuModuli, e->emu_n_items);
  return BA_OK;
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

static int launch_syrk_emu(ba_engine* e, const ba_lm_state* ctl, cudaStream_t s) {
  CUtensorMap map;
  BA_TRY(make_plane_map(&map, e->Yq, e->n_pad, e->k_pad));
  BA_CUDA(cudaFuncSetAttribute(emu_residue_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kResSmemBytes));
  BA_CUDA(cudaFuncSetAttribute(syrk_i8_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEmuSmemBytes));
  BA_CUDA(cudaFuncSetAttribute(syrk_i8_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEmuSmemBytes));
  const int n_tiles = e->syrk_n_tiles;
  ProfScope ps(e, PG_SYRK, s);
  BA_CUDA(cudaMemsetAsync(e->colmax, 0, (size_t)e->n_pad * sizeof(unsigned long long), s));
  BA_CUDA(cudaMemsetAsync(e->Pmod, 0, (size_t)kEmuModuli * n_tiles * kEmuTile * kEmuTile * sizeof(uint32_t), s));
  {
    const int gx = (e->n_pad / 2 + 127) / 128;
    const int64_t gy = std::max<int64_t>(1, std::min<int64_t>(e->k_pad / 64, (int64_t)16 * e->num_sms / gx));
    emu_colmax_kernel<<<dim3(gx, (unsigned)gy), 128, 0, s>>>(e->Yt, e->k_pad, e->n_pad, e->colmax, ctl);
    BA_LAUNCH_CHECK();
  }
  emu_residue_kernel<<<dim3((unsigned)((e->k_pad + kResTK - 1) / kResTK), (e->n_pad + kResTA - 1) / kResTA),
                       kResThreads, kResSmemBytes, s>>>(e->Yt, e->k_pad, e->n_pad, e->colmax, e->emu_bits, e->Yq, ctl);
  BA_LAUNCH_CHECK();
  if (e->emu_n_full > 0) {
    syrk_i8_pair_kernel<false><<<2 * e->emu_n_full, kEmuThreads, kEmuSmemBytes, s>>>(map, e->emu_items, e->Pmod,
                                                                                     n_tiles, e->n_pad, ctl);
    BA_LAUNCH_CHECK();
  }
  if (e->emu_n_items > e->emu_n_full) {
    syrk_i8_pair_kernel<true><<<2 * (e->emu_n_items - e->emu_n_full), kEmuThreads, kEmuSmemBytes, s>>>(
        map, e->emu_items + e->emu_n_full, e->Pmod, n_tiles, e->n_pad, ctl);
    BA_LAUNCH_CHECK();
  }
  emu_reconstruct_kernel<<<dim3(n_tiles, 16), 256, 0, s>>>(e->Pmod, n_tiles, e->colmax, e->emu_bits, e->P(), e->n_pad,
                                                          e->n_pad, emu_consts(), ctl);
  BA_LAUNCH_CHECK();
  return BA_OK;
}

template <int TILE, int WR, int WC, int KC>
static int launch_syrk(ba_engine* e, const ba_lm_state* ctl, cudaStream_t s) {
  const int64_t n_chunks = e->k_pad / KC;
  if (TILE == kTmaTile && KC == kTmaKC && syrk_use_tma()) {
    CUtensorMap mapA, mapB;
    BA_TRY(make_operand_map(&mapA, e->Yt, e->n_pad, e->k_pad, e->n_pad, kTmaLda));
    BA_TRY(make_operand_map(&mapB, e->Yt, e->n_pad, e->k_pad, e->n_pad, kTmaLdb));
    BA_CUDA(cudaFuncSetAttribute(syrk_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)kTmaSmemBytes));
    ProfScope ps(e, PG_SYRK, s);
    syrk_tma_kernel<false><<<e->syrk_n_ctas, kTmaThreads, kTmaSmemBytes, s>>>(
        mapA, mapB, e->n_pad, e->n_pad, n_chunks, e->syrk_items, e->syrk_cta_first, e->Spart, ctl, 0,
        SubSplit{0, 1, 0, 0, {}});
    BA_LAUNCH_CHECK();
  } else {
    const size_t smem = (size_t)2 * kStages * KC * (TILE + 4) * sizeof(double);
    BA_CUDA(cudaFuncSetAttribute(syrk_dmma_kernel<TILE, WR, WC, KC, false>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ProfScope ps(e, PG_SYRK, s);
    syrk_dmma_kernel<TILE, WR, WC, KC, false><<<e->syrk_n_items, WR * WC * 32, smem, s>>>(
        e->Yt, e->n_pad, e->n_pad, n_chunks, e->syrk_items, e->Spart, ctl, 0, SubSplit{0, 1, 0, 0, {}});
    BA_LAUNCH_CHECK();
  }
  const int n_tiles = e->syrk_n_tiles;
  // enough blocks to fill the GPU (C2: 10 tiles x 8 slabs = 80 blocks took 33 us for 38 MB), at
  // least one pair of doubles per thread
  const int slabs_max = TILE * TILE / 2 / 256;
  int slabs = 1;
  while (slabs < slabs_max && n_tiles * slabs < 4 * e->num_sms) slabs *= 2;
  syrk_reduce_kernel<TILE><<<dim3(n_tiles, slabs), 256, 0, s>>>(e->Spart, e->syrk_tile_first,
                                                               e->syrk_tile_items, e->P(), e->n_pad,
                                                               e->n_pad, ctl);
  BA_LAUNCH_CHECK();
  return BA_OK;
}

// S[t0:, t0:] -= Lt[:, t0:]^T Lt[:, t0:]  (lower triangle, rows < n_rows) with Lt k-major
// [depth][ld]: the wide trailing update of the two-level blocked Cholesky.
template <int TILE, int WR, int WC, int KC>
static int launch_syrk_sub(double* S, int ld, int n_rows, int t0, const double* Lt, int depth,
                           const ba_lm_state* ctl, cudaStream_t s, const CholSplit* split) {
  const int n_store = n_rows - t0;
  const int n_valid = (n_store + 7) / 8 * 8;  // <= ld - t0: ld is a multiple of 8, t0 of 64
  const int nt1 = (n_valid + TILE - 1) / TILE;
  const int n_tiles = nt1 * (nt1 + 1) / 2;
  const int n_chunks = depth / KC;
  const size_t smem = (size_t)2 * kStages * KC * (TILE + 4) * sizeof(double);
  BA_CUDA(cudaFuncSetAttribute(syrk_dmma_kernel<TILE, WR, WC, KC, true>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const size_t origin = (size_t)t0 * ld + t0;
  SubSplit sp{0, 1, 0, 0, {}};
  if (split && split->world > 1) {
    sp.rank = split->rank;
    sp.world = split->world;
    sp.tile_row0 = t0 / TILE;
    sp.push_cols = split->push_cols;
    for (int q = 0; q < split->world; ++q) sp.peer[q] = split->S_peer[q] + origin;
  }
  if (TILE == kTmaTile && KC == kTmaKC && syrk_use_tma()) {
    CUtensorMap mapA, mapB;
    BA_TRY(make_operand_map(&mapA, Lt + t0, n_valid, depth, ld, kTmaLda));
    BA_TRY(make_operand_map(&mapB, Lt + t0, n_valid, depth, ld, kTmaLdb));
    BA_CUDA(cudaFuncSetAttribute(syrk_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)kTmaSmemBytes));
    syrk_tma_kernel<true><<<n_tiles, kTmaThreads, kTmaSmemBytes, s>>>(mapA, mapB, ld, n_valid, n_chunks, nullptr,
                                                                      nullptr, S + origin, ctl, n_store, sp);
    BA_LAUNCH_CHECK();
    return BA_OK;
  }
  syrk_dmma_kernel<TILE, WR, WC, KC, true><<<n_tiles, WR * WC * 32, smem, s>>>(
      Lt + t0, ld, n_valid, n_chunks, nullptr, S + origin, ctl, n_store, sp);
  BA_LAUNCH_CHECK();
  return BA_OK;
}

// 128-tiles (one CTA per SM) once there are enough of them, 64-tiles (four per SM) below.  Only
// the 128-tile form is divided over the ranks of a sharded run.
int launch_chol_wide_update(double* S, int ld, int n_rows, int t0, const double* Lt, int depth,
                            const ba_lm_state* ctl, cudaStream_t s, const CholSplit* split) {
  if (n_rows - t0 >= kCholSplitMinRows)
    return launch_syrk_sub<128, 4, 4, 32>(S, ld, n_rows, t0, Lt, depth, ctl, s, split);
  return launch_syrk_sub<64, 2, 2, 16>(S, ld, n_rows, t0, Lt, depth, ctl, s, nullptr);
}

int launch_k3(ba_engine* e, bool conditional, cudaStream_t s) {
  const ba_lm_state* ctl = conditional ? e->ctl : nullptr;
  {
    const int n = e->M * 90;
    stage_camera_blocks_kernel<<<(n + 255) / 256, 256, 0, s>>>(n, e->Uloc, e->U(), ctl);
    BA_LAUNCH_CHECK();
  }
  if (e->dense) {
    if (e->syrk_emu) return launch_syrk_emu(e, ctl, s);
    if (e->syrk_tile == 128) return launch_syrk<128, 4, 4, 32>(e, ctl, s);
    return launch_syrk<64, 2, 2, 16>(e, ctl, s);
  }
  return launch_schur_sparse(e, ctl, s);
}

// ---- Gram matrix of an arbitrary k-major operand (used by the projective-depth iteration) --------
// P = Yt^T Yt (lower triangle incl. the diagonal pairs) for Yt [k_pad][n_pad], with the 64-tile
// kernel and the same planner as the Schur product.
int gram_prepare(GramWorkspace* ws, int n_pad, int64_t k_pad, int num_sms, cudaStream_t s) {
  *ws = GramWorkspace();
  const SyrkPlan& plan = cached_plan(n_pad, 64, k_pad, num_sms);
  ws->n_pad = n_pad;
  ws->k_pad = k_pad;
  ws->num_sms = num_sms;
  ws->n_items = (int)plan.items.size();
  const int nt1 = (n_pad + 63) / 64;
  ws->n_tiles = nt1 * (nt1 + 1) / 2;
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws->items), plan.items.size() * sizeof(SyrkItem), s));
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws->tile_first), plan.tile_first.size() * sizeof(int), s));
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws->tile_items), plan.tile_items.size() * sizeof(int), s));
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws->Spart), plan.items.size() * (size_t)64 * 64 * sizeof(double), s));
  BA_CUDA(cudaMemcpyAsync(ws->items, plan.items.data(), plan.items.size() * sizeof(SyrkItem), cudaMemcpyHostToDevice, s));
  BA_CUDA(cudaMemcpyAsync(ws->tile_first, plan.tile_first.data(), plan.tile_first.size() * sizeof(int), cudaMemcpyHostToDevice, s));
  BA_CUDA(cudaMemcpyAsync(ws->tile_items, plan.tile_items.data(), plan.tile_items.size() * sizeof(int), cudaMemcpyHostToDevice, s));
  BA_CUDA(cudaStreamSynchronize(s));  // the plan's host vectors are cached, but keep the copies simple
  return BA_OK;
}

int gram_launch(const GramWorkspace* ws, const double* Yt, double* P, cudaStream_t s) {
  constexpr int TILE = 64, KC = 16;
  const size_t smem = (size_t)2 * kStages * KC * (TILE + 4) * sizeof(double);
  BA_CUDA(cudaFuncSetAttribute(syrk_dmma_kernel<TILE, 2, 2, KC, false>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  syrk_dmma_kernel<TILE, 2, 2, KC, false><<<ws->n_items, 128, smem, s>>>(
      Yt, ws->n_pad, ws->n_pad, ws->k_pad / KC, ws->items, ws->Spart, nullptr, 0, SubSplit{0, 1, 0, 0, {}});
  BA_LAUNCH_CHECK();
  int slabs = 1;
  while (slabs < TILE * TILE / 2 / 256 && ws->n_tiles * slabs < 4 * ws->num_sms) slabs *= 2;
  syrk_reduce_kernel<TILE><<<dim3(ws->n_tiles, slabs), 256, 0, s>>>(ws->Spart, ws->tile_first, ws->tile_items, P,
                                                                  ws->n_pad, ws->n_pad, nullptr);
  BA_LAUNCH_CHECK();
  return BA_OK;
}

void gram_release(GramWorkspace* ws, cudaStream_t s) {
  void* ptrs[] = {ws->items, ws->tile_first, ws->tile_items, ws->Spart};
  for (void* p : ptrs)
    if (p) cudaFreeAsync(p, s);
  *ws = GramWorkspace();
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
    work += tile_weight(tile, tile == 128 ? 4 : 2, tile == 128 ? 4 : 2, syrk_occupancy(tile), ti, t - ti * (ti + 1) / 2, n_pad, k_pad) * (double)k_pad;
  }
  if (n_items) *n_items = (int)plan.items.size();
  if (n_tiles) *n_tiles = nt;
  if (makespan_rows) *makespan_rows = plan.makespan;
  if (ideal_rows) *ideal_rows = work / num_sms;
  return BA_OK;
}

}  // namespace ba
