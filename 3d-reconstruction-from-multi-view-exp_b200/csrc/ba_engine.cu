// Engine object and the C ABI of include/ba_b200.h: memory layout in HBM, observation
// ingestion (camera-major index built on the device), phase sequencing of the LM loop.
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <new>
#include <chrono>
#include <mutex>
#include <thread>
#include <vector>

#include "ba_common.cuh"

namespace ba {

int64_t g_launch_count = 0;
static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int launch_lm_adopt(ba_engine* e, cudaStream_t s);

template <typename T>
static int dev_alloc(T** p, size_t n) {
  *p = nullptr;
  if (n == 0) n = 1;
  // stream-ordered allocation from the device's default pool; the pool keeps freed memory
  // (release threshold raised in create_engine), so engines created one after the other -- the
  // usual way the reference's class is used -- do not pay cudaMalloc/cudaFree again
  BA_CUDA(cudaMallocAsync(reinterpret_cast<void**>(p), n * sizeof(T), (cudaStream_t)0));
  return BA_OK;
}

static void dev_free(void* p) {
  if (p) cudaFreeAsync(p, (cudaStream_t)0);
}

static int retain_pool_memory(int device) {
  cudaMemPool_t pool;
  BA_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
  uint64_t keep = UINT64_MAX;
  BA_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
  return BA_OK;
}

// Pinned control blocks (4 ba_lm_state each) are recycled for the life of the process:
// cudaMallocHost / cudaFreeHost synchronise the device and take 15+ ms, which is more than a whole
// C2 adjustment, so an engine must not pay them.
static std::mutex g_pin_mutex;
static std::vector<ba_lm_state*> g_pin_free;

static ba_lm_state* pinned_block_acquire() {
  std::lock_guard<std::mutex> lock(g_pin_mutex);
  if (g_pin_free.empty()) {
    constexpr int kSlab = 8;
    ba_lm_state* slab = nullptr;
    if (cudaMallocHost(reinterpret_cast<void**>(&slab), kSlab * 4 * sizeof(ba_lm_state)) != cudaSuccess) return nullptr;
    for (int k = 0; k < kSlab; ++k) g_pin_free.push_back(slab + 4 * k);
  }
  ba_lm_state* p = g_pin_free.back();
  g_pin_free.pop_back();
  return p;
}

static void pinned_block_release(ba_lm_state* p) {
  if (!p) return;
  std::lock_guard<std::mutex> lock(g_pin_mutex);
  g_pin_free.push_back(p);
}

static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }
static inline int64_t round_up64(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

// Large uploads from PAGEABLE host memory (the reference's call hands over ordinary NumPy arrays: the
// dense observation block of C3 is 320 MB): cudaMemcpy stages them through the driver's own pinned
// buffer on one thread, ~6.5 GB/s measured here -- 50 ms of a 20-iteration C3 call.  staged_upload
// does the staging with kUpThreads host threads, each copying its chunks into its own pinned buffers
// (kept for the life of the process) and sending them on its own stream while it copies the next;
// the caller's stream waits for all of them.  Pinned or small sources take the plain path.
constexpr int kUpThreads = 8, kUpBufs = 2;
constexpr size_t kUpChunk = (size_t)1 << 20, kUpMin = (size_t)64 << 20;  // 16 MB pinned in all (page-locking costs ~3 ms per MB, once per process)
struct UploadPool {
  int device = -1;
  void* buf[kUpThreads][kUpBufs] = {};
  cudaEvent_t ev[kUpThreads][kUpBufs] = {};
  cudaEvent_t done[kUpThreads] = {}, start = nullptr;
  cudaStream_t st[kUpThreads] = {};
};
static std::mutex g_up_mutex;
static UploadPool g_up;

static bool upload_pool_ready(int device) {
  if (g_up.device == device) return true;
  if (g_up.device >= 0) return false;  // one device per process uses the pool; others take the plain path
  // ONE pinned slab (cudaMallocHost synchronises the device and costs tens of milliseconds per call)
  char* slab = nullptr;
  if (cudaMallocHost(reinterpret_cast<void**>(&slab), (size_t)kUpThreads * kUpBufs * kUpChunk) != cudaSuccess) return false;
  for (int t = 0; t < kUpThreads; ++t) {
    if (cudaStreamCreateWithFlags(&g_up.st[t], cudaStreamNonBlocking) != cudaSuccess) return false;
    if (cudaEventCreateWithFlags(&g_up.done[t], cudaEventDisableTiming) != cudaSuccess) return false;
    for (int b = 0; b < kUpBufs; ++b) {
      g_up.buf[t][b] = slab + ((size_t)t * kUpBufs + b) * kUpChunk;
      if (cudaEventCreateWithFlags(&g_up.ev[t][b], cudaEventDisableTiming) != cudaSuccess) return false;
    }
  }
  if (cudaEventCreateWithFlags(&g_up.start, cudaEventDisableTiming) != cudaSuccess) return false;
  g_up.device = device;
  return true;
}

static bool staged_upload(void* dst, const void* src, size_t bytes, cudaStream_t s) {
  if (bytes < kUpMin) return false;
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, src) != cudaSuccess) { cudaGetLastError(); return false; }
  if (attr.type != cudaMemoryTypeUnregistered) return false;  // pinned / managed: the DMA engine reads it directly
  int device = 0;
  if (cudaGetDevice(&device) != cudaSuccess) return false;
  std::lock_guard<std::mutex> lock(g_up_mutex);
  if (!upload_pool_ready(device)) { cudaGetLastError(); return false; }
  // the copies must not overtake what the caller's stream still does with dst
  if (cudaEventRecord(g_up.start, s) != cudaSuccess) return false;
  const size_t n_chunks = (bytes + kUpChunk - 1) / kUpChunk;
  bool failed[kUpThreads] = {};
  // the ranks of a multi-GPU job on one node share the host cores (torchrun exports LOCAL_WORLD_SIZE)
  int n_threads = kUpThreads;
  {
    const char* lws = std::getenv("LOCAL_WORLD_SIZE");
    const int ranks = lws ? std::max(1, std::atoi(lws)) : 1;
    const int cores = (int)std::thread::hardware_concurrency();
    if (cores > 0) n_threads = std::min(kUpThreads, std::max(1, cores / (2 * ranks)));
  }
  if (n_threads < 2) return false;
  std::vector<std::thread> workers;
  for (int t = 0; t < n_threads; ++t)
    workers.emplace_back([&, t]() {
      if (cudaSetDevice(device) != cudaSuccess || cudaStreamWaitEvent(g_up.st[t], g_up.start, 0) != cudaSuccess) {
        failed[t] = true;
        return;
      }
      int round = 0;
      for (size_t c = (size_t)t; c < n_chunks; c += (size_t)n_threads, ++round) {
        const int b = round % kUpBufs;
        const size_t off_b = c * kUpChunk, len = bytes - off_b < kUpChunk ? bytes - off_b : kUpChunk;
        if (round >= kUpBufs && cudaEventSynchronize(g_up.ev[t][b]) != cudaSuccess) { failed[t] = true; return; }
        std::memcpy(g_up.buf[t][b], static_cast<const char*>(src) + off_b, len);
        if (cudaMemcpyAsync(static_cast<char*>(dst) + off_b, g_up.buf[t][b], len, cudaMemcpyHostToDevice, g_up.st[t]) != cudaSuccess ||
            cudaEventRecord(g_up.ev[t][b], g_up.st[t]) != cudaSuccess) {
          failed[t] = true;
          return;
        }
      }
      if (cudaEventRecord(g_up.done[t], g_up.st[t]) != cudaSuccess) failed[t] = true;
    });
  for (auto& w : workers) w.join();
  bool ok = true;
  for (int t = 0; t < n_threads; ++t) {
    // the staging buffers are reused by the next call: their transfers must have left them
    if (failed[t] || cudaStreamWaitEvent(s, g_up.done[t], 0) != cudaSuccess || cudaEventSynchronize(g_up.done[t]) != cudaSuccess)
      ok = false;
  }
  if (!ok) cudaGetLastError();
  return ok;
}

static int copy_in(void* dst, const void* src, size_t bytes, int mem, cudaStream_t s) {
  if (bytes == 0) return BA_OK;
  if (mem == BA_MEM_HOST && staged_upload(dst, src, bytes, s)) return BA_OK;
  BA_CUDA(cudaMemcpyAsync(dst, src, bytes,
                          mem == BA_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
  return BA_OK;
}
static int copy_out(void* dst, const void* src, size_t bytes, int mem, cudaStream_t s) {
  if (bytes == 0) return BA_OK;
  BA_CUDA(cudaMemcpyAsync(dst, src, bytes,
                          mem == BA_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
  return BA_OK;
}

// ---- observation index kernels ---------------------------------------------------------------
__global__ void fill_obs_pt_kernel(int64_t N, const int64_t* __restrict__ obs_ptr,
                                   int32_t* __restrict__ obs_pt) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t j = warp; j < N; j += nwarps)
    for (int64_t o = obs_ptr[j] + lane; o < obs_ptr[j + 1]; o += 32) obs_pt[o] = (int32_t)j;
}

__global__ void iota_kernel(int64_t n, int32_t* __restrict__ v) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) v[k] = (int32_t)k;
}

// cam_ptr[i] = first position in the camera-sorted key array with key >= i
__global__ void cam_ptr_kernel(int M, int64_t n, const int32_t* __restrict__ keys,
                               int64_t* __restrict__ cam_ptr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > M) return;
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (keys[mid] < i) lo = mid + 1; else hi = mid;
  }
  cam_ptr[i] = lo;
}

// obs_ptr of a dense scene: point j owns observations [j M, (j + 1) M)
__global__ void dense_ptr_kernel(int64_t N, int M, int64_t* __restrict__ obs_ptr) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j <= N; j += stride) obs_ptr[j] = j * M;
}

// Camera-major image points src[M][N] (one double2 each) -> point-major dst[N][M]: 32 x 32 tiles
// through shared memory, both sides coalesced.  grid = (ceil(N/32), ceil(M/32)), block = (32, 8).
__global__ void transpose_xy_kernel(int64_t N, int M, const double2* __restrict__ src,
                                    double2* __restrict__ dst) {
  __shared__ double2 tile[32][33];
  const int64_t j0 = (int64_t)blockIdx.x * 32;
  const int i0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int i = i0 + r;
    const int64_t j = j0 + threadIdx.x;
    if (i < M && j < N) tile[r][threadIdx.x] = src[(int64_t)i * N + j];
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int64_t j = j0 + r;
    const int i = i0 + threadIdx.x;
    if (i < M && j < N) dst[j * M + i] = tile[threadIdx.x][r];
  }
}

// Stable (hence deterministic) radix sort of observation ids by camera: cm_perm, cam_ptr.
int build_camera_major_index(ba_engine* e, cudaStream_t s) {
  const int64_t n = e->nobs;
  if (n >= (int64_t)1 << 31) {
    set_error("more than 2^31 observations per engine are not supported");
    return BA_ERR_INVALID;
  }
  int32_t *keys_out = nullptr, *vals_in = nullptr;
  BA_TRY(dev_alloc(&keys_out, (size_t)n));
  BA_TRY(dev_alloc(&vals_in, (size_t)n));
  iota_kernel<<<e->num_sms * 4, 256, 0, s>>>(n, vals_in);
  BA_LAUNCH_CHECK();
  int bits = 1;
  while ((1 << bits) < e->M) ++bits;
  size_t tmp_bytes = 0;
  BA_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, e->obs_cam, keys_out, vals_in,
                                          e->cm_perm, (int)n, 0, bits, s));
  void* tmp = nullptr;
  BA_CUDA(cudaMallocAsync(&tmp, tmp_bytes ? tmp_bytes : 1, (cudaStream_t)0));
  BA_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, e->obs_cam, keys_out, vals_in, e->cm_perm,
                                          (int)n, 0, bits, s));
  cam_ptr_kernel<<<(e->M + 1 + 127) / 128, 128, 0, s>>>(e->M, n, keys_out, e->cam_ptr);
  BA_LAUNCH_CHECK();
  BA_CUDA(cudaStreamSynchronize(s));
  dev_free(tmp);
  dev_free(keys_out);
  dev_free(vals_in);
  return BA_OK;
}

static void free_engine(ba_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  if (e->own_stream) cudaStreamSynchronize(e->own_stream);
  prof_resolve(e, false);
  comm_free(e);  // closes the peers' windows and frees this rank's (which holds red)
  void* ptrs[] = {e->obs_ptr, e->obs_cam, e->obs_pt, e->obs_xy, e->cam_ptr, e->cm_perm, e->X[0],
                  e->X[1], e->cam[0].f, e->cam[1].f, e->camtab[0], e->camtab[1], e->JP, e->JC, e->V,
                  e->GPT, e->Upart, e->Uloc, e->LINV, e->Z, e->Yt, e->Ysp, e->red_in_window ? nullptr : e->red, e->Lt, e->Winv,
                  e->dxi, e->cost_part, e->cost_buf, e->ctl, e->rec, e->ywork, e->chol_bar, e->gauge};
  for (void* p : ptrs)
    dev_free(p);
  syrk_release(&e->syrk, (cudaStream_t)0);
  pairs_release(&e->pairs, (cudaStream_t)0);
  for (int k = 0; k < 2; ++k) {
    if (e->solve_graph[k]) cudaGraphExecDestroy(e->solve_graph[k]);
    if (e->solve_ev[k]) cudaEventDestroy(e->solve_ev[k]);
  }
  if (e->own_stream) {
    cudaStreamSynchronize(e->own_stream);  // nothing may still be copying into the pinned block
    cudaStreamDestroy(e->own_stream);
  }
  pinned_block_release(e->ctl_host);
  if (e->ev0) cudaEventDestroy(e->ev0);
  if (e->ev1) cudaEventDestroy(e->ev1);
  delete e;
}

static int alloc_cam(CamState* c, int M) {
  double* base = nullptr;
  BA_TRY(dev_alloc(&base, (size_t)15 * M));
  c->f = base;
  c->u = base + M;
  c->R = base + 3 * (size_t)M;
  c->t = base + 12 * (size_t)M;
  return BA_OK;
}

struct StepTimer {
  bool on = std::getenv("BA_TIMING") != nullptr;
  std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
  void lap(const char* what) {
    if (!on) return;
    const auto n = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[ba timing] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(n - t).count());
    t = n;
  }
};

static int create_engine(const ba_problem* p, ba_engine** out) {
  StepTimer tm;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_error("no CUDA device: this engine has no CPU path");
    return BA_ERR_NO_DEVICE;
  }
  if (!p || !out) { set_error("null argument"); return BA_ERR_INVALID; }
  if (p->axis != BA_AXIS_X_RIGHT && p->axis != BA_AXIS_X_UP) {
    set_error("unknown gauge axis %d", p->axis);
    return BA_ERR_INVALID;
  }
  if (p->n_cams < 2 || p->n_points < 1 || p->n_obs < 1 || !(p->f0 != 0.0)) {
    set_error("need >= 2 cameras, >= 1 point, >= 1 observation and f0 != 0");
    return BA_ERR_INVALID;
  }
  if (p->dense && p->n_obs != p->n_points * (int64_t)p->n_cams) {
    set_error("dense problem needs n_obs == n_points * n_cams");
    return BA_ERR_INVALID;
  }
  if (p->device < 0 || p->device >= ndev) {
    set_error("device %d out of range (%d devices)", p->device, ndev);
    return BA_ERR_INVALID;
  }
  BA_CUDA(cudaSetDevice(p->device));
  BA_TRY(require_tensor_map_encoder());
  tm.lap("device count / set device");
  BA_TRY(retain_pool_memory(p->device));
  tm.lap("pool attribute");
  ba_engine* e = new (std::nothrow) ba_engine();
  if (!e) { set_error("out of host memory"); return BA_ERR_CUDA; }
  e->prob = *p;
  e->N = p->n_points; e->nobs = p->n_obs; e->M = p->n_cams; e->dense = p->dense ? 1 : 0;
  e->axis = p->axis; e->device = p->device; e->f0 = p->f0;
  BA_CUDA(cudaDeviceGetAttribute(&e->num_sms, cudaDevAttrMultiProcessorCount, p->device));
  tm.lap("device attribute");

  e->n_full = 9 * e->M;
  e->rhs_row = e->n_full;
  const int n_aug = e->n_full + 1;
  e->n_pad = round_up(n_aug, 8);  // fragment granularity; edge tiles of the SYRK are partial
  e->k_pad = round_up64(3 * e->N, 32);
  // camera_blocks_kernel: 3 blocks per SM (162 registers); ~8 waves of blocks so that the last,
  // partly filled wave costs little (ncu, C3: 600 blocks = 1.35 waves ran at 55 % of HBM bandwidth)
  e->cam_chunks = (8 * 3 * e->num_sms + e->M - 1) / e->M;
  if (e->cam_chunks < 1) e->cam_chunks = 1;
  {
    const int64_t per_cam = e->nobs / e->M + 1;
    const int64_t maxc = per_cam / 1024 > 0 ? per_cam / 1024 : 1;  // >= 8 observations per thread
    if (e->cam_chunks > maxc) e->cam_chunks = (int)maxc;
  }
  {
    const int64_t b = (e->nobs + 255) / 256;
    const int64_t cap = (int64_t)e->num_sms * 4;
    e->cost_blocks = (int)(b < cap ? b : cap);
  }

  int st = BA_OK;
#define A(expr) if (st == BA_OK) st = (expr)
  // first: a camera count past the pair kernels' launch limit is refused before anything is allocated
  if (!e->dense) A(pairs_prepare(&e->pairs, e->M, e->N, (cudaStream_t)0));
  A(dev_alloc(&e->obs_ptr, (size_t)e->N + 1));
  A(dev_alloc(&e->obs_xy, (size_t)e->nobs * 2));
  if (!e->dense) {
    A(dev_alloc(&e->obs_cam, (size_t)e->nobs));
    A(dev_alloc(&e->obs_pt, (size_t)e->nobs));
    A(dev_alloc(&e->cm_perm, (size_t)e->nobs));
    A(dev_alloc(&e->cam_ptr, (size_t)e->M + 1));
  }
  for (int w = 0; w < 2; ++w) {
    A(dev_alloc(&e->X[w], (size_t)3 * e->N));
    A(alloc_cam(&e->cam[w], e->M));
    A(dev_alloc(&e->camtab[w], (size_t)e->M * kCamTab));
  }
  A(dev_alloc(&e->gauge, (size_t)16));
  A(dev_alloc(&e->JP, (size_t)e->nobs * kJP));
  A(dev_alloc(&e->JC, (size_t)e->nobs * kJC));
  A(dev_alloc(&e->V, (size_t)6 * e->N));
  A(dev_alloc(&e->GPT, (size_t)3 * e->N));
  A(dev_alloc(&e->Upart, (size_t)e->M * e->cam_chunks * kUPart));
  A(dev_alloc(&e->Uloc, (size_t)e->M * 90));
  A(dev_alloc(&e->LINV, (size_t)6 * e->N));
  A(dev_alloc(&e->Z, (size_t)3 * e->N));
  e->red_len = (int64_t)e->n_pad * e->n_pad + (int64_t)e->M * 90;
  A(dev_alloc(&e->red, (size_t)e->red_len));
  if (e->dense) {
    A(dev_alloc(&e->Yt, (size_t)e->k_pad * e->n_pad));
    A(syrk_prepare(&e->syrk, SYRK_AUTO, e->n_pad, e->k_pad, e->num_sms, (cudaStream_t)0));
  } else {
    A(dev_alloc(&e->Ysp, (size_t)e->nobs * 27));
  }
  A(dev_alloc(&e->Lt, (size_t)kCholOB * e->n_pad));
  A(dev_alloc(&e->ywork, (size_t)e->n_pad));
  A(dev_alloc(&e->chol_bar, (size_t)4));
  A(dev_alloc(&e->Winv, (size_t)((e->n_full + kCholNB - 1) / kCholNB) * kCholNB * kCholNB));
  A(dev_alloc(&e->dxi, (size_t)e->n_full));
  A(dev_alloc(&e->cost_part, (size_t)e->num_sms * 16 + 1024));
  A(dev_alloc(&e->cost_buf, (size_t)4));
  A(dev_alloc(&e->ctl, (size_t)1));
  A(dev_alloc(&e->rec, (size_t)kMaxRecords));
#undef A
  tm.lap("device allocations");
  if (st == BA_OK && !(e->ctl_host = pinned_block_acquire())) {
    set_error("cudaMallocHost failed");
    st = BA_ERR_CUDA;
  }
  tm.lap("pinned control block");
  if (st == BA_OK) {
    cudaEventCreate(&e->ev0);
    cudaEventCreate(&e->ev1);
    cudaMemset(e->red, 0, (size_t)e->red_len * sizeof(double));
    if (e->Yt) cudaMemset(e->Yt, 0, (size_t)e->k_pad * e->n_pad * sizeof(double));
    cudaMemset(e->ctl, 0, sizeof(ba_lm_state));
    cudaMemset(e->cost_buf, 0, 4 * sizeof(double));
    cudaMemset(e->dxi, 0, (size_t)e->n_full * sizeof(double));
    if (cudaDeviceSynchronize() != cudaSuccess) {
      set_error("device initialisation failed: %s", cudaGetErrorString(cudaGetLastError()));
      st = BA_ERR_CUDA;
    }
  }
  tm.lap("events, memsets, sync");
  if (st != BA_OK) {
    free_engine(e);
    return st;
  }
  *out = e;
  return BA_OK;
}

static int check_ready(ba_engine* e) {
  if (!e) { set_error("null engine"); return BA_ERR_INVALID; }
  if (!e->have_obs || !e->have_state) {
    set_error("observations and state must be set first");
    return BA_ERR_STATE;
  }
  if (cudaSetDevice(e->device) != cudaSuccess) { set_error("cudaSetDevice failed"); return BA_ERR_CUDA; }
  return BA_OK;
}

static int phase_reduce(ba_engine* e, bool conditional, double c_host, cudaStream_t s) {
  if (conditional) {
    BA_TRY(launch_lm_adopt(e, s));
    { ProfScope ps(e, PG_K1, s); BA_TRY(launch_k1(e, s, true)); }
    { ProfScope ps(e, PG_K2, s); BA_TRY(launch_k2a(e, s, true)); BA_TRY(launch_camera_blocks(e, s, true)); }
  }
  { ProfScope ps(e, PG_K2, s); BA_TRY(launch_k2b(e, conditional, c_host, s)); }
  { ProfScope ps(e, PG_K3, s); BA_TRY(launch_k3(e, conditional, s)); }
  if (e->comm) BA_TRY(launch_comm_allreduce_red(e, conditional, s));
  return BA_OK;
}

static int phase_solve(ba_engine* e, bool conditional, double c_host, cudaStream_t s) {
  ProfScope ps(e, PG_K4, s);
  BA_TRY(launch_assemble(e, conditional, c_host, s));
  { ProfScope pc(e, PG_CHOL, s); BA_TRY(launch_cholesky_solve(e, conditional, s)); }
  BA_TRY(launch_update_trial(e, conditional, s));
  if (e->comm) BA_TRY(launch_comm_allreduce_cost(e, 1, conditional, s));
  return BA_OK;
}

static int read_ctl(ba_engine* e, ba_lm_state* out, cudaStream_t s) {
  BA_CUDA(cudaMemcpyAsync(e->ctl_host, e->ctl, sizeof(ba_lm_state), cudaMemcpyDeviceToHost, s));
  BA_CUDA(cudaStreamSynchronize(s));
  if (out) *out = *e->ctl_host;
  return BA_OK;
}

static int status_from_ctl(const ba_lm_state& st) {
  if (st.status == BA_ERR_SINGULAR) {
    set_error("Singular matrix");  // numpy.linalg.LinAlgError text of the reference (:128)
    return BA_ERR_SINGULAR;
  }
  if (st.status == BA_ERR_COMM) {
    set_error("a peer rank did not answer within the spin limit of the NVLink exchange");
    return BA_ERR_COMM;
  }
  if (st.status == BA_ERR_BARRIER) {
    set_error("grid barrier of the back substitution timed out: its blocks were not co-resident "
              "(is another kernel holding the GPU?)");
    return BA_ERR_BARRIER;
  }
  if (st.status == BA_ERR_STALL) {
    set_error("inner LM loop exceeded %d retries without decreasing the cost", st.max_retries);
    return BA_ERR_STALL;
  }
  return BA_OK;
}

}  // namespace ba

using namespace ba;

extern "C" {

int ba_version(void) { return BA_B200_VERSION; }
const char* ba_last_error(void) { return g_err; }

int ba_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int ba_create(const ba_problem* problem, ba_engine** out) { return create_engine(problem, out); }

int ba_destroy(ba_engine* e) {
  free_engine(e);
  return BA_OK;
}

int ba_set_observations(ba_engine* e, const int64_t* obs_ptr, const int32_t* obs_cam,
                        const double* obs_xy, int mem, void* stream) {
  if (!e || !obs_xy || (!e->dense && (!obs_ptr || !obs_cam))) {
    set_error("null argument");
    return BA_ERR_INVALID;
  }
  cudaStream_t s = (cudaStream_t)stream;
  BA_CUDA(cudaSetDevice(e->device));
  if (mem == BA_MEM_HOST && obs_ptr) {
    if (obs_ptr[0] != 0 || obs_ptr[e->N] != e->nobs) {
      set_error("obs_ptr must start at 0 and end at n_obs");
      return BA_ERR_INVALID;
    }
    for (int64_t j = 0; j < e->N; ++j)
      if (obs_ptr[j + 1] < obs_ptr[j]) { set_error("obs_ptr not monotone"); return BA_ERR_INVALID; }
    if (!e->dense)
      for (int64_t o = 0; o < e->nobs; ++o)
        if (obs_cam[o] < 0 || obs_cam[o] >= e->M) { set_error("camera index out of range"); return BA_ERR_INVALID; }
  }
  if (obs_ptr) {
    BA_TRY(copy_in(e->obs_ptr, obs_ptr, ((size_t)e->N + 1) * sizeof(int64_t), mem, s));
  } else {
    std::vector<int64_t> p((size_t)e->N + 1);
    for (int64_t j = 0; j <= e->N; ++j) p[(size_t)j] = j * e->M;
    BA_CUDA(cudaMemcpyAsync(e->obs_ptr, p.data(), p.size() * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    BA_CUDA(cudaStreamSynchronize(s));
  }
  BA_TRY(copy_in(e->obs_xy, obs_xy, (size_t)e->nobs * 2 * sizeof(double), mem, s));
  if (!e->dense) {
    BA_TRY(copy_in(e->obs_cam, obs_cam, (size_t)e->nobs * sizeof(int32_t), mem, s));
    fill_obs_pt_kernel<<<e->num_sms * 8, 256, 0, s>>>(e->N, e->obs_ptr, e->obs_pt);
    BA_LAUNCH_CHECK();
    BA_TRY(build_camera_major_index(e, s));
    // captured solves launch the pair kernel of the previous index, on lists pairs_index frees:
    // ba_lm_run captures them again
    for (int k = 0; k < 2; ++k)
      if (e->solve_graph[k]) {
        BA_CUDA(cudaGraphExecDestroy(e->solve_graph[k]));
        e->solve_graph[k] = nullptr;
      }
    BA_TRY(pairs_index(&e->pairs, e->nobs, e->obs_cam, e->obs_pt, e->num_sms, s));
  }
  BA_CUDA(cudaStreamSynchronize(s));
  e->have_obs = true;
  return BA_OK;
}

int ba_set_observations_dense(ba_engine* e, const double* x, int64_t stride_pt, int64_t stride_cam,
                              int mem, void* stream) {
  if (!e || !x) { set_error("null argument"); return BA_ERR_INVALID; }
  if (!e->dense) { set_error("ba_set_observations_dense needs a dense problem"); return BA_ERR_INVALID; }
  cudaStream_t s = (cudaStream_t)stream;
  BA_CUDA(cudaSetDevice(e->device));
  const int64_t N = e->N;
  const int M = e->M;
  const size_t bytes = (size_t)e->nobs * 2 * sizeof(double);
  if (stride_pt == 2 * (int64_t)M && stride_cam == 2) {
    BA_TRY(copy_in(e->obs_xy, x, bytes, mem, s));  // already point-major
  } else if (stride_pt == 2 && stride_cam == 2 * N) {
    // camera-major block (np.stack(x_list).transpose(1, 0, 2)): copy it as it lies in memory into the
    // camera-side Jacobian buffer (20 doubles per observation, not in use before the first
    // linearisation) and re-order on the device
    BA_TRY(copy_in(e->JC, x, bytes, mem, s));
    const dim3 grid((unsigned)((N + 31) / 32), (unsigned)((M + 31) / 32));
    transpose_xy_kernel<<<grid, dim3(32, 8), 0, s>>>(N, M, reinterpret_cast<const double2*>(e->JC),
                                                     reinterpret_cast<double2*>(e->obs_xy));
    BA_LAUNCH_CHECK();
  } else {
    set_error("dense observations must be one point-major or camera-major block (strides %lld, %lld)",
              (long long)stride_pt, (long long)stride_cam);
    return BA_ERR_INVALID;
  }
  dense_ptr_kernel<<<e->num_sms, 256, 0, s>>>(N, M, e->obs_ptr);
  BA_LAUNCH_CHECK();
  BA_CUDA(cudaStreamSynchronize(s));
  e->have_obs = true;
  return BA_OK;
}

int ba_set_state(ba_engine* e, const double* X, const double* R, const double* t, const double* f,
                 const double* u, int mem, void* stream) {
  if (!e) { set_error("null engine"); return BA_ERR_INVALID; }
  cudaStream_t s = (cudaStream_t)stream;
  BA_CUDA(cudaSetDevice(e->device));
  const size_t d = sizeof(double);
  if (X) BA_TRY(copy_in(e->X[0], X, (size_t)3 * e->N * d, mem, s));
  if (R) BA_TRY(copy_in(e->cam[0].R, R, (size_t)9 * e->M * d, mem, s));
  if (t) BA_TRY(copy_in(e->cam[0].t, t, (size_t)3 * e->M * d, mem, s));
  if (f) BA_TRY(copy_in(e->cam[0].f, f, (size_t)e->M * d, mem, s));
  if (u) BA_TRY(copy_in(e->cam[0].u, u, (size_t)2 * e->M * d, mem, s));
  if (mem == BA_MEM_HOST) BA_CUDA(cudaStreamSynchronize(s));
  e->have_state = true;
  return BA_OK;
}

int ba_get_state(ba_engine* e, int which, double* X, double* R, double* t, double* f, double* u,
                 int mem, void* stream) {
  if (!e || (which != 0 && which != 1)) { set_error("bad argument"); return BA_ERR_INVALID; }
  cudaStream_t s = (cudaStream_t)stream;
  BA_CUDA(cudaSetDevice(e->device));
  const size_t d = sizeof(double);
  if (X) BA_TRY(copy_out(X, e->X[which], (size_t)3 * e->N * d, mem, s));
  if (R) BA_TRY(copy_out(R, e->cam[which].R, (size_t)9 * e->M * d, mem, s));
  if (t) BA_TRY(copy_out(t, e->cam[which].t, (size_t)3 * e->M * d, mem, s));
  if (f) BA_TRY(copy_out(f, e->cam[which].f, (size_t)e->M * d, mem, s));
  if (u) BA_TRY(copy_out(u, e->cam[which].u, (size_t)2 * e->M * d, mem, s));
  if (mem == BA_MEM_HOST) BA_CUDA(cudaStreamSynchronize(s));
  return BA_OK;
}

int ba_cost(ba_engine* e, int which, void* stream) {
  BA_TRY(check_ready(e));
  if (which != 0 && which != 1) { set_error("bad state selector"); return BA_ERR_INVALID; }
  cudaStream_t s = (cudaStream_t)stream;
  ProfScope ps(e, PG_COST, s);
  BA_TRY(launch_cam_prep(e, which, s));
  return launch_cost(e, which, which, s);
}

int ba_linearize(ba_engine* e, void* stream) {
  BA_TRY(check_ready(e));
  cudaStream_t s = (cudaStream_t)stream;
  { ProfScope ps(e, PG_K1, s); BA_TRY(launch_k1(e, s, false)); }
  { ProfScope ps(e, PG_K2, s); BA_TRY(launch_k2a(e, s, false)); BA_TRY(launch_camera_blocks(e, s, false)); }
  return BA_OK;
}

int ba_build_reduced(ba_engine* e, double c, void* stream) {
  BA_TRY(check_ready(e));
  return phase_reduce(e, false, c, (cudaStream_t)stream);
}

int ba_solve_trial(ba_engine* e, double c, void* stream) {
  BA_TRY(check_ready(e));
  return phase_solve(e, false, c, (cudaStream_t)stream);
}

int ba_lm_begin(ba_engine* e, double scale_factor, double delta_tol, int max_iter, int max_retries,
                void* stream) {
  BA_TRY(check_ready(e));
  cudaStream_t s = (cudaStream_t)stream;
  if (max_retries <= 0) max_retries = 200;
  BA_TRY(launch_lm_begin(e, scale_factor, delta_tol, max_iter, max_retries, s));
  {
    ProfScope ps(e, PG_COST, s);
    BA_TRY(launch_cam_prep(e, 0, s));
    BA_TRY(launch_cost(e, 0, 0, s));
  }
  if (e->comm) BA_TRY(launch_comm_allreduce_cost(e, 0, true, s));
  return BA_OK;
}

int ba_lm_phase_reduce(ba_engine* e, void* stream) {
  BA_TRY(check_ready(e));
  return phase_reduce(e, true, 0.0, (cudaStream_t)stream);
}

int ba_lm_phase_solve(ba_engine* e, void* stream) {
  BA_TRY(check_ready(e));
  return phase_solve(e, true, 0.0, (cudaStream_t)stream);
}

int ba_lm_phase_decide(ba_engine* e, void* stream) {
  BA_TRY(check_ready(e));
  cudaStream_t s = (cudaStream_t)stream;
  ProfScope ps(e, PG_OTHER, s);
  return launch_decide(e, s);
}

int ba_lm_state_get(ba_engine* e, ba_lm_state* out, void* stream) {
  if (!e || !out) { set_error("null argument"); return BA_ERR_INVALID; }
  BA_CUDA(cudaSetDevice(e->device));
  return read_ctl(e, out, (cudaStream_t)stream);
}

int ba_lm_state_post(ba_engine* e, int slot, void* stream) {
  if (!e || (slot != 0 && slot != 1)) { set_error("bad argument"); return BA_ERR_INVALID; }
  cudaStream_t s = (cudaStream_t)stream;
  BA_CUDA(cudaSetDevice(e->device));
  if (!e->solve_ev[slot]) BA_CUDA(cudaEventCreateWithFlags(&e->solve_ev[slot], cudaEventDisableTiming));
  BA_CUDA(cudaMemcpyAsync(e->ctl_host + 1 + slot, e->ctl, sizeof(ba_lm_state), cudaMemcpyDeviceToHost, s));
  BA_CUDA(cudaEventRecord(e->solve_ev[slot], s));
  return BA_OK;
}

int ba_lm_state_wait(ba_engine* e, int slot, ba_lm_state* out) {
  if (!e || !out || (slot != 0 && slot != 1) || !e->solve_ev[slot]) { set_error("bad argument"); return BA_ERR_INVALID; }
  BA_CUDA(cudaEventSynchronize(e->solve_ev[slot]));
  *out = e->ctl_host[1 + slot];
  return BA_OK;
}

int ba_lm_iterate(ba_engine* e, ba_lm_state* out, void* stream) {
  BA_TRY(check_ready(e));
  cudaStream_t s = (cudaStream_t)stream;
  ba_lm_state st;
  BA_TRY(read_ctl(e, &st, s));
  const int count0 = st.count;
  while (!st.done && st.count == count0) {
    BA_TRY(phase_reduce(e, true, 0.0, s));
    BA_TRY(phase_solve(e, true, 0.0, s));
    { ProfScope ps(e, PG_OTHER, s); BA_TRY(launch_decide(e, s)); }
    BA_TRY(read_ctl(e, &st, s));
  }
  if (out) *out = st;
  return status_from_ctl(st);
}

int ba_lm_records(ba_engine* e, ba_iter_record* records, int max_records, int* n_records,
                  void* stream) {
  if (!e || !n_records) { set_error("null argument"); return BA_ERR_INVALID; }
  cudaStream_t s = (cudaStream_t)stream;
  ba_lm_state st;
  BA_TRY(read_ctl(e, &st, s));
  int n = st.count < kMaxRecords ? st.count : kMaxRecords;
  if (n > max_records) n = max_records;
  if (n > 0 && records) {
    BA_CUDA(cudaMemcpyAsync(records, e->rec, (size_t)n * sizeof(ba_iter_record), cudaMemcpyDeviceToHost, s));
    BA_CUDA(cudaStreamSynchronize(s));
  }
  *n_records = n;
  return BA_OK;
}

// One inner solve (linearise if needed, reduce, factor, solve, trial, decide) captured as a CUDA
// graph.  Every kernel of the sequence takes its decisions from the device-resident control
// block, so the same graph serves every solve; it ends with the copy of the control block into
// pinned slot `slot`.
static int capture_solve_graph(ba_engine* e, int slot) {
  cudaStream_t s = e->own_stream;
  const int64_t before = g_launch_count;
  cudaGraph_t graph = nullptr;
  BA_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  int st = phase_reduce(e, true, 0.0, s);
  if (st == BA_OK) st = phase_solve(e, true, 0.0, s);
  if (st == BA_OK) st = launch_decide(e, s);
  if (st == BA_OK &&
      cudaMemcpyAsync(e->ctl_host + 1 + slot, e->ctl, sizeof(ba_lm_state), cudaMemcpyDeviceToHost, s) != cudaSuccess)
    st = BA_ERR_CUDA;
  const cudaError_t ce = cudaStreamEndCapture(s, &graph);
  e->graph_launches = g_launch_count - before;
  g_launch_count = before;  // nothing ran yet; every graph launch adds graph_launches
  if (st != BA_OK || ce != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    if (st == BA_OK) set_error("graph capture failed: %s", cudaGetErrorString(ce));
    cudaGetLastError();
    return st != BA_OK ? st : BA_ERR_CUDA;
  }
  const cudaError_t ie = cudaGraphInstantiate(&e->solve_graph[slot], graph, 0);
  cudaGraphDestroy(graph);
  if (ie != cudaSuccess) {
    set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(ie));
    return BA_ERR_CUDA;
  }
  if (!e->solve_ev[slot]) BA_CUDA(cudaEventCreateWithFlags(&e->solve_ev[slot], cudaEventDisableTiming));
  return BA_OK;
}

// The whole LM loop.  Without profiling the solves run as CUDA graphs on the engine's own stream,
// one solve ahead of the host: graph n+1 is launched before the control block of solve n is read,
// so the device never waits for the host (after termination the extra graph is a chain of
// early-exit kernels).  With profiling on (per-phase event timing) the launches stay eager.
int ba_lm_run(ba_engine* e, double scale_factor, double delta_tol, int max_iter, int max_retries,
              ba_iter_record* records, int max_records, int* n_records, ba_lm_state* final_state,
              void* stream) {
  BA_TRY(check_ready(e));
  cudaStream_t user = (cudaStream_t)stream;
  ba_lm_state st;
  std::memset(&st, 0, sizeof(st));
  if (e->profiling || std::getenv("BA_NO_GRAPH")) {
    BA_TRY(ba_lm_begin(e, scale_factor, delta_tol, max_iter, max_retries, stream));
    while (!st.done) {
      BA_TRY(phase_reduce(e, true, 0.0, user));
      BA_TRY(phase_solve(e, true, 0.0, user));
      { ProfScope ps(e, PG_OTHER, user); BA_TRY(launch_decide(e, user)); }
      BA_TRY(read_ctl(e, &st, user));
    }
  } else {
    if (!e->own_stream) BA_CUDA(cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
    cudaStream_t s = e->own_stream;
    // order after whatever the caller queued on its stream
    BA_CUDA(cudaEventRecord(e->ev0, user));
    BA_CUDA(cudaStreamWaitEvent(s, e->ev0, 0));
    BA_TRY(ba_lm_begin(e, scale_factor, delta_tol, max_iter, max_retries, s));
    for (int k = 0; k < 2; ++k)
      if (!e->solve_graph[k]) BA_TRY(capture_solve_graph(e, k));
    int n = 0;  // graphs launched
    BA_CUDA(cudaGraphLaunch(e->solve_graph[0], s));
    BA_CUDA(cudaEventRecord(e->solve_ev[0], s));
    g_launch_count += e->graph_launches;
    n = 1;
    while (true) {
      // speculative: the next solve is queued before this one's decision is known
      const int nxt = n & 1;
      BA_CUDA(cudaGraphLaunch(e->solve_graph[nxt], s));
      BA_CUDA(cudaEventRecord(e->solve_ev[nxt], s));
      g_launch_count += e->graph_launches;
      ++n;
      BA_CUDA(cudaEventSynchronize(e->solve_ev[nxt ^ 1]));
      st = e->ctl_host[1 + (nxt ^ 1)];
      if (st.done) break;
    }
    BA_CUDA(cudaStreamSynchronize(s));  // the speculative tail (no-ops) must not outlive the call
  }
  if (final_state) *final_state = st;
  if (n_records) BA_TRY(ba_lm_records(e, records, max_records, n_records, stream));
  return status_from_ctl(st);
}

int ba_reduce_buffer(ba_engine* e, void** device_ptr, int64_t* n_doubles) {
  if (!e || !device_ptr || !n_doubles) { set_error("null argument"); return BA_ERR_INVALID; }
  *device_ptr = e->red;
  *n_doubles = e->red_len;
  return BA_OK;
}

int ba_cost_buffer(ba_engine* e, void** device_ptr, int64_t* n_doubles) {
  if (!e || !device_ptr || !n_doubles) { set_error("null argument"); return BA_ERR_INVALID; }
  *device_ptr = e->cost_buf;
  *n_doubles = 4;
  return BA_OK;
}

static int buffer_info(ba_engine* e, int id, const double** p, int64_t* n) {
  switch (id) {
    case BA_BUF_JP: *p = e->JP; *n = e->nobs * kJP; break;
    case BA_BUF_JC: *p = e->JC; *n = e->nobs * kJC; break;
    case BA_BUF_V: *p = e->V; *n = 6 * e->N; break;
    case BA_BUF_GPT: *p = e->GPT; *n = 3 * e->N; break;
    case BA_BUF_U: *p = e->Uloc; *n = (int64_t)81 * e->M; break;
    case BA_BUF_GCAM: *p = e->Uloc + (size_t)81 * e->M; *n = (int64_t)9 * e->M; break;
    case BA_BUF_S: *p = e->red; *n = (int64_t)e->n_pad * e->n_pad; break;
    case BA_BUF_DXI: *p = e->dxi; *n = e->n_full; break;
    case BA_BUF_LINV: *p = e->LINV; *n = 6 * e->N; break;
    case BA_BUF_Z: *p = e->Z; *n = 3 * e->N; break;
    case BA_BUF_REDUCE: *p = e->red; *n = e->red_len; break;
    case BA_BUF_COST: *p = e->cost_buf; *n = 4; break;
    case BA_BUF_YT:
      if (!e->dense) { set_error("buffer YT exists on dense engines only"); return BA_ERR_INVALID; }
      *p = e->Yt; *n = e->k_pad * e->n_pad; break;
    default: set_error("unknown buffer id %d", id); return BA_ERR_INVALID;
  }
  return BA_OK;
}

int ba_buffer_size(ba_engine* e, int id, int64_t* n_doubles) {
  if (!e || !n_doubles) { set_error("null argument"); return BA_ERR_INVALID; }
  const double* p;
  return buffer_info(e, id, &p, n_doubles);
}

int ba_buffer_read(ba_engine* e, int id, double* host_out, int64_t n_doubles, void* stream) {
  if (!e || !host_out) { set_error("null argument"); return BA_ERR_INVALID; }
  const double* p;
  int64_t n;
  BA_TRY(buffer_info(e, id, &p, &n));
  if (n_doubles != n) { set_error("buffer %d holds %lld doubles, caller asked for %lld", id, (long long)n, (long long)n_doubles); return BA_ERR_INVALID; }
  cudaStream_t s = (cudaStream_t)stream;
  BA_CUDA(cudaSetDevice(e->device));
  // dense matrix-free engines do not keep the Jacobian rows: K1 writes them for this read
  if ((id == BA_BUF_JP || id == BA_BUF_JC) && dense_matrix_free(e) && e->have_obs && e->have_state)
    BA_TRY(launch_k1(e, s, false, true));
  BA_CUDA(cudaMemcpyAsync(host_out, p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, s));
  BA_CUDA(cudaStreamSynchronize(s));
  return BA_OK;
}

int ba_reduced_layout(ba_engine* e, int32_t* n_pad, int32_t* n_full, int32_t* rhs_row) {
  if (!e) { set_error("null engine"); return BA_ERR_INVALID; }
  if (n_pad) *n_pad = e->n_pad;
  if (n_full) *n_full = e->n_full;
  if (rhs_row) *rhs_row = e->rhs_row;
  return BA_OK;
}

int64_t ba_launch_count(void) { return g_launch_count; }

int ba_profile_enable(ba_engine* e, int on) {
  if (!e) { set_error("null engine"); return BA_ERR_INVALID; }
  e->profiling = on != 0;
  return BA_OK;
}

static int group_id(const char* g) {
  static const char* names[PG_COUNT] = {"k1", "k2", "k3", "k4", "cost", "other", "syrk", "chol", "comm"};
  for (int i = 0; i < PG_COUNT; ++i)
    if (g && std::strcmp(g, names[i]) == 0) return i;
  return -1;
}

int ba_profile_get(ba_engine* e, const char* group, double* total_ms, int64_t* launches) {
  const int g = group_id(group);
  if (!e || g < 0) { set_error("unknown profile group"); return BA_ERR_INVALID; }
  prof_resolve(e, true);
  if (total_ms) *total_ms = e->prof[g].ms;
  if (launches) *launches = e->prof[g].launches;
  return BA_OK;
}

int ba_profile_reset(ba_engine* e) {
  if (!e) { set_error("null engine"); return BA_ERR_INVALID; }
  prof_resolve(e, false);
  for (int i = 0; i < PG_COUNT; ++i) e->prof[i] = ProfSlot();
  return BA_OK;
}

int ba_covariance(ba_engine* e, double* point_cov, double* cam_cov, double* sigma2, int mem, void* stream) {
  BA_TRY(check_ready(e));
  return covariance(e, point_cov, cam_cov, sigma2, mem, (cudaStream_t)stream);
}

int ba_fp64_peak(int device, int use_dmma, double* tflops) { return fp64_peak(device, use_dmma, tflops); }

int ba_matrix_free(ba_engine* e) { return e && dense_matrix_free(e) ? 1 : 0; }

int ba_syrk_plan_info(int n_cams, int64_t n_points, int tile, int num_sms, int* n_items, int* n_tiles,
                      double* makespan_rows, double* ideal_rows) {
  return syrk_plan_selftest(n_cams, n_points, tile, num_sms, n_items, n_tiles, makespan_rows, ideal_rows);
}

int ba_syrk_emu_info(int64_t k_pad, int32_t* moduli, int* n_moduli, int* bits) {
  return syrk_emu_info(k_pad, moduli, n_moduli, bits);
}
int ba_syrk_emulated(ba_engine* e) { return e && e->syrk.kind == SYRK_EMULATED ? 1 : 0; }

}  // extern "C"
