// Peak rate of tcgen05.mma kind::i8 (B200) with both operands resident in shared memory: no TMA, no
// epilogue, one MMA-issuing thread per CTA (1-SM shapes) or per cluster of two (the 2-SM shape), one
// CTA per SM on every SM.  Reports TOPS, the SM clock measured in the kernel (clock64 against the
// global timer) and the power limit, so that the three come from the same run.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o ubench_i8 tools/ubench_i8.cu && ./ubench_i8
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cuda_runtime.h>

#define CK(x)                                                                                 \
  do {                                                                                        \
    cudaError_t e_ = (x);                                                                     \
    if (e_ != cudaSuccess) {                                                                  \
      std::fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_));         \
      std::exit(1);                                                                           \
    }                                                                                         \
  } while (0)

constexpr int kSmem = 160 * 1024;  // operands (48 KB) + padding: one CTA per SM

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t desc_sw128(unsigned a) {
  return (uint64_t)((a & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)2 << 61);
}

// M x N x 32 int8 MMAs, `iters` of them, accumulating into one int32 accumulator.
template <bool PAIR, int M, int N>
__global__ void __launch_bounds__(128, 1) i8_loop(int iters, long long* cycles, unsigned long long* ns) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t bar;
  __shared__ unsigned tmem_slot;
  const unsigned base = (smem_u32(smem) + 1023u) & ~1023u;
  unsigned rank = 0;
  if (PAIR) asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  for (int i = threadIdx.x; i < 48 * 1024 / 4; i += blockDim.x) reinterpret_cast<unsigned*>(smem + (base - smem_u32(smem)))[i] = 0x01010101u * (i & 7);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x < 32) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(N) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(N) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // operands written by threads, read by the MMA
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if (PAIR) asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
  else __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const unsigned tmem = tmem_slot;
  // S8 x S8 -> S32, K-major; N at bits 17..22, M at 24..28
  const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
  const uint64_t da = desc_sw128(base), db = desc_sw128(base + 16384);
  long long c0 = clock64();
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  if (threadIdx.x == 0 && rank == 0) {
    for (int i = 0; i < iters; ++i) {
      const int k = i & 3;
      if (PAIR)
        asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n}\n"
                     ::"r"(tmem), "l"(da + 2u * k), "l"(db + 2u * k), "r"(idesc), "r"(i));
      else
        asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n"
                     ::"r"(tmem), "l"(da + 2u * k), "l"(db + 2u * k), "r"(idesc), "r"(i));
    }
    if (PAIR)
      asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                   ::"r"(smem_u32(&bar)), "h"((unsigned short)3) : "memory");
    else
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&bar)) : "memory");
  }
  __syncwarp();
  unsigned ok = 0;
  while (!ok)
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(smem_u32(&bar)) : "memory");
  long long c1 = clock64();
  unsigned long long t1;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
  if (threadIdx.x == 0) {
    cycles[blockIdx.x] = c1 - c0;
    ns[blockIdx.x] = t1 - t0;
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if (PAIR) asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
  else __syncthreads();
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(N) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(N) : "memory");
  }
}

template <bool PAIR, int M, int N>
static void run(const char* name, int sms, int iters) {
  auto kern = i8_loop<PAIR, M, N>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
  long long* cyc;
  unsigned long long* ns;
  CK(cudaMalloc(&cyc, sms * sizeof(long long)));
  CK(cudaMalloc(&ns, sms * sizeof(unsigned long long)));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(sms);
  cfg.blockDim = dim3(128);
  cfg.dynamicSmemBytes = kSmem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = PAIR ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  for (int w = 0; w < 2; ++w) CK(cudaLaunchKernelEx(&cfg, kern, iters / 8, cyc, ns));  // warm-up, clocks up
  cudaEvent_t a, b;
  CK(cudaEventCreate(&a));
  CK(cudaEventCreate(&b));
  const int reps = 5;
  CK(cudaEventRecord(a));
  for (int r = 0; r < reps; ++r) CK(cudaLaunchKernelEx(&cfg, kern, iters, cyc, ns));
  CK(cudaEventRecord(b));
  CK(cudaEventSynchronize(b));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, a, b));
  long long hc[1024];
  unsigned long long hn[1024];
  CK(cudaMemcpy(hc, cyc, sms * sizeof(long long), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hn, ns, sms * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  double mhz = 0.0;
  for (int i = 0; i < sms; ++i) mhz += (double)hc[i] / (double)hn[i] * 1e3 / sms;
  const int issuers = PAIR ? sms / 2 : sms;
  const double ops = 2.0 * M * N * 32.0 * iters * issuers * reps;
  const double per_sm_clk = 2.0 * M * N * 32.0 * iters / (PAIR ? 2.0 : 1.0) / ((double)hc[0]);
  std::printf("{\"shape\": \"%s\", \"sms\": %d, \"mma_per_issuer\": %d, \"ms\": %.3f, \"TOPS\": %.1f, "
              "\"sm_clock_MHz\": %.0f, \"int8_ops_per_sm_clk\": %.0f}\n",
              name, sms, iters, ms / reps, ops / (ms * 1e-3) / 1e12, mhz, per_sm_clk);
  CK(cudaFree(cyc));
  CK(cudaFree(ns));
}

int main() {
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  const int sms = prop.multiProcessorCount & ~1;
  if (FILE* f = popen("nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader -i 0", "r")) {
    char line[256] = {0};
    if (fgets(line, sizeof line, f)) std::printf("{\"gpu\": \"%s\", \"nvidia_smi\": \"%.*s\"}\n", prop.name, (int)strcspn(line, "\n"), line);
    pclose(f);
  }
  const int iters = 1 << 18;
  run<false, 128, 128>("1sm_128x128x32", sms, iters);
  run<false, 128, 256>("1sm_128x256x32", sms, iters / 2);
  run<true, 256, 256>("2sm_256x256x32", sms, iters / 2);
  return 0;
}
