// Micro-benchmark (diagnostic, not on the product path): how fast can one CTA stream a shared 4.2 MB weight
// image from L2 into a shared-memory mbarrier ring with cp.async.bulk, as a function of stage size, ring depth
// and cluster multicast?  Mirrors the weight-producer/consumer handshake of point_tc.cu without the MMAs.
#include <cstdio>
#include <vector>

#include "common.cuh"
#include "tc_common.cuh"

namespace disn {
namespace {

constexpr int MAX_STAGES = 16;

struct ProbeSmem {
  alignas(8) uint64_t full[MAX_STAGES];
  uint64_t empty[MAX_STAGES];
};

// mode 0: every CTA loads its own copy of each stage (what point_tc.cu does today)
// mode 1: cluster of CS CTAs; stage g is loaded by CTA (g % CS) and multicast to all CS CTAs
template <int CS>
__global__ void __launch_bounds__(128, 1)
probe_kernel(const uint8_t* __restrict__ src, uint32_t image_bytes, uint32_t stage_bytes, int nstages, int iters,
             int mode, int consume_delay, unsigned long long* __restrict__ out) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
  ProbeSmem& s = *reinterpret_cast<ProbeSmem*>(base);
  uint8_t* ring = base + 1024;
  const uint32_t cta = (CS > 1) ? tc::cluster_ctarank() : 0;
  const int tid = threadIdx.x;
  if (tid == 0) {
    for (int i = 0; i < nstages; ++i) { tc::mbar_init(&s.full[i], 1); tc::mbar_init(&s.empty[i], (mode == 1) ? CS : 1); }
    tc::fence_barrier_init();
  }
  if (CS > 1) tc::cluster_sync(); else __syncthreads();
  const int per_image = image_bytes / stage_bytes;
  const int total = per_image * iters;
  long long t0 = clock64();
  const int P = (mode >= 20) ? (mode - 20) : 1;     // mode 20+P: P producer lanes, stage g issued by lane g % P
  if (mode >= 20) {
    if (tid < P) {
      for (int g = tid; g < total; g += P) {
        const int st = g % nstages;
        tc::mbar_wait(&s.empty[st], ((g / nstages) & 1) ^ 1);
        tc::mbar_arrive_expect_tx(&s.full[st], stage_bytes);
        tc::bulk_g2s(ring + (size_t)st * stage_bytes, src + (size_t)(g % per_image) * stage_bytes, stage_bytes, &s.full[st]);
      }
    }
  } else if (mode == 3) {
    if (tid == 0) {
      for (int g = 0; g < total; ++g) {
        const int st = g % nstages;
        tc::mbar_wait(&s.empty[st], ((g / nstages) & 1) ^ 1);
        tc::mbar_arrive_expect_tx(&s.full[st], stage_bytes);
        const uint8_t* p = src + (size_t)(g % per_image) * stage_bytes;
        tc::bulk_g2s(ring + (size_t)st * stage_bytes, p, stage_bytes / 2, &s.full[st]);
        tc::bulk_g2s(ring + (size_t)st * stage_bytes + stage_bytes / 2, p + stage_bytes / 2, stage_bytes / 2, &s.full[st]);
      }
    }
  } else if (mode == 4) {    // burst: issue `nstages` copies back to back, wait for all; repeated -> are bulk copies pipelined?
    unsigned long long acc = 0, acc_issue = 0;
    for (int rep = 0; rep < 16; ++rep) {
      __syncthreads();
      const long long tb = clock64();
      if (tid == 0) {
        for (int st = 0; st < nstages; ++st) {
          tc::mbar_arrive_expect_tx(&s.full[st], stage_bytes);
          tc::bulk_g2s(ring + (size_t)st * stage_bytes, src + (size_t)((rep * nstages + st) % per_image) * stage_bytes, stage_bytes, &s.full[st]);
        }
        acc_issue += (unsigned long long)(clock64() - tb);
        for (int st = 0; st < nstages; ++st) tc::mbar_wait(&s.full[st], rep & 1);
        acc += (unsigned long long)(clock64() - tb);
      }
    }
    __syncthreads();
    if (tid == 0) { out[blockIdx.x] = acc / 16; out[256 + blockIdx.x] = acc_issue / 16; }
    return;
  } else if (tid == 0) {            // producer
    unsigned long long wsum = 0;
    for (int g = 0; g < total; ++g) {
      const int st = g % nstages;
      const long long tw = clock64();
      tc::mbar_wait(&s.empty[st], ((g / nstages) & 1) ^ 1);
      wsum += (unsigned long long)(clock64() - tw);
      if (g == total - 1) out[256 + blockIdx.x] = wsum;
      tc::mbar_arrive_expect_tx(&s.full[st], stage_bytes);
      const uint8_t* p = src + (size_t)(g % per_image) * stage_bytes;
      if (mode == 0) {
        tc::bulk_g2s(ring + (size_t)st * stage_bytes, p, stage_bytes, &s.full[st]);
      } else if ((uint32_t)(g % CS) == cta) {
        const uint16_t mask = (uint16_t)((1u << CS) - 1u);
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;"
            ::"r"(tc::smem_u32(ring + (size_t)st * stage_bytes)), "l"(p), "r"(stage_bytes), "r"(tc::smem_u32(&s.full[st])),
              "h"(mask)
            : "memory");
      }
    }
  }
  if (tid == 32) {    // consumer
    unsigned long long wsum = 0;
    for (int g = 0; g < total; ++g) {
      const int st = g % nstages;
      const long long tw = clock64();
      tc::mbar_wait(&s.full[st], (g / nstages) & 1);
      wsum += (unsigned long long)(clock64() - tw);
      if (g == total - 1) out[384 + blockIdx.x] = wsum;
      if (consume_delay) { long long t = clock64(); while (clock64() - t < consume_delay) {} }
      if (mode == 1) { for (int c = 0; c < CS; ++c) tc::mbar_arrive_cluster(&s.empty[st], c); }
      else tc::mbar_arrive(&s.empty[st]);
    }
  }
  __syncthreads();
  if (CS > 1) tc::cluster_sync();
  if (tid == 0) out[blockIdx.x] = (unsigned long long)(clock64() - t0);
}

}  // namespace
}  // namespace disn

// Prints bytes/clk/SM for a sweep; returns 0.  Diagnostic entry point (tests/bench never depend on it).
extern "C" int disn_tc_stream_probe(int device) {
  using namespace disn;
  DISN_CUDA_OK(cudaSetDevice(device));
  const uint32_t image = 4u << 20;
  DevBuf bsrc, bout;
  if (bsrc.reserve(image) || bout.reserve(512 * sizeof(unsigned long long))) return -1;
  uint8_t* src = bsrc.get<uint8_t>();
  unsigned long long* out = bout.get<unsigned long long>();
  DISN_CUDA_OK(cudaMemset(src, 1, image));
  const int grid = 148;
  auto run = [&](int cs, int mode, uint32_t stage, int ns, int delay) -> int {
    const int smem = 2048 + (int)stage * ns + 1024;
    const int iters = 8;
    void (*k)(const uint8_t*, uint32_t, uint32_t, int, int, int, int, unsigned long long*) =
        cs == 1 ? probe_kernel<1> : cs == 2 ? probe_kernel<2> : cs == 4 ? probe_kernel<4> : probe_kernel<8>;
    DISN_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid - grid % cs);
    cfg.blockDim = dim3(128);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    for (int rep = 0; rep < 2; ++rep) {
      DISN_CUDA_OK(cudaLaunchKernelEx(&cfg, k, (const uint8_t*)src, image, stage, ns, iters, mode, delay, out));
      DISN_CUDA_OK(cudaDeviceSynchronize());
    }
    std::vector<unsigned long long> h(512);
    DISN_CUDA_OK(cudaMemcpy(h.data(), out, 512 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    double mx = 0;
    for (int i = 0; i < grid - grid % cs; ++i) mx = std::max(mx, (double)h[i]);
    if (mode == 0 && cs == 1)
      printf("[probe]   per stage: producer waits on empty %.0f cycles, consumer waits on full %.0f cycles\n",
             (double)h[256] / ((double)(image / stage) * iters), (double)h[384] / ((double)(image / stage) * iters));
    printf("[probe] cluster=%d mode=%-9s stage=%2uKB depth=%2d (ring %3u KB) delay=%4d : %6.1f B/clk/SM into smem, %7.0f cycles/stage\n",
           cs, mode == 0 ? "private" : mode == 1 ? "multicast" : mode == 3 ? "2copies" : mode == 4 ? "freerun" : mode == 22 ? "2lanes" : mode == 24 ? "4lanes" : "?", stage >> 10, ns, (stage * ns) >> 10, delay,
           (double)image * iters / mx, mx / ((double)(image / stage) * iters));
    return 0;
  };
  // burst latency: n copies issued back to back by one thread, time until all have landed
  for (uint32_t stage : {4096u, 16384u, 32768u})
    for (int ns : {1, 2, 4, 6}) {
      if ((int)stage * ns > 200 * 1024) continue;
      const int smem = 2048 + (int)stage * ns + 1024;
      DISN_CUDA_OK(cudaFuncSetAttribute(probe_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      probe_kernel<1><<<148, 128, smem>>>(src, image, stage, ns, 1, 4, 0, out);
      DISN_CUDA_OK(cudaDeviceSynchronize());
      std::vector<unsigned long long> h(512);
      DISN_CUDA_OK(cudaMemcpy(h.data(), out, 512 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
      double a = 0, b = 0;
      for (int i = 0; i < 148; ++i) { a += (double)h[i] / 148; b += (double)h[256 + i] / 148; }
      printf("[probe] burst of %d x %2u KB copies: issue %6.0f cycles, all landed after %6.0f cycles (%5.1f B/clk/SM)\n", ns,
             stage >> 10, b, a, (double)stage * ns / a);
    }
  for (uint32_t stage : {16384u}) {
    if (run(1, 0, stage, 2, 0)) return -1;
    if (run(1, 0, stage, 6, 0)) return -1;
  }
  if (run(1, 0, 16384u, 6, 384)) return -1;     // consumer paced like the MMA at full rate (16 KB / 384 clk)
  if (run(1, 0, 32768u, 3, 768)) return -1;
  fflush(stdout);
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// Issue-cost micro-benchmark of the synchronisation instructions on the MMA warp's path (diagnostic).
// One warp, ITER back-to-back instances of each op; prints average cycles per op.
// ---------------------------------------------------------------------------------------------------------
namespace disn {
namespace {

__global__ void __launch_bounds__(32, 1) op_cost_kernel(unsigned long long* __restrict__ out) {
  __shared__ alignas(8) uint64_t done_bar;    // phase 0 completed -> try_wait(parity 0) succeeds immediately
  __shared__ alignas(8) uint64_t big_bar;     // huge count: arrivals never complete a phase
  __shared__ volatile uint32_t flag;
  const int lane = threadIdx.x;
  if (lane == 0) {
    tc::mbar_init(&done_bar, 1);
    tc::mbar_init(&big_bar, 1u << 19);
    tc::fence_barrier_init();
    flag = 1;
  }
  __syncwarp();
  if (lane == 0) tc::mbar_arrive(&done_bar);
  __syncwarp();
  constexpr int ITER = 64;
  uint32_t acc = 0;
  const uint32_t db = tc::smem_u32(&done_bar), bb = tc::smem_u32(&big_bar);
  long long t;
  int slot = 0;
#define MEASURE(cond, body)                                          \
  __syncwarp();                                                      \
  t = clock64();                                                     \
  if (cond) {                                                        \
    _Pragma("unroll 1") for (int i = 0; i < ITER; ++i) { body; }     \
  }                                                                  \
  __syncwarp();                                                      \
  if (lane == 0) out[slot] = (unsigned long long)(clock64() - t) / ITER; \
  ++slot;

  // 0: empty loop
  MEASURE(true, asm volatile("" ::: "memory"));
  // 1: try_wait (default acquire.cta), all 32 lanes
  MEASURE(true, { uint32_t ok; asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(db), "r"(0u) : "memory"); acc += ok; });
  // 2: try_wait, lane 0 only
  MEASURE(lane == 0, { uint32_t ok; asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(db), "r"(0u) : "memory"); acc += ok; });
  // 3: try_wait.relaxed.cta, all lanes
  MEASURE(true, { uint32_t ok; asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.relaxed.cta.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(db), "r"(0u) : "memory"); acc += ok; });
  // 4: try_wait.relaxed.cta, lane 0
  MEASURE(lane == 0, { uint32_t ok; asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.relaxed.cta.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(db), "r"(0u) : "memory"); acc += ok; });
  // 5: test_wait, all lanes
  MEASURE(true, { uint32_t ok; asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(db), "r"(0u) : "memory"); acc += ok; });
  // 6: test_wait, lane 0
  MEASURE(lane == 0, { uint32_t ok; asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(db), "r"(0u) : "memory"); acc += ok; });
  // 7: mbarrier.arrive lane 0
  MEASURE(lane == 0, asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bb) : "memory"));
  // 8: tcgen05.commit (cta_group::1, nothing outstanding), lane 0
  MEASURE(lane == 0, asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bb) : "memory"));
  // 9: volatile shared load, all lanes (dependent chain through acc)
  MEASURE(true, acc += flag);
  // 10: tcgen05.fence::after_thread_sync
  MEASURE(true, tc::tc_fence_after_sync());
  // 11: fence.proxy.async.shared::cta
  MEASURE(true, tc::fence_proxy_async_smem());
  // 12: elect_one + branch
  MEASURE(true, if (tc::elect_one()) acc += 1);
  // 13: try_wait all lanes followed by tcgen05 fence (the MMA warp's pattern)
  MEASURE(true, { uint32_t ok; asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(db), "r"(0u) : "memory"); acc += ok; tc::tc_fence_after_sync(); });
#undef MEASURE
  if (acc == 0xFFFFFFFFu) out[63] = acc;
}

}  // namespace
}  // namespace disn

extern "C" int disn_tc_op_probe(int device) {
  using namespace disn;
  DISN_CUDA_OK(cudaSetDevice(device));
  DevBuf bd;
  if (bd.reserve(64 * sizeof(unsigned long long))) return -1;
  unsigned long long* d = bd.get<unsigned long long>();
  DISN_CUDA_OK(cudaMemset(d, 0, 64 * sizeof(unsigned long long)));
  op_cost_kernel<<<1, 32>>>(d);
  DISN_CUDA_OK(cudaGetLastError());
  DISN_CUDA_OK(cudaDeviceSynchronize());
  unsigned long long h[64];
  DISN_CUDA_OK(cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost));
  const char* names[14] = {"empty loop", "try_wait acquire (32 lanes)", "try_wait acquire (1 lane)", "try_wait relaxed (32 lanes)",
                           "try_wait relaxed (1 lane)", "test_wait (32 lanes)", "test_wait (1 lane)", "mbarrier.arrive (1 lane)",
                           "tcgen05.commit idle (1 lane)", "ld.volatile.shared (32 lanes)", "tcgen05.fence::after_thread_sync",
                           "fence.proxy.async.shared::cta", "elect.sync + branch", "try_wait + tcgen05 fence (32 lanes)"};
  for (int i = 0; i < 14; ++i) printf("[op_probe] %-40s %llu cycles/op\n", names[i], h[i]);
  fflush(stdout);
  return 0;
}
