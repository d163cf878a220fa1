// Self-test of the tcgen05 cta_group::2 building blocks used by the tensor-core point kernel:
// one CTA pair computes D[128 x 256] = A[128 x 64] * B[256 x 64]^T (bf16 in, fp32 accumulate) twice
// (second pass accumulates), exercising TMEM allocation, SW128 K-major descriptors written by threads
// (A) and by the bulk-copy engine from a host-swizzled image (B), the peer-CTA full-barrier relay,
// multicast commit, and the 2x2 datapath TMEM layout read back with tcgen05.ld.32x32b.
#include <vector>

#include "common.cuh"
#include "tc_common.cuh"

namespace disn {
namespace {

struct SelfSmem {
  alignas(1024) uint8_t a_tile[64 * 128];     // 64 rows x 64 bf16, SW128
  alignas(1024) uint8_t b_tile[128 * 128];    // 128 rows x 64 bf16, SW128
  alignas(8) uint64_t b_full;                 // bulk copy of this CTA's B half landed
  uint64_t peer_full;                         // (leader) peer CTA's operands are ready
  uint64_t mma_done;                          // accumulators complete (multicast to both CTAs)
  uint32_t tmem_base;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1)
tc_selftest_kernel(const __nv_bfloat16* __restrict__ A,       // [128][64] row-major
                   const uint8_t* __restrict__ Bimg,          // 2 x 16 KB pre-swizzled halves
                   float* __restrict__ D,                     // [2 ctas][128 lanes][128 cols]
                   int passes) {
  extern __shared__ uint8_t smem_raw[];
  // dynamic smem is only 16-B aligned by contract: round the shared-window address up to 1024 B
  SelfSmem& s = *reinterpret_cast<SelfSmem*>(smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u));
  const uint32_t cta = tc::cluster_ctarank();
  const int tid = threadIdx.x, warp = tid / 32;

  if (tid == 0) {
    tc::mbar_init(&s.b_full, 1);
    tc::mbar_init(&s.peer_full, 1);
    tc::mbar_init(&s.mma_done, 1);
    tc::fence_barrier_init();
  }
  if (warp == 0) {
    tc::tmem_alloc_cg2(&s.tmem_base, 256);
    tc::tmem_relinquish_cg2();
  }
  // A half of this CTA written by threads exactly like the epilogue will: thread = row, 8 x 16 B chunks
  if (tid < 64) {
    const uint4* src = reinterpret_cast<const uint4*>(A + (size_t)(cta * 64 + tid) * 64);
#pragma unroll
    for (int c = 0; c < 8; ++c) *reinterpret_cast<uint4*>(s.a_tile + tc::sw128_offset(tid, c)) = src[c];
  }
  tc::fence_proxy_async_smem();
  tc::tc_fence_before_sync();
  tc::cluster_sync();
  tc::tc_fence_after_sync();
  const uint32_t tmem = s.tmem_base;

  if (tid == 0) {   // B half via the bulk-copy engine
    tc::mbar_arrive_expect_tx(&s.b_full, 128 * 128);
    tc::bulk_g2s(s.b_tile, Bimg + (size_t)cta * 128 * 128, 128 * 128, &s.b_full);
  }
  if (cta == 1 && tid == 32) {   // relay: tell the leader that this CTA's A (fenced above) and B are in place
    tc::mbar_wait(&s.b_full, 0);
    tc::mbar_arrive_cluster(&s.peer_full, 0);
  }
  if (cta == 0 && tid == 32) {   // MMA issuer
    tc::mbar_wait(&s.b_full, 0);
    tc::mbar_wait_cluster(&s.peer_full, 0);
    tc::tc_fence_after_sync();
    const uint32_t idesc = tc::make_idesc_bf16(128, 256);
    const uint64_t adesc = tc::make_desc_sw128(tc::smem_u32(s.a_tile));
    const uint64_t bdesc = tc::make_desc_sw128(tc::smem_u32(s.b_tile));
    for (int p = 0; p < passes; ++p)
      for (int k = 0; k < 4; ++k)
        tc::mma_cg2(tmem, tc::desc_advance_k(adesc, k * 16), tc::desc_advance_k(bdesc, k * 16), idesc,
                    (p | k) ? 1u : 0u);
    tc::commit_cg2(&s.mma_done, 0b11);
  }
  __syncwarp();
  tc::mbar_wait(&s.mma_done, 0);
  tc::tc_fence_after_sync();
  // read back: thread -> lane 32*warp + t, 128 columns
  const int lane_row = warp * 32 + (tid & 31);
  for (int c0 = 0; c0 < 128; c0 += 32) {
    uint32_t r[32];
    tc::tmem_ld_x32(tmem + ((uint32_t)(warp * 32) << 16) + c0, r);
    tc::tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 32; ++j) D[((size_t)cta * 128 + lane_row) * 128 + c0 + j] = __uint_as_float(r[j]);
  }
  tc::tc_fence_before_sync();
  tc::cluster_sync();
  if (warp == 0) tc::tmem_dealloc_cg2(tmem, 256);
}

}  // namespace
}  // namespace disn

// Returns 0 and max |D - ref| in *max_err. Host pointers: A [128*64] fp32 values (rounded to bf16 inside),
// B [256*64] fp32.  Exposed through the C ABI for the GPU test-suite.
extern "C" int disn_tc_selftest(int device, const float* A, const float* B, int passes, float* D_out /*[2*128*128]*/) {
  using namespace disn;
  DISN_CUDA_OK(cudaSetDevice(device));
  std::vector<__nv_bfloat16> a(128 * 64);
  for (int i = 0; i < 128 * 64; ++i) a[i] = __float2bfloat16(A[i]);
  std::vector<uint8_t> bimg(2 * 128 * 128);
  for (int n = 0; n < 256; ++n)
    for (int k = 0; k < 64; ++k) {
      __nv_bfloat16 v = __float2bfloat16(B[n * 64 + k]);
      int half = n / 128, row = n % 128;
      uint32_t off = tc::sw128_offset(row, k / 8) + (k % 8) * 2;
      memcpy(&bimg[(size_t)half * 128 * 128 + off], &v, 2);
    }
  DevBuf bA, bB, bD;
  if (bA.reserve(a.size() * 2) || bB.reserve(bimg.size()) || bD.reserve(2 * 128 * 128 * sizeof(float))) return -1;
  __nv_bfloat16* dA = bA.get<__nv_bfloat16>();
  uint8_t* dB = bB.get<uint8_t>();
  float* dD = bD.get<float>();
  DISN_CUDA_OK(cudaMemcpy(dA, a.data(), a.size() * 2, cudaMemcpyHostToDevice));
  DISN_CUDA_OK(cudaMemcpy(dB, bimg.data(), bimg.size(), cudaMemcpyHostToDevice));
  DISN_CUDA_OK(cudaMemset(dD, 0xff, 2 * 128 * 128 * sizeof(float)));
  DISN_CUDA_OK(cudaFuncSetAttribute(tc_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)sizeof(SelfSmem) + 1024));
  tc_selftest_kernel<<<2, 128, sizeof(SelfSmem) + 1024>>>(dA, dB, dD, passes);
  DISN_CUDA_OK(cudaGetLastError());
  DISN_CUDA_OK(cudaDeviceSynchronize());
  DISN_CUDA_OK(cudaMemcpy(D_out, dD, 2 * 128 * 128 * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// Mixed-kind self-test (building block of DISN_PREC_F16F8): one accumulator receives
//   D = fp16(A16) * fp16(B16)^T   (kind::f16, SW128 tiles, 4 x K=16)
//     + e5m2(A8) * e5m2(B8)^T     (kind::f8f6f4, SW64 tiles of bytes, 2 x K=32)
// mode bit 0 enables the f16 part, bit 1 the f8 part.
// ---------------------------------------------------------------------------------------------------------
#include <cuda_fp16.h>
#include <cuda_fp8.h>

namespace disn {
namespace {

struct MixSmem {
  alignas(1024) uint8_t a16[64 * 128];
  alignas(1024) uint8_t b16[128 * 128];
  alignas(1024) uint8_t a8[64 * 64];
  alignas(1024) uint8_t b8[128 * 64];
  alignas(8) uint64_t b_full;
  uint64_t peer_full;
  uint64_t mma_done;
  uint32_t tmem_base;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1)
tc_selftest_mixed_kernel(const __half* __restrict__ A16, const uint8_t* __restrict__ A8,      // [128][64] row-major
                         const uint8_t* __restrict__ Bimg,   // per CTA: 16 KB SW128 fp16 + 8 KB SW64 e5m2
                         float* __restrict__ D, int mode) {
  extern __shared__ uint8_t smem_raw[];
  MixSmem& s = *reinterpret_cast<MixSmem*>(smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u));
  const uint32_t cta = tc::cluster_ctarank();
  const int tid = threadIdx.x, warp = tid / 32;
  if (tid == 0) {
    tc::mbar_init(&s.b_full, 1);
    tc::mbar_init(&s.peer_full, 1);
    tc::mbar_init(&s.mma_done, 1);
    tc::fence_barrier_init();
  }
  if (warp == 0) {
    tc::tmem_alloc_cg2(&s.tmem_base, 256);
    tc::tmem_relinquish_cg2();
  }
  if (tid < 64) {
    const uint4* src = reinterpret_cast<const uint4*>(A16 + (size_t)(cta * 64 + tid) * 64);
#pragma unroll
    for (int c = 0; c < 8; ++c) *reinterpret_cast<uint4*>(s.a16 + tc::sw128_offset(tid, c)) = src[c];
    const uint4* src8 = reinterpret_cast<const uint4*>(A8 + (size_t)(cta * 64 + tid) * 64);
#pragma unroll
    for (int c = 0; c < 4; ++c) *reinterpret_cast<uint4*>(s.a8 + tc::sw64_offset(tid, c)) = src8[c];
  }
  tc::fence_proxy_async_smem();
  tc::tc_fence_before_sync();
  tc::cluster_sync();
  tc::tc_fence_after_sync();
  const uint32_t tmem = s.tmem_base;
  if (tid == 0) {
    tc::mbar_arrive_expect_tx(&s.b_full, 128 * 128 + 128 * 64);
    tc::bulk_g2s(s.b16, Bimg + (size_t)cta * (128 * 192), 128 * 128, &s.b_full);
    tc::bulk_g2s(s.b8, Bimg + (size_t)cta * (128 * 192) + 128 * 128, 128 * 64, &s.b_full);
  }
  if (cta == 1 && tid == 32) {
    tc::mbar_wait(&s.b_full, 0);
    tc::mbar_arrive_cluster(&s.peer_full, 0);
  }
  if (cta == 0 && tid == 32) {
    tc::mbar_wait(&s.b_full, 0);
    tc::mbar_wait_cluster(&s.peer_full, 0);
    tc::tc_fence_after_sync();
    const uint32_t a16 = tc::desc_lo(tc::smem_u32(s.a16)), b16 = tc::desc_lo(tc::smem_u32(s.b16));
    const uint32_t a8 = tc::desc_lo(tc::smem_u32(s.a8)), b8 = tc::desc_lo(tc::smem_u32(s.b8));
    uint32_t acc = 0;
    if (mode & 1)
      for (int k = 0; k < 4; ++k) { tc::mma_cg2_lo(tmem, a16 + 2u * k, b16 + 2u * k, tc::make_idesc_f16(128, 256), acc); acc = 1; }
    if (mode & 2)
      for (int k = 0; k < 2; ++k) { tc::mma_cg2_f8_lo(tmem, a8 + 2u * k, b8 + 2u * k, tc::make_idesc_e5m2(128, 256), acc); acc = 1; }
    tc::commit_cg2(&s.mma_done, 0b11);
  }
  __syncwarp();
  tc::mbar_wait(&s.mma_done, 0);
  tc::tc_fence_after_sync();
  const int lane_row = warp * 32 + (tid & 31);
  for (int c0 = 0; c0 < 128; c0 += 32) {
    uint32_t r[32];
    tc::tmem_ld_x32(tmem + ((uint32_t)(warp * 32) << 16) + c0, r);
    tc::tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 32; ++j) D[((size_t)cta * 128 + lane_row) * 128 + c0 + j] = __uint_as_float(r[j]);
  }
  tc::tc_fence_before_sync();
  tc::cluster_sync();
  if (warp == 0) tc::tmem_dealloc_cg2(tmem, 256);
}

}  // namespace
}  // namespace disn

// Host fp32 inputs A16,A8 [128*64], B16,B8 [256*64]; the e5m2 roundings actually used are returned in A8q/B8q so the
// caller can form the exact reference.  D_out [2*128*128] in TMEM (cta, lane, column) order.
extern "C" int disn_tc_selftest_mixed(int device, const float* A16, const float* B16, const float* A8, const float* B8,
                                      int mode, float* A8q, float* B8q, float* D_out) {
  using namespace disn;
  DISN_CUDA_OK(cudaSetDevice(device));
  std::vector<__half> a16(128 * 64);
  std::vector<uint8_t> a8(128 * 64), bimg(2 * 128 * 192);
  for (int i = 0; i < 128 * 64; ++i) {
    a16[i] = __float2half_rn(A16[i]);
    a8[i] = (uint8_t)__nv_cvt_float_to_fp8(A8[i], __NV_SATFINITE, __NV_E5M2);
    A8q[i] = __half2float(__half(__nv_cvt_fp8_to_halfraw(a8[i], __NV_E5M2)));
  }
  for (int n = 0; n < 256; ++n)
    for (int k = 0; k < 64; ++k) {
      const int half = n / 128, row = n % 128;
      __half v = __float2half_rn(B16[n * 64 + k]);
      memcpy(&bimg[(size_t)half * 128 * 192 + tc::sw128_offset(row, k / 8) + (k % 8) * 2], &v, 2);
      const uint8_t q = (uint8_t)__nv_cvt_float_to_fp8(B8[n * 64 + k], __NV_SATFINITE, __NV_E5M2);
      bimg[(size_t)half * 128 * 192 + 128 * 128 + tc::sw64_offset(row, k / 16) + (k % 16)] = q;
      B8q[n * 64 + k] = __half2float(__half(__nv_cvt_fp8_to_halfraw(q, __NV_E5M2)));
    }
  DevBuf bA, bA8, bB, bD;
  if (bA.reserve(a16.size() * 2) || bA8.reserve(a8.size()) || bB.reserve(bimg.size()) ||
      bD.reserve(2 * 128 * 128 * sizeof(float)))
    return -1;
  __half* dA = bA.get<__half>();
  uint8_t *dA8 = bA8.get<uint8_t>(), *dB = bB.get<uint8_t>();
  float* dD = bD.get<float>();
  DISN_CUDA_OK(cudaMemcpy(dA, a16.data(), a16.size() * 2, cudaMemcpyHostToDevice));
  DISN_CUDA_OK(cudaMemcpy(dA8, a8.data(), a8.size(), cudaMemcpyHostToDevice));
  DISN_CUDA_OK(cudaMemcpy(dB, bimg.data(), bimg.size(), cudaMemcpyHostToDevice));
  DISN_CUDA_OK(cudaMemset(dD, 0xff, 2 * 128 * 128 * sizeof(float)));
  DISN_CUDA_OK(cudaDeviceSynchronize());
  DISN_CUDA_OK(cudaFuncSetAttribute(tc_selftest_mixed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)sizeof(MixSmem) + 1024));
  tc_selftest_mixed_kernel<<<2, 128, sizeof(MixSmem) + 1024>>>(dA, dA8, dB, dD, mode);
  DISN_CUDA_OK(cudaGetLastError());
  DISN_CUDA_OK(cudaDeviceSynchronize());
  DISN_CUDA_OK(cudaMemcpy(D_out, dD, 2 * 128 * 128 * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}
