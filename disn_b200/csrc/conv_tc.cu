// Implicit-GEMM convolution / GEMM on tcgen05 tensor cores for the image encoder (sm_100a).
//
//   C[M, N] = act( A[M, K] * W[K, N] + bias ),  A = NHWC activations viewed through a 3x3 SAME im2col
//   (K = 9*Cin, k = tap*Cin + ci -- the row order of TF's HWIO weights) or a plain row-major matrix.
//
// Same precision scheme as the point kernel: every fp32 operand is split into bf16 hi + lo and each product is
// three MMAs (hi*hi + lo*hi + hi*lo) with fp32 accumulation in TMEM, so the encoder keeps fp32-level accuracy
// (the reference runs VGG in fp32; models/CNN/vgg.py:187-196, models/model_normalization.py:76).
//
// One CTA = one SM: UMMA M=128 (pixels) x N=128 (output channels) x K=16, 64-wide K slices.
//   warps 8-15  A producers (two groups of 4 warps alternate slices): a half-warp gathers the 64 channels of one
//               filter tap of one pixel row (256 contiguous bytes, coalesced; zeros outside the image), splits to
//               bf16 hi/lo and writes the K-major 128B-swizzled A tile
//   warp 0      B producer: host-packed [W_hi | W_lo] 32 KB stage images via cp.async.bulk
//   warp 1      MMA issuer (warp-uniform loop, elected lane), two TMEM accumulators (ping-pong across jobs)
//   warps 4-7   epilogue: TMEM -> +bias, ReLU -> fp32 NHWC store (or raw split-K partials to the workspace)
// Jobs = (m-tile, n-block, k-split); a persistent grid walks them.  Under-filled layers are split along K and
// reduced by splitk_reduce_kernel.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "tc_common.cuh"

namespace disn {
namespace {

constexpr int CT_THREADS = 512;
constexpr int CT_NA = 4;            // A ring slots (2 per producer group)
constexpr int CT_NB = 3;            // B ring slots
constexpr int CT_A_HALF = 16384;    // 128 rows x 64 k x bf16
constexpr int CT_B_TILE = 16384;    // 128 rows x 64 k x bf16
constexpr int CT_B_STAGE = 2 * CT_B_TILE;

struct ConvTcSmem {
  alignas(1024) uint8_t a[CT_NA][2][CT_A_HALF];    // [slot][hi|lo]   128 KB
  alignas(1024) uint8_t b[CT_NB][CT_B_STAGE];      // [slot][hi|lo]    96 KB
  alignas(8) uint64_t afull[CT_NA];
  uint64_t aempty[CT_NA];
  uint64_t bfull[CT_NB];
  uint64_t bempty[CT_NB];
  uint64_t acc_full[2];
  uint64_t acc_free[2];
  uint32_t tmem_base;
};

struct ConvTcJob {
  const float* A;          // NHWC activations [B,H,W,Cin] or row-major [M,K]
  const uint8_t* wpk;      // packed weights: [n-block][k-slice][hi|lo][128 x 64 SW128]
  const float* bias;       // [N] or nullptr
  float* C;                // [M,N] fp32
  float* ws;               // split-K workspace [splits][M][N] or nullptr
  int M, N, K;             // K multiple of 64
  int H, W, Cin;           // im2col geometry (Cin multiple of 64); H == 0 -> plain matrix
  int relu;
  int m_tiles, n_blocks, splits, slices_per_split;
};

// kMeasure: every warp's lane 0 accounts the cycles it spends blocked on each barrier class (DISN_CONV_MEASURE=1)
enum { CW_BEMPTY = 0, CW_ACCFREE, CW_AFULL, CW_BFULL, CW_ACCFULL, CW_AEMPTY, CW_NCLS };
template <bool kMeasure>
__global__ void __launch_bounds__(CT_THREADS, 1) conv_tc_kernel(ConvTcJob job, unsigned long long* __restrict__ dbg) {
  unsigned long long wt[CW_NCLS] = {0, 0, 0, 0, 0, 0};
  const long long t_start = kMeasure ? clock64() : 0;
#define CWAIT(cls, bar, par)                                         \
  do {                                                               \
    if constexpr (kMeasure) {                                        \
      const long long _t = clock64();                                \
      tc::mbar_wait(bar, par);                                       \
      wt[cls] += (unsigned long long)(clock64() - _t);               \
    } else {                                                         \
      tc::mbar_wait(bar, par);                                       \
    }                                                                \
  } while (0)
  extern __shared__ uint8_t smem_raw[];
  ConvTcSmem& s = *reinterpret_cast<ConvTcSmem*>(smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int total_jobs = job.m_tiles * job.n_blocks * job.splits;
  const int my_jobs = ((int)blockIdx.x < total_jobs) ? (total_jobs - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int nsl = job.slices_per_split;

  if (tid == 0) {
    for (int i = 0; i < CT_NA; ++i) { tc::mbar_init(&s.afull[i], 4); tc::mbar_init(&s.aempty[i], 1); }
    for (int i = 0; i < CT_NB; ++i) { tc::mbar_init(&s.bfull[i], 1); tc::mbar_init(&s.bempty[i], 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&s.acc_full[i], 1); tc::mbar_init(&s.acc_free[i], 4); }
    tc::fence_barrier_init();
  }
  if (warp == 2) {
    tc::tmem_alloc_cg1(&s.tmem_base, 256);
    tc::tmem_relinquish_cg1();
  }
  tc::tc_fence_before_sync();
  __syncthreads();
  tc::tc_fence_after_sync();
  const uint32_t tmem = s.tmem_base;

  // job index -> (m-tile, n-block, split): n-block fastest so neighbouring CTAs share the A rows in L2
  auto decode = [&](int j, int& mt, int& nb, int& sp) {
    nb = j % job.n_blocks;
    const int r = j / job.n_blocks;
    mt = r % job.m_tiles;
    sp = r / job.m_tiles;
  };

  if (warp == 0) {
    // ===================== B producer =====================
    if (lane == 0) {
      uint32_t seq = 0;
      for (int jj = 0; jj < my_jobs; ++jj) {
        int mt, nb, sp;
        decode((int)blockIdx.x + jj * (int)gridDim.x, mt, nb, sp);
        const uint8_t* src = job.wpk + ((size_t)nb * (job.K / 64) + (size_t)sp * nsl) * CT_B_STAGE;
        for (int t = 0; t < nsl; ++t, ++seq) {
          const int st = seq % CT_NB;
          CWAIT(CW_BEMPTY, &s.bempty[st], ((seq / CT_NB) & 1) ^ 1);
          tc::mbar_arrive_expect_tx(&s.bfull[st], CT_B_STAGE);
          tc::bulk_g2s(s.b[st], src + (size_t)t * CT_B_STAGE, CT_B_STAGE, &s.bfull[st]);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t idesc = tc::make_idesc_bf16(128, 128);
    const uint32_t a_lo0 = tc::desc_lo(tc::smem_u32(s.a[0][0]));
    const uint32_t b_lo0 = tc::desc_lo(tc::smem_u32(s.b[0]));
    uint32_t ast = 0, aph = 0, bst = 0, bph = 0;
    for (int jj = 0; jj < my_jobs; ++jj) {
      const int buf = jj & 1;
      if (jj >= 2) {      // the epilogue must have drained this accumulator (job jj-2)
        CWAIT(CW_ACCFREE, &s.acc_free[buf], ((jj >> 1) - 1) & 1);
        tc::tc_fence_after_sync();
      }
      const uint32_t d = tmem + (uint32_t)buf * 128u;
      for (int t = 0; t < nsl; ++t) {
        CWAIT(CW_AFULL, &s.afull[ast], aph);
        CWAIT(CW_BFULL, &s.bfull[bst], bph);
        tc::tc_fence_after_sync();
        const uint32_t a_hi = a_lo0 + ast * ((2 * CT_A_HALF) >> 4), a_lo = a_hi + (CT_A_HALF >> 4);
        const uint32_t b_hi = b_lo0 + bst * (CT_B_STAGE >> 4), b_lo = b_hi + (CT_B_TILE >> 4);
        if (tc::elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k) tc::mma_cg1_lo(d, a_hi + 2u * k, b_hi + 2u * k, idesc, (t | k) ? 1u : 0u);
#pragma unroll
          for (int k = 0; k < 4; ++k) tc::mma_cg1_lo(d, a_lo + 2u * k, b_hi + 2u * k, idesc, 1u);
#pragma unroll
          for (int k = 0; k < 4; ++k) tc::mma_cg1_lo(d, a_hi + 2u * k, b_lo + 2u * k, idesc, 1u);
          tc::commit_cg1(&s.aempty[ast]);
          tc::commit_cg1(&s.bempty[bst]);
        }
        __syncwarp();
        if (++ast == CT_NA) { ast = 0; aph ^= 1u; }
        if (++bst == CT_NB) { bst = 0; bph ^= 1u; }
      }
      if (tc::elect_one()) tc::commit_cg1(&s.acc_full[buf]);
      __syncwarp();
    }
  } else if (warp >= 4 && warp < 8) {
    // ===================== epilogue =====================
    const int ew = warp - 4;
    const int row = ew * 32 + lane;
    for (int jj = 0; jj < my_jobs; ++jj) {
      int mt, nb, sp;
      decode((int)blockIdx.x + jj * (int)gridDim.x, mt, nb, sp);
      const int buf = jj & 1;
      CWAIT(CW_ACCFULL, &s.acc_full[buf], (jj >> 1) & 1);
      tc::tc_fence_after_sync();
      const int m = mt * 128 + row;
      const uint32_t taddr = tmem + ((uint32_t)(ew * 32) << 16) + (uint32_t)buf * 128u;
      float* dst = job.ws ? job.ws + ((size_t)sp * job.M + m) * job.N + (size_t)nb * 128
                          : job.C + (size_t)m * job.N + (size_t)nb * 128;
      for (int c0 = 0; c0 < 128; c0 += 32) {
        uint32_t r[32];
        tc::tmem_ld_x32(taddr + c0, r);
        tc::tmem_ld_wait();
        if (m < job.M && nb * 128 + c0 < job.N) {     // N is a multiple of 32; the padded columns are never stored
          const bool fin = !job.ws;                    // final values (bias, ReLU) or raw split-K partials
          const float4* bp = (fin && job.bias) ? reinterpret_cast<const float4*>(job.bias + nb * 128 + c0) : nullptr;
          const float lo = (fin && job.relu) ? 0.f : -INFINITY;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 b4 = bp ? __ldg(bp + (j >> 2)) : make_float4(0.f, 0.f, 0.f, 0.f);
            float4 o;
            o.x = fmaxf(__uint_as_float(r[j]) + b4.x, lo);
            o.y = fmaxf(__uint_as_float(r[j + 1]) + b4.y, lo);
            o.z = fmaxf(__uint_as_float(r[j + 2]) + b4.z, lo);
            o.w = fmaxf(__uint_as_float(r[j + 3]) + b4.w, lo);
            *reinterpret_cast<float4*>(dst + c0 + j) = o;
          }
        }
      }
      tc::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&s.acc_free[buf]);
    }
  } else if (warp >= 8) {
    // ===================== A producers: two groups of 4 warps, alternating slices =====================
    // Warp w of a group owns rows [32w, 32w+32) of the tile.  Loads are coalesced: in iteration j a half-warp reads the 256
    // contiguous bytes (64 channels of one filter tap) of one row -- lane l takes float4 (l & 15) of row 32w + 2j + (l >> 4).
    // The producers are latency bound (ncu: they sit on the first use of the loaded values), so the loop is software
    // pipelined in half-slices of 8 row pairs: while one half is converted to bf16 hi / lo and stored, the next half's 8
    // loads (the next slice's, possibly the next job's) are already in flight.
    const int grp = (warp - 8) >> 2;                 // 0 / 1
    const int w4 = (warp - 8) & 3;
    const int half = lane >> 4, f4 = lane & 15;      // row parity within the iteration, float4 index within the row
    // iterator over this group's slices (global slice counter parity == grp), across jobs
    int it_jj = 0, it_t = -1, it_sp = 0;
    uint32_t it_seq = 0xFFFFFFFFu;
    // rows of the iterator's current job: element offset of the row's own pixel (or matrix row) -- the per-slice part of the
    // address (tap offset, channel block) is the same for every row -- and, for the im2col view, a 9-bit mask per row of
    // the filter taps that fall inside the image (3 rows per word).  Round 1 recomputed coordinates, bounds and a 64-bit
    // product per load: ~40 instructions per LDG.128, which made the producers instruction bound.
    int64_t rbase[16];
    uint32_t rmask[6];
    auto load_job = [&](int jj) {
      int mt, nb, sp;
      decode((int)blockIdx.x + jj * (int)gridDim.x, mt, nb, sp);
      it_sp = sp;
#pragma unroll
      for (int k = 0; k < 6; ++k) rmask[k] = 0u;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int m = mt * 128 + w4 * 32 + 2 * j + half;
        rbase[j] = -1;
        if (m < job.M) {
          if (job.H > 0) {
            const int r = m % (job.H * job.W);
            const int y = r / job.W, x = r % job.W;
            rbase[j] = (int64_t)m * job.Cin;
            uint32_t mk = 0u;
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
              if (yy >= 0 && yy < job.H && xx >= 0 && xx < job.W) mk |= 1u << tap;
            }
            rmask[j / 3] |= mk << (9 * (j % 3));
          } else {
            rbase[j] = (int64_t)m * job.K;
          }
        }
      }
    };
    // advance to the next slice of this group; false when the work is exhausted
    auto advance = [&]() -> bool {
      while (true) {
        if (it_jj >= my_jobs) return false;
        ++it_t; ++it_seq;
        if (it_t >= nsl) { it_t = 0; ++it_jj; if (it_jj >= my_jobs) return false; load_job(it_jj); }
        if ((int)(it_seq & 1u) == grp) return true;
      }
    };
    auto issue = [&](float4* v, int b) {             // loads of half-slice b (row pairs 8b .. 8b+7) of the iterator's slice
      const int k0 = (it_sp * nsl + it_t) * 64;
      int tap = 0;
      int64_t soff = k0;                             // plain matrix: column offset
      if (job.H > 0) {
        tap = k0 / job.Cin;
        soff = (int64_t)((tap / 3 - 1) * job.W + (tap % 3 - 1)) * job.Cin + (k0 % job.Cin);
      }
      const float4* base = reinterpret_cast<const float4*>(job.A + soff) + f4;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int j = 8 * b + i;
        bool ok = rbase[j] >= 0;
        if (job.H > 0) ok = ok && ((rmask[j / 3] >> (9 * (j % 3) + tap)) & 1u);
        v[i] = ok ? __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + rbase[j]))
                  : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    auto store = [&](const float4* v, int b, int slot) {
      uint8_t* ahi = s.a[slot][0];
      uint8_t* alo = s.a[slot][1];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        uint32_t h0, h1, l0, l1;
        tc::split_bf16x2(v[i].x, v[i].y, h0, l0);
        tc::split_bf16x2(v[i].z, v[i].w, h1, l1);
        const uint32_t row = (uint32_t)(w4 * 32 + 2 * (8 * b + i) + half);
        const uint32_t off = tc::sw128_offset(row, (uint32_t)(f4 >> 1)) + (uint32_t)(f4 & 1) * 8u;
        *reinterpret_cast<uint2*>(ahi + off) = make_uint2(h0, h1);
        *reinterpret_cast<uint2*>(alo + off) = make_uint2(l0, l1);
      }
    };
    float4 va[8], vb[8];
    bool have = false;
    if (my_jobs > 0) { load_job(0); have = advance(); }
    if (have) issue(va, 0);
    while (have) {
      const uint32_t seq = it_seq;                   // the slice whose first half sits in `va`
      const int slot = (int)(seq & 3u);              // the consumer walks the ring in slice order
      issue(vb, 1);
      CWAIT(CW_AEMPTY, &s.aempty[slot], ((seq >> 2) & 1) ^ 1);
      store(va, 0, slot);
      have = advance();                              // may switch rpix / ryx to the next job: stores do not need them
      if (have) issue(va, 0);
      store(vb, 1, slot);
      tc::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&s.afull[slot]);
    }
  }
  if constexpr (kMeasure) {
    if (lane == 0 && dbg) {
      unsigned long long* o = dbg + ((size_t)blockIdx.x * 16 + warp) * (CW_NCLS + 1);
      for (int k = 0; k < CW_NCLS; ++k) o[k] = wt[k];
      o[CW_NCLS] = (unsigned long long)(clock64() - t_start);
    }
  }
  tc::tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc_cg1(tmem, 256);
#undef CWAIT
}

}  // namespace

// [K, N] fp32 row-major (device) -> packed B stage images [N/128][K/64][hi|lo][128 x 64 SW128 bf16] (device)
int conv_tc_pack(disn_ctx* c, const float* d_w, int K, int N, DevBuf& out) {
  std::vector<float> w((size_t)K * N);
  DISN_CUDA_OK(cudaMemcpyAsync(w.data(), d_w, w.size() * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  const int ns = K / 64, nbk = (N + 127) / 128;
  std::vector<uint8_t> img((size_t)nbk * ns * CT_B_STAGE, 0);   // rows beyond N stay zero
  for (int nb = 0; nb < nbk; ++nb)
    for (int t = 0; t < ns; ++t)
      for (int part = 0; part < 2; ++part) {
        uint8_t* dst = img.data() + ((size_t)nb * ns + t) * CT_B_STAGE + (size_t)part * CT_B_TILE;
        for (int nl = 0; nl < 128 && nb * 128 + nl < N; ++nl)
          for (int k = 0; k < 64; ++k) {
            const float v = w[(size_t)(t * 64 + k) * N + nb * 128 + nl];
            const __nv_bfloat16 hi = __float2bfloat16(v);
            const __nv_bfloat16 o = part == 0 ? hi : __float2bfloat16(v - __bfloat162float(hi));
            memcpy(dst + tc::sw128_offset(nl, k / 8) + (k % 8) * 2, &o, 2);
          }
      }
  // copy on the context's (non-blocking) stream and wait: a plain cudaMemcpy from pageable memory may return before
  // the DMA has landed and is not ordered against kernels on a non-blocking stream
  if (out.reserve(img.size())) return -1;
  DISN_CUDA_OK(cudaMemcpyAsync(out.get<void>(), img.data(), img.size(), cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}

// returns the number of K splits used (>= 1); when > 1 the caller reduces `ws` (splits x M x N) afterwards
int launch_conv_tc(disn_ctx* c, const float* A, const uint8_t* wpk, const float* bias, float* C, float* ws,
                   int64_t ws_elems, int M, int N, int K, int H, int W, int Cin, int relu, int* splits_out) {
  DISN_REQUIRE(K % 64 == 0 && N % 32 == 0 && (H == 0 || Cin % 64 == 0), "conv_tc: K%64, N%32, Cin%64");
  const int smem = (int)sizeof(ConvTcSmem) + 1024;
  if (!c->attr_conv_tc) {    // per context (= per device): the attribute is a property of the function ON a device
    DISN_CUDA_OK(cudaFuncSetAttribute(conv_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    DISN_CUDA_OK(cudaFuncSetAttribute(conv_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    c->attr_conv_tc = true;
  }
  const int sms = c->num_sms;
  ConvTcJob job{};
  job.A = A; job.wpk = wpk; job.bias = bias; job.C = C; job.M = M; job.N = N; job.K = K;
  job.H = H; job.W = W; job.Cin = Cin; job.relu = relu;
  job.m_tiles = (M + 127) / 128;
  job.n_blocks = (N + 127) / 128;
  const int slices = K / 64;
  int splits = 1;
  const int tiles = job.m_tiles * job.n_blocks;
  if (tiles < sms) {                     // under-filled: split K so that ~2 waves of jobs exist
    int want = (2 * sms + tiles - 1) / tiles;
    for (int d = std::min(want, slices); d >= 1; --d)
      if (slices % d == 0 && (int64_t)d * M * N <= ws_elems) { splits = d; break; }
  }
  job.splits = splits;
  job.slices_per_split = slices / splits;
  job.ws = splits > 1 ? ws : nullptr;
  const int total = tiles * splits;
  const int grid = std::min(total, sms);
  static const bool measure = getenv("DISN_CONV_MEASURE") != nullptr;
  if (!measure) {
    conv_tc_kernel<false><<<grid, CT_THREADS, smem, c->stream>>>(job, nullptr);
  } else {      // diagnostics: synchronous, prints the per-role blocked time of this launch
    const size_t n = (size_t)grid * 16 * (CW_NCLS + 1);
    DevBuf dbg;
    if (dbg.reserve(n * sizeof(unsigned long long))) return -1;
    DISN_CUDA_OK(cudaMemsetAsync(dbg.get<void>(), 0, n * sizeof(unsigned long long), c->stream));
    conv_tc_kernel<true><<<grid, CT_THREADS, smem, c->stream>>>(job, dbg.get<unsigned long long>());
    std::vector<unsigned long long> h(n);
    DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
    DISN_CUDA_OK(cudaMemcpy(h.data(), dbg.get<void>(), n * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    static const char* cls[CW_NCLS] = {"bempty", "accfree", "afull", "bfull", "accfull", "aempty"};
    static const int show[5] = {0, 1, 4, 8, 12};
    static const char* role[5] = {"Bprod", "MMA", "epi.q0", "Aprod.g0", "Aprod.g1"};
    double tot = 0;
    for (int b = 0; b < grid; ++b) tot += (double)h[((size_t)b * 16 + 1) * (CW_NCLS + 1) + CW_NCLS] / grid;
    fprintf(stderr, "[DISN_CONV_MEASURE] M=%d N=%d K=%d H=%d splits=%d jobs=%d grid=%d: %.0f cycles/CTA, tensor work %.0f cycles/CTA |",
            M, N, K, H, splits, total, grid, tot, (double)total / grid * job.slices_per_split * 768.0);
    for (int r = 0; r < 5; ++r) {
      fprintf(stderr, " %s{", role[r]);
      for (int k = 0; k < CW_NCLS; ++k) {
        double a = 0;
        for (int b = 0; b < grid; ++b) a += (double)h[((size_t)b * 16 + show[r]) * (CW_NCLS + 1) + k] / grid;
        if (a >= 0.02 * tot) fprintf(stderr, "%s=%.0f%% ", cls[k], 100.0 * a / tot);
      }
      fprintf(stderr, "}");
    }
    fprintf(stderr, "\n");
  }
  c->launches++;
  DISN_CUDA_OK(cudaGetLastError());
  *splits_out = splits;
  return 0;
}

}  // namespace disn
