// Fused per-point SDF kernel on tcgen05 tensor cores (DISN_PREC_BF16X3 / DISN_PREC_F16F8), sm_100a.
//
// Same math as point_fp32.cu (projection -> gather of the folded feature map -> two point-MLP streams
// -> sum; models/model_normalization.py:241-251,169-206, models/sdfnet.py:69-92,171-190), but the four
// wide layers of each stream run on the 5th-gen tensor cores.  To hold the reference's 1e-4 bar the fp32 operands
// are split (template parameter kMode, DESIGN.md section 3):
//   MODE_BF16X3  x = hi + lo (two bf16), each product = 3 kind::f16 MMAs (hi*hi + lo*hi + hi*lo), error ~2^-17;
//   MODE_F16F8   fp16 main product + e5m2 first-order correction products (kind::f8f6f4, twice the rate) into the
//                same fp32 accumulator in TMEM: both corrections (2 MMA-units per product instead of 3) in every layer
//                but fold2/conv1, which keeps one (1.5 units): 1.76 units per product overall.
//
// Organisation (one CTA pair = one cluster of 2, cta_group::2, UMMA M=128 x N=256 x K=16|32):
//   * a pair-tile is 128 query points, 64 per CTA (the 2x2 datapath keeps a 512-wide fp32 layer output
//     for 64 points in 256 TMEM columns, so one layer's input and output accumulators fit in TMEM);
//   * activations never leave the SM: layer l's accumulator is drained 32 columns at a time by the
//     epilogue warps (bias / folded image features, ReLU, operand split) into a 3-slot ring of
//     K-major swizzled A tiles that layer l+1's MMAs consume (K-outer), so MMA and epilogue pipeline; for the 512-wide
//     layers each N-block has its own "accumulator complete" barrier, so draining starts while the other block runs;
//     fold1/conv1 (3 -> 64, fp32 FMA) is staged into the same ring by epilogue group 0 from the points the front end
//     publishes, in the ring position the issue order needs (... X4_n, X2_{n+1}, X5_n, X3_{n+1} ...);
//   * the two streams are skewed by one layer: L0 of stream n+1 (one stage) is issued before L3 of stream n,
//     into the 128 TMEM columns that are free then (even/odd streams use mirrored column maps, acc_col()), so the next
//     stream's first drain overlaps this stream's last layer;
//   * weights are pre-split, pre-permuted and pre-swizzled on the host into the exact shared-memory images the
//     B operand needs (32 KB per (K-slice, N-block) and CTA), packed in consumption order, and streamed
//     by the bulk-copy engine (cp.async.bulk) through a 4-slot mbarrier ring; each CTA loads only its half of every
//     B tile; producers (warps 0 and 2) own fixed slots, never wait for the data and post the byte count after issuing
//     the copies; on the peer CTA warp 1 forwards "my half landed" to the leader;
//   * two MMA issuer warps on the leader CTA (warp 1: N-block 0 and all single-block layers, warp 3: N-block 1;
//     warp-uniform loops, one elected lane issues).  Their accumulators are disjoint, so the summation order and the
//     results stay bitwise deterministic.  One "stage landed" barrier per (issuer, slot): a stage's copies signal the
//     barrier of the issuer that will consume it (static stage -> issuer map), so every barrier is waited on, phase
//     after phase, by one agent only (a parity wait is meaningless for a waiter that skipped a phase; the protocol is
//     modelled in tools/tc_protocol_sim.py: x2_in_ring=1, NW=4, issuers=2, split_wfull=1);
//   * warps 4-11 epilogue in two groups taking alternate slices (one warp per TMEM lane quarter in each group),
//     warps 12-15 front end (points, projection, bilinear gather of the projected feature map into a shared-memory ring);
//   * the small per-stream parameters (biases, fold1/conv1, fold2/conv5) are a __grid_constant__ kernel parameter
//     (constant bank, warp-uniform indexed loads).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_fp16.h>
#include <cuda_fp8.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace disn {
namespace {

constexpr int NW = 4;                 // weight ring stages
constexpr int CORR_DEFAULT = 0xDF;    // correction mask of DISN_PREC_F16F8 (see kCorr below): every correction except the
                                      // a.(w - h(w)) product of fold2/conv1 -- measured on B200 (profiles/r02_corr_mask_sweep.txt)
#include "point_tc_shared.cuh"

constexpr int RING_PER_STREAM = 21;   // X3 (4) + X4 (8) + next stream's X2 (1) + X5 (8)

struct SmallParams { float v[2][SB_STRIDE]; };   // per stream: b2 b3 b4 b5 w6 w1 b1 at the SB_* offsets

struct TcSmem {
  alignas(1024) uint8_t w[NW][W_STAGE];
  alignas(1024) uint8_t x[NX][2][X_HALF];      // activation ring (all four tensor-core layers' A operands)
  float g[NG][64 * G_LD];                      // gathered image features [h*32+j][point]
  float px[2][PTS], py[2][PTS], pz[2][PTS];    // query points by tile parity
  int tap_off[2][PTS][4];
  float tap_w[2][PTS][4];
  float part[2][2][2][2][PTS];                 // [tile parity][stream][half][epilogue group][point]
  alignas(8) uint64_t wfull[2][NW];           // [consuming issuer][slot]   (peer CTA: only [0][slot], for the relay)
  uint64_t wempty[NW];
  uint64_t xfull[NX];
  uint64_t xempty[NX];
  uint64_t pfull[2];                           // points of tile parity published by the front end
  uint64_t gfull[NG];
  uint64_t gempty[NG];
  uint64_t acc_full[4][2];
  uint64_t acc5_free;
  uint32_t tmem_base;
};

// issuer (0/1) that consumes weight stage `g` of the consumption sequence (g = 0: first stream's L0; then the per-tile cycle
// G.L1(8) G.L2(16) L.L0(1) G.L3(8) L.L1(8) L.L2(16) G.L0(1) L.L3(8); the last tile has no G.L0 entry)
__device__ __forceinline__ void stage_info(uint32_t g, int my_tiles, uint32_t& img_stage, int& issuer) {
  img_stage = FIRST_L0_POS;
  issuer = 0;
  if (g == 0) return;
  const uint32_t cidx = g - 1, last0 = (uint32_t)(my_tiles - 1) * (2 * STAGES_PER_STREAM);
  uint32_t r = cidx % (2 * STAGES_PER_STREAM);
  if (cidx >= last0 && cidx - last0 >= (uint32_t)FIRST_L0_POS) r = cidx - last0 + 1;
  img_stage = r;
  if (r < 24) issuer = (int)(r & 1u);                    // G.L1, G.L2: N-blocks alternate
  else if (r >= 33 && r < 57) issuer = (int)((r - 33) & 1u);   // L.L1, L.L2
}

// position of an activation slice in the ring: kind 2 = fold1/conv1 output of stream sn, 3/4/5 = outputs of tensor-core
// layers 0/1/2 of stream sn (tools/tc_protocol_sim.py: seq_of)
__device__ __forceinline__ uint32_t ring_seq(int sn, int kind, int t, int nstreams) {
  if (kind == 2) return sn == 0 ? 0u : (uint32_t)(1 + RING_PER_STREAM * (sn - 1) + 12);
  const uint32_t base = 1u + (uint32_t)RING_PER_STREAM * (uint32_t)sn;
  if (kind == 5) return base + 12u + (sn + 1 < nstreams ? 1u : 0u) + (uint32_t)t;
  return base + (kind == 3 ? 0u : 4u) + (uint32_t)t;
}

// kVar bit 0: measurement build -- `expt` masks MMA groups (1 main product, 2 first correction, 4 second correction) and
//             every CTA reports its cycle count (DISN_TC_MEASURE=1 [DISN_TC_EXPT=<mask>]; masked results are wrong by
//             construction).  The product build carries none of it.
// kCorr (MODE_F16F8): which correction products each tensor layer keeps -- bit 2l: (a - h(a)).w ("first"), bit 2l+1:
//             a.(w - h(w)) ("second") for tensor layer l = 0..3 (fold1/conv2, fold1/conv3, fold2/conv1, fold2/conv2).  A dropped
//             correction saves its MMAs, its 8 KB weight tile per stage (not copied) and its e5m2 A tile (not produced by
//             the epilogue).  0xFF = every correction (2 bf16-rate units per product); the shipped mask is CORR_DEFAULT.
#define WAIT(bar, par) tc::mbar_wait(bar, par)
// measurement build: cycles this thread spends blocked, by barrier class (see the report in launch_var)
#define TWAIT(cls, bar, par)                                           \
  do {                                                                 \
    if constexpr ((kVar & 1) != 0) {                                   \
      const long long _t = clock64();                                  \
      tc::mbar_wait(bar, par);                                         \
      wt[cls] += (unsigned long long)(clock64() - _t);                 \
    } else {                                                           \
      tc::mbar_wait(bar, par);                                         \
    }                                                                  \
  } while (0)
enum { W_WEMPTY = 0, W_RELAY, W_ACC5, W_XFULL, W_WFULL, W_PFULL, W_XEMPTY, W_ACCFULL, W_GFULL, W_GEMPTY, W_NCLS };
// tensor layer of a weight stage from its position in the per-tile consumption cycle
//   G.L1 0..7 | G.L2 8..23 | L.L0 24 | G.L3 25..32 | L.L1 33..40 | L.L2 41..56 | G.L0 57 | L.L3 58..65
__host__ __device__ constexpr int stage_layer(uint32_t r) {
  return r < 8 ? 1 : r < 24 ? 2 : r == 24 ? 0 : r < 33 ? 3 : r < 41 ? 1 : r < 57 ? 2 : r == 57 ? 0 : 3;
}
template <int kMode, int kVar, int kCorr>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
point_tc_kernel(PointJob job, const __grid_constant__ SmallParams sp, const uint8_t* __restrict__ wpk,
                 int64_t tiles_per_img, unsigned long long* __restrict__ dbg, int expt) {
  extern __shared__ uint8_t smem_raw[];
  TcSmem& s = *reinterpret_cast<TcSmem*>(smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u));
  const uint32_t cta = tc::cluster_ctarank();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tid = threadIdx.x;
  constexpr int kC = (kMode == MODE_F16F8) ? kCorr : 0xFF;      // bf16x3 has no droppable products
  auto keep1 = [](int layer) { return ((kC >> (2 * layer)) & 1) != 0; };
  auto keep2 = [](int layer) { return ((kC >> (2 * layer + 1)) & 1) != 0; };
  const int num_pairs = gridDim.x >> 1, pair = blockIdx.x >> 1;
  const int64_t total_tiles = tiles_per_img * job.B;
  const int my_tiles = (pair < total_tiles) ? (int)((total_tiles - pair + num_pairs - 1) / num_pairs) : 0;
  const int nstreams = 2 * my_tiles;
  const uint32_t total_stages = (uint32_t)my_tiles * (2 * STAGES_PER_STREAM);

  if (tid == 0) {
    for (int i = 0; i < NW; ++i) {
      // leader: {its producer's expect_tx arrival, the peer relay's arrival}; peer: {its producer's expect_tx arrival}
      tc::mbar_init(&s.wfull[0][i], cta == 0 ? 2 : 1);
      tc::mbar_init(&s.wfull[1][i], cta == 0 ? 2 : 1);
      tc::mbar_init(&s.wempty[i], 1);
    }
    for (int i = 0; i < NX; ++i) { tc::mbar_init(&s.xfull[i], 8); tc::mbar_init(&s.xempty[i], 2); }
    tc::mbar_init(&s.pfull[0], 1);
    tc::mbar_init(&s.pfull[1], 1);
    for (int i = 0; i < NG; ++i) { tc::mbar_init(&s.gfull[i], 4); tc::mbar_init(&s.gempty[i], 4); }
    for (int i = 0; i < 4; ++i) { tc::mbar_init(&s.acc_full[i][0], 1); tc::mbar_init(&s.acc_full[i][1], 1); }
    tc::mbar_init(&s.acc5_free, 16);
    tc::fence_barrier_init();
  }
  __syncthreads();
  if (warp == 2) {
    tc::tmem_alloc_cg2(&s.tmem_base, 512);
    tc::tmem_relinquish_cg2();
  }
  tc::tc_fence_before_sync();
  tc::cluster_sync();
  tc::tc_fence_after_sync();
  const uint32_t tmem = s.tmem_base;
  const long long t_start = (kVar & 1) ? clock64() : 0;
  unsigned long long wt[W_NCLS] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};     // measurement build only

  if (warp == 0 || warp == 2) {
    // ===================== weight producers: warp 0 = even stages (slots 0, 2), warp 2 = odd stages (slots 1, 3) ==========
    const uint32_t pw = (warp == 0) ? 0u : 1u;
    if (lane < 2) {          // two lanes issue one 16 KB tile each so the copies overlap
      for (uint32_t g = pw; g < total_stages; g += 2) {
        const uint32_t slot = g % NW, use = g / NW;
        TWAIT(W_WEMPTY, &s.wempty[slot], (use & 1) ^ 1);
        uint32_t img_stage;
        int issuer;
        stage_info(g, my_tiles, img_stage, issuer);
        uint64_t* bar = &s.wfull[cta == 0 ? issuer : 0][slot];
        const uint8_t* src = wpk + (size_t)img_stage * (2 * W_STAGE) + (size_t)cta * W_STAGE + (size_t)lane * W_TILE;
        // lane 0: the main tile; lane 1: the e5m2 tiles of the corrections this layer keeps ([e5m2 w | e5m2 residual of w])
        const int sl = stage_layer(img_stage);
        const bool k1 = keep1(sl), k2 = keep2(sl);
        // measurement build, expt bit 3: copy a quarter of every tile (results invalid) -- is the kernel L2-bandwidth bound?
        const uint32_t shr = ((kVar & 1) && (expt & 8)) ? 2u : 0u;
        if (lane == 0) tc::bulk_g2s(s.w[slot], src, W_TILE >> shr, bar);
        else if (k1 || k2)
          tc::bulk_g2s(s.w[slot] + W_TILE + (k1 ? 0 : W8_TILE), src + (k1 ? 0 : W8_TILE), ((k1 && k2) ? W_TILE : W8_TILE) >> shr, bar);
        // the byte count may be posted after the copies: the phase cannot complete before this arrival
        if (lane == 0) tc::mbar_arrive_expect_tx(bar, (W_TILE + (k1 ? W8_TILE : 0) + (k2 ? W8_TILE : 0)) >> shr);
        __syncwarp(0x3);
      }
    }
  } else if (warp == 1 && cta == 1) {
    // ===================== peer CTA: forward "my half of the stage has landed" to the consuming issuer's barrier ==========
    if (lane == 0) {
      for (uint32_t g = 0; g < total_stages; ++g) {
        const uint32_t slot = g % NW;
        uint32_t img_stage;
        int issuer;
        stage_info(g, my_tiles, img_stage, issuer);
        TWAIT(W_RELAY, &s.wfull[0][slot], (g / NW) & 1);
        tc::mbar_arrive_cluster(&s.wfull[issuer][slot], 0);
      }
    }
  } else if (warp == 1 || warp == 3) {
    if (cta == 0) {
      // ===================== MMA issuers (leader CTA): warp 1 = N-block 0 + single-block layers, warp 3 = N-block 1 =========
      // Warp-uniform loop, one elected lane issues.  Both issuers wait for every activation slice (that keeps them within
      // one ring of each other and orders their TMEM writes after the epilogue's reads) and both release it (xempty = 2).
      const int which = (warp == 3) ? 1 : 0;
      const uint32_t idesc = (kMode == MODE_BF16X3) ? tc::make_idesc_bf16(128, 256) : tc::make_idesc_f16(128, 256);
      const uint32_t idesc8 = tc::make_idesc_e5m2(128, 256);
      const uint32_t w_lo0 = tc::desc_lo(tc::smem_u32(s.w[0]));
      const uint32_t x_lo0 = tc::desc_lo(tc::smem_u32(s.x[0][0]));
      uint32_t g = 0;                       // weight stage counter (consumption order, all stages of both issuers)
      uint32_t wuse[NW] = {0, 0, 0, 0};    // this issuer's uses of each slot so far (phase of its own barrier)
      uint32_t xsl = 0, xph = 0;            // activation ring slot / phase parity
      for (int grp = -1; grp < nstreams; ++grp) {
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
          const int layer = (q == 0) ? 1 : (q == 1 ? 2 : (q == 2 ? 0 : 3));
          const int sn = (q == 2) ? grp + 1 : grp;
          if (sn < 0 || sn >= nstreams) continue;
          const int sidx = sn & 1;
          const int nsl = (layer == 0) ? 1 : (layer == 1 ? 4 : 8);
          const int nnb = (layer == 1 || layer == 2) ? 2 : 1;
          const uint32_t colbase = acc_col(layer, sidx);
          if (layer == 2 && sn > 0) {        // acc4 overwrites the columns the previous stream's acc5 used
            TWAIT(W_ACC5, &s.acc5_free, (uint32_t)(sn - 1) & 1);
            tc::tc_fence_after_sync();
          }
#pragma unroll 1
          for (int t = 0; t < nsl; ++t) {
            const uint32_t slot = xsl;
            TWAIT(W_XFULL, &s.xfull[slot], xph);
            tc::tc_fence_after_sync();
            const uint32_t a_hi = x_lo0 + slot * ((2 * X_HALF) >> 4);
            const uint32_t a_lo = a_hi + (X_HALF >> 4);
            const int nb = (nnb == 2) ? which : 0;
            const bool mine = (nnb == 2) || which == 0;
            if (mine) {
              const uint32_t st = (g + (uint32_t)nb) % NW;
              TWAIT(W_WFULL, &s.wfull[which][st], wuse[st] & 1);
              ++wuse[st];
              tc::tc_fence_after_sync();
              const uint32_t d = tmem + colbase + (uint32_t)nb * 128u;
              const uint32_t b_hi = w_lo0 + st * (W_STAGE >> 4);
              const uint32_t b_lo = b_hi + (W_TILE >> 4);
              if (tc::elect_one()) {
                if constexpr (kMode == MODE_BF16X3) {
#pragma unroll
                  for (int k = 0; k < 4; ++k) tc::mma_cg2_lo(d, a_hi + 2u * k, b_hi + 2u * k, idesc, (t | k) ? 1u : 0u);
#pragma unroll
                  for (int k = 0; k < 4; ++k) tc::mma_cg2_lo(d, a_lo + 2u * k, b_hi + 2u * k, idesc, 1u);
#pragma unroll
                  for (int k = 0; k < 4; ++k) tc::mma_cg2_lo(d, a_hi + 2u * k, b_lo + 2u * k, idesc, 1u);
                } else {
                  const bool x0 = !(kVar & 1) || !(expt & 1), x1 = !(kVar & 1) || !(expt & 2), x2 = !(kVar & 1) || !(expt & 4);
                  if (x0) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) tc::mma_cg2_lo(d, a_hi + 2u * k, b_hi + 2u * k, idesc, (t | k) ? 1u : 0u);
                  }
                  if (x1 && keep1(layer)) {
#pragma unroll
                    for (int k = 0; k < 2; ++k) tc::mma_cg2_f8_lo(d, a_lo + 2u * k, b_lo + 2u * k, idesc8, 1u);
                  }
                  if (x2 && keep2(layer)) {
#pragma unroll
                    for (int k = 0; k < 2; ++k)
                      tc::mma_cg2_f8_lo(d, a_lo + (X8_TILE >> 4) + 2u * k, b_lo + (W8_TILE >> 4) + 2u * k, idesc8, 1u);
                  }
                }
                tc::commit_cg2(&s.wempty[st], 0b11);
                if (t == nsl - 1) tc::commit_cg2(&s.acc_full[layer][nb], 0b11);
                tc::commit_cg2(&s.xempty[slot], 0b11);     // second arrival comes from the other issuer
              }
            } else {
              // single-block layer, issuer 1: nothing to issue; its arrival only completes the slice's release count
              if (tc::elect_one()) tc::commit_cg2(&s.xempty[slot], 0b11);
            }
            g += (uint32_t)nnb;
            if (++xsl == NX) { xsl = 0; xph ^= 1u; }
          }
        }
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ===================== epilogue: TMEM -> bias/ReLU/split -> activation ring (two groups, alternate slices) ==========
    const int eg = (warp >= 8) ? 1 : 0;
    const int ew = warp & 3;
    const int row = ew * 32 + lane;
    const int p = row & 63, h = row >> 6;
    const uint32_t tlane = tmem + ((uint32_t)(ew * 32) << 16);
    uint32_t gseq = 0;
    __half2 amax = __float2half2_rn(0.f);   // running maximum of this thread's fp16 A-operand values (MODE_F16F8)

    auto arrive_xfull = [&](int slot) {
      tc::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        if (cta == 0) tc::mbar_arrive(&s.xfull[slot]);
        else tc::mbar_arrive_cluster(&s.xfull[slot], 0);
      }
    };
    // fold1/conv1 (3 -> 64, fp32 FMA) of stream sn from the published points -> its ring slice (group 0 only)
    auto stage_first = [&](int sn) {
      const int tile = sn >> 1, sx = sn & 1;
      const uint32_t seq = ring_seq(sn, 2, 0, nstreams);
      const int slot = (int)(seq % NX);
      TWAIT(W_PFULL, &s.pfull[tile & 1], (uint32_t)(tile >> 1) & 1);
      const float x = s.px[tile & 1][p], y = s.py[tile & 1][p], z = s.pz[tile & 1][p];
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int f = h * 32 + j;
        float a = sp.v[sx][SB_B1 + f];
        a = fmaf(x, sp.v[sx][SB_W1 + f], a);
        a = fmaf(y, sp.v[sx][SB_W1 + 64 + f], a);
        a = fmaf(z, sp.v[sx][SB_W1 + 128 + f], a);
        v[j] = fmaxf(a, 0.f);
      }
      TWAIT(W_XEMPTY, &s.xempty[slot], ((seq / NX) & 1) ^ 1);
      store_slice<kMode>(s.x[slot][0], s.x[slot][1], p, h, v, job.act_scale[sx][0][0], job.act_scale[sx][0][1], amax, keep1(0), keep2(0));
      arrive_xfull(slot);
    };
    // drain thread-columns [32t, 32t+32) of the accumulator at `col0` into ring slice `seq`; the bias comes from the
    // parameter table (sb_off, stream sx) or, for the global stream's fold2/conv1, from the per-image folded bias in HBM
    auto drain = [&](uint32_t col0, int t, int sx, int sb_off, const float* gbias, uint32_t seq, bool gather, float sc_lo,
                     float sc_hi, uint64_t* accbar, uint32_t accpar, int next_layer) {
      const int slot = (int)(seq % NX);
      if (accbar) {
        TWAIT(W_ACCFULL, accbar, accpar);
        tc::tc_fence_after_sync();
      }
      uint32_t r[32];
      tc::tmem_ld_x32(tlane + col0 + 32u * t, r);
      const int f0 = fout(h, 32 * t);
      float v[32];
      if (gbias) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 bq = *reinterpret_cast<const float4*>(gbias + f0 + j);
          v[j] = bq.x; v[j + 1] = bq.y; v[j + 2] = bq.z; v[j + 3] = bq.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = sp.v[sx][sb_off + f0 + j];
      }
      const int gs = t & (NG - 1);           // gather slice t lives in ring slot t % NG (= this group's parity)
      if (gather) {
        TWAIT(W_GFULL, &s.gfull[gs], gseq & 1);
        const float* gp = s.g[gs] + (h * 32) * G_LD + p;
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += gp[j * G_LD];
        ++gseq;
      }
      tc::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = fmaxf(__uint_as_float(r[j]) + v[j], 0.f);
      TWAIT(W_XEMPTY, &s.xempty[slot], ((seq / NX) & 1) ^ 1);
      store_slice<kMode>(s.x[slot][0], s.x[slot][1], p, h, v, sc_lo, sc_hi, amax, keep1(next_layer), keep2(next_layer));
      arrive_xfull(slot);
      if (gather && lane == 0) tc::mbar_arrive(&s.gempty[gs]);
    };
    auto drain_x3 = [&](int sn) {
      const int sx = sn & 1;
      for (int t = eg; t < 4; t += 2)
        drain(acc_col(0, sx), t, sx, SB_B2, nullptr, ring_seq(sn, 3, t, nstreams), false, job.act_scale[sx][1][0],
              job.act_scale[sx][1][1], t == eg ? &s.acc_full[0][0] : nullptr, (uint32_t)sn & 1, 1);
    };

    // ring order: X2_0, then per stream n: X3_n (4), X4_n (8), X2_{n+1}, X5_n (8); X3_{n+1} before stream n's final layer
    if (nstreams > 0) {
      if (eg == 0) stage_first(0);
      drain_x3(0);
    }
    for (int sn = 0; sn < nstreams; ++sn) {
      const int sidx = sn & 1, it = sn >> 1;
      const TileCoord tc0 = tile_coord((int64_t)pair + (int64_t)it * num_pairs, tiles_per_img);
      const uint32_t par = (uint32_t)sn & 1;
      for (int t = eg; t < 8; t += 2)
        drain(acc_col(1, sidx), t, sidx, SB_B3, nullptr, ring_seq(sn, 4, t, nstreams), false, job.act_scale[sidx][2][0],
              job.act_scale[sidx][2][1], t == eg ? &s.acc_full[1][0] : (t == eg + 4 ? &s.acc_full[1][1] : nullptr), par, 2);
      if (eg == 0 && sn + 1 < nstreams) stage_first(sn + 1);
      const float* gb = sidx ? nullptr : (job.gbias + (int64_t)tc0.b * kHidden);
      for (int t = eg; t < 8; t += 2)
        drain(acc_col(2, sidx), t, sidx, SB_B4, gb, ring_seq(sn, 5, t, nstreams), sidx == 1, job.act_scale[sidx][3][0],
              job.act_scale[sidx][3][1], t == eg ? &s.acc_full[2][0] : (t == eg + 4 ? &s.acc_full[2][1] : nullptr), par, 3);
      if (sn + 1 < nstreams) drain_x3(sn + 1);
      // fold2/conv2 output (256) -> ReLU -> fold2/conv5 dot product
      TWAIT(W_ACCFULL, &s.acc_full[3][0], par);
      tc::tc_fence_after_sync();
      float part = 0.f;
      for (int t = 2 * eg; t < 2 * eg + 2; ++t) {
        uint32_t r[32];
        tc::tmem_ld_x32(tlane + acc_col(3, sidx) + 32u * t, r);
        const int f0 = fout(h, 32 * t);
        tc::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float a = fmaxf(__uint_as_float(r[j]) + sp.v[sidx][SB_B5 + f0 + j], 0.f);
          part = fmaf(a, sp.v[sidx][SB_W6 + f0 + j], part);
        }
      }
      tc::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) {
        if (cta == 0) tc::mbar_arrive(&s.acc5_free);
        else tc::mbar_arrive_cluster(&s.acc5_free, 0);
      }
      s.part[it & 1][sidx][h][eg][p] = part;
      if (sidx == 0) continue;
      named_bar_sync(1, 256);
      if (h == 0 && eg == 0) {
        const int64_t n = tc0.n0 + (int64_t)cta * PTS + p;
        if (n < job.N) {
          const float (*pp)[2][2][PTS] = s.part[it & 1];
          float rg = ((pp[0][0][0][p] + pp[0][0][1][p]) + (pp[0][1][0][p] + pp[0][1][1][p])) + __ldg(job.g.b6);
          float rl = ((pp[1][0][0][p] + pp[1][0][1][p]) + (pp[1][1][0][p] + pp[1][1][1][p])) + __ldg(job.l.b6);
          if (job.out_global) job.out_global[(int64_t)tc0.b * job.N + n] = rg;
          if (job.out_local) job.out_local[(int64_t)tc0.b * job.N + n] = rl;
          float r = rg + rl;
          if (job.tanh_out) r = tanhf(r);
          job.out_pred[(int64_t)tc0.b * job.N + n] = __fdiv_rn(r, job.out_div);
        }
      }
    }
    if constexpr (kMode == MODE_F16F8) {
      // fp16 range guard: +inf here means an activation exceeded 65504 and the result is meaningless
      if ((__hisinf(__low2half(amax)) || __hisinf(__high2half(amax))) && job.status) atomicOr(job.status, DISN_STATUS_FP16_OVERFLOW);
    }
  } else if (warp >= 12) {
    // ===================== front end: points, projection, taps (published per tile), feature gather =====================
    const int ft = tid - 384;
    const int fw = warp - 12;
    const int Wm = job.img_w, Hm = job.img_h;

    auto compute_points = [&](int it) {
      const TileCoord tc0 = tile_coord((int64_t)pair + (int64_t)it * num_pairs, tiles_per_img);
      const int b = tc0.b;
      const int pb = it & 1;
      named_bar_sync(2, 128);          // every front-end thread is done with this parity's previous contents
      if (ft < PTS) {
        const int64_t n = tc0.n0 + (int64_t)cta * PTS + ft;
        float x = 0.f, y = 0.f, z = 0.f, xr = 0.f, yr = 0.f, zr = 0.f;
        if (n < job.N) {
          if (job.pts) {
            const float* q = job.pts + ((int64_t)b * job.N + n) * 3;
            x = q[0]; y = q[1]; z = q[2];
            if (job.pts_rot) {
              const float* r = job.pts_rot + ((int64_t)b * job.N + n) * 3;
              xr = r[0]; yr = r[1]; zr = r[2];
            } else { xr = x; yr = y; zr = z; }
          } else {
            const int R = job.R;
            const int ix = (int)(n % R);
            const int64_t tt = n / R;
            const int iy = (int)(tt % R);
            const int iz = (int)(tt / R) + job.z0;
            const float* ax = job.axes + (int64_t)b * 3 * R;
            x = ax[ix]; y = ax[R + iy]; z = ax[2 * R + iz];
            xr = x; yr = y; zr = z;
          }
        }
        const float* T = job.trans_mat + b * 12;
        const float q0 = fmaf(z, T[6], fmaf(y, T[3], x * T[0])) + T[9];
        const float q1 = fmaf(z, T[7], fmaf(y, T[4], x * T[1])) + T[10];
        const float q2 = fmaf(z, T[8], fmaf(y, T[5], x * T[2])) + T[11];
        const float u = fminf(job.clamp_max, fmaxf(0.f, q0 / q2));
        const float v = fminf(job.clamp_max, fmaxf(0.f, q1 / q2));
        s.px[pb][ft] = xr; s.py[pb][ft] = yr; s.pz[pb][ft] = zr;
        if (job.out_uv && n < job.N) {
          float* o = job.out_uv + ((int64_t)b * job.N + n) * 2;
          o[0] = u; o[1] = v;
        }
        int off[4] = {-1, -1, -1, -1};
        float wg[4] = {0.f, 0.f, 0.f, 0.f};
        if (job.pfeat) {        // explicit per-point features: one "tap" of weight 1 at this point's row of pfeat
          if (n < job.N) { off[0] = (int)(((int64_t)b * job.N + n) * kHidden); wg[0] = 1.f; }
        } else if (u > -1.f && v > -1.f && u < (float)Wm && v < (float)Hm) {
          const int fx = (int)floorf(u), fy = (int)floorf(v);
          const int cx = fx + 1, cy = fy + 1;
          const float dx = (float)cx - u, dy = (float)cy - v;
          const int tx[4] = {fx, cx, fx, cx}, ty[4] = {fy, cy, cy, fy};
          const float ww[4] = {dx * dy, (1.f - dx) * (1.f - dy), dx * (1.f - dy), (1.f - dx) * dy};
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (tx[k] >= 0 && tx[k] < Wm && ty[k] >= 0 && ty[k] < Hm) {
              off[k] = (ty[k] * Wm + tx[k]) * kHidden;
              wg[k] = ww[k];
            }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) { s.tap_off[pb][ft][k] = off[k]; s.tap_w[pb][ft][k] = wg[k]; }
      }
      named_bar_sync(2, 128);
      if (ft == 0) tc::mbar_arrive(&s.pfull[pb]);      // epilogue group 0 computes fold1/conv1 from these points
    };

    // the next tile's points are published before this tile's gather: the epilogue stages stream n+1's first slice while
    // stream n is still in its last layers
    if (my_tiles > 0) compute_points(0);
    for (int it = 0; it < my_tiles; ++it) {
      const TileCoord tc0 = tile_coord((int64_t)pair + (int64_t)it * num_pairs, tiles_per_img);
      const int b = tc0.b;
      const int pb = it & 1;
      if (it + 1 < my_tiles) compute_points(it + 1);
      const float* pm = job.pfeat ? job.pfeat : job.pmap + (int64_t)b * Hm * Wm * kHidden;
      const int grp = lane >> 3, q = lane & 7;
      const bool pf = (job.pts == nullptr);
      auto prefetch_slice = [&](int t) {
        const int ppt = fw * 16 + (lane >> 1), phh = lane & 1;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int off = s.tap_off[pb][ppt][k];
          if (off >= 0) tc::prefetch_l1(pm + off + fout(phh, 32 * t));
        }
      };
      if (pf) prefetch_slice(0);
      for (int t = 0; t < 8; ++t) {
        const uint32_t gsq = (uint32_t)it * 8 + t;
        const int gs = gsq % NG;
        if (pf && t + 1 < 8) prefetch_slice(t + 1);
        TWAIT(W_GEMPTY, &s.gempty[gs], ((gsq / NG) & 1) ^ 1);
        float* gdst = s.g[gs];
#pragma unroll
        for (int i2 = 0; i2 < 4; i2 += 2) {       // two point groups at a time: 16 x 16 B loads in flight per lane
          float4 m[2][2][4];
          float wg[2][4];
          int pts[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int pt = fw * 16 + (i2 + u) * 4 + grp;
            pts[u] = pt;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int off = s.tap_off[pb][pt][k];
              wg[u][k] = s.tap_w[pb][pt][k];          // zero for taps outside the map
              const float* src = pm + (off >= 0 ? off : 0);
#pragma unroll
              for (int hh = 0; hh < 2; ++hh)
                m[u][hh][k] = __ldg(reinterpret_cast<const float4*>(src + fout(hh, 32 * t) + q * 4));
            }
          }
#pragma unroll
          for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                a.x = fmaf(wg[u][k], m[u][hh][k].x, a.x); a.y = fmaf(wg[u][k], m[u][hh][k].y, a.y);
                a.z = fmaf(wg[u][k], m[u][hh][k].z, a.z); a.w = fmaf(wg[u][k], m[u][hh][k].w, a.w);
              }
              float* d = gdst + (hh * 32 + q * 4) * G_LD + pts[u];
              d[0] = a.x; d[G_LD] = a.y; d[2 * G_LD] = a.z; d[3 * G_LD] = a.w;
            }
        }
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&s.gfull[gs]);
      }
    }
  }

  // ---- teardown ----
  tc::tc_fence_before_sync();
  tc::cluster_sync();
  if ((kVar & 1) && dbg) {
    if (threadIdx.x == 0) dbg[blockIdx.x] = (unsigned long long)(clock64() - t_start);
    if (lane == 0) {
      unsigned long long* o = dbg + gridDim.x + ((size_t)blockIdx.x * 16 + warp) * W_NCLS;
      for (int k = 0; k < W_NCLS; ++k) o[k] = wt[k];
    }
  }
  if (warp == 2) tc::tmem_dealloc_cg2(tmem, 512);
}

// K-slice t, position k (0..63) of a layer whose input activations have width `K` -> input feature index
inline int fin_of(int layer, int t, int k) {
  if (layer == 0) return k;                           // X2 is written in natural order
  const int c = 32 * t + (k % 32);
  return fout(k / 32, c);
}

template <int kMode, int kVar, int kCorr>
int launch_var(disn_ctx* c, const PointJob& job, const SmallParams& sp, const void* wpk, int pairs, int smem,
               int64_t tiles_per_img) {
  // the attribute belongs to (function, device): set per context, not per process (a second engine on another device
  // in the same process would otherwise launch with the 48 KB default)
  auto key = (const void*)point_tc_kernel<kMode, kVar, kCorr>;
  if (!c->attr_done.count(key)) {
    DISN_CUDA_OK(cudaFuncSetAttribute(point_tc_kernel<kMode, kVar, kCorr>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    c->attr_done.insert(key);
  }
  DevBuf dbg;
  int expt = 0;
  if constexpr ((kVar & 1) != 0) {
    expt = getenv("DISN_TC_EXPT") ? atoi(getenv("DISN_TC_EXPT")) : 0;
    if (dbg.reserve((size_t)pairs * 2 * (1 + 16 * W_NCLS) * sizeof(unsigned long long))) return -1;
    DISN_CUDA_OK(cudaMemsetAsync(dbg.get<void>(), 0, dbg.bytes(), c->stream));
  }
  point_tc_kernel<kMode, kVar, kCorr><<<pairs * 2, NTHREADS, smem, c->stream>>>(
      job, sp, reinterpret_cast<const uint8_t*>(wpk), tiles_per_img, dbg.get<unsigned long long>(), expt);
  if constexpr ((kVar & 1) != 0) {
    std::vector<unsigned long long> h((size_t)pairs * 2 * (1 + 16 * W_NCLS));
    DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
    DISN_CUDA_OK(cudaMemcpy(h.data(), dbg.get<void>(), h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    const int nc = pairs * 2;
    double sum = 0, mx = 0;
    for (int i = 0; i < nc; ++i) { sum += (double)h[i]; mx = std::max(mx, (double)h[i]); }
    const double tiles = (double)(tiles_per_img * job.B) / pairs;
    fprintf(stderr, "[DISN_TC_MEASURE expt=%d corr=0x%02x] CTA cycles: mean %.0f max %.0f  -> %.1f Kcycles per tile (%.1f tiles per pair)\n",
            expt, kCorr, sum / nc, mx, sum / nc / tiles / 1000.0, tiles);
    // blocked cycles per tile by role and barrier class (leader CTAs: even blocks; peer CTAs: odd blocks)
    static const char* cls[W_NCLS] = {"wempty", "relay", "acc5", "xfull", "wfull", "pfull", "xempty", "accfull", "gfull", "gempty"};
    static const char* role[16] = {"prod0", "issuer0/relay", "prod1", "issuer1", "epi0.q0", "epi0.q1", "epi0.q2", "epi0.q3", "epi1.q0",
                                   "epi1.q1", "epi1.q2", "epi1.q3", "front0", "front1", "front2", "front3"};
    for (int ctak = 0; ctak < 2; ++ctak)
      for (int w = 0; w < 16; ++w) {
        double acc[W_NCLS] = {0};
        for (int p = 0; p < pairs; ++p)
          for (int k = 0; k < W_NCLS; ++k) acc[k] += (double)h[(size_t)nc + ((size_t)(2 * p + ctak) * 16 + w) * W_NCLS + k] / pairs / tiles;
        std::string line;
        for (int k = 0; k < W_NCLS; ++k)
          if (acc[k] >= 50.0) { char b[64]; snprintf(b, sizeof b, " %s=%.0f", cls[k], acc[k]); line += b; }
        if (!line.empty()) fprintf(stderr, "[DISN_TC_MEASURE]   %s %-14s blocked cycles/tile:%s\n", ctak ? "peer  " : "leader", role[w], line.c_str());
      }
  }
  return 0;
}

}  // namespace

// Pack both streams' tensor-core layers into the kernel's B-operand stage images:
//   for stream, layer, slice t, N-block nb : CTA half c : part (hi, lo) : 16 KB [128 rows n][64 k] SW128 bf16
// first position of (stream kind, layer) in the per-tile weight consumption cycle of the MMA warp:
//   G.L1(8) G.L2(16) L.L0(1) G.L3(8) L.L1(8) L.L2(16) G.L0(1) L.L3(8)      (L0 of the next stream is issued before L3)
static const int kCyclePos[2][4] = {{FIRST_L0_POS, 0, 8, 25}, {24, 33, 41, 58}};

int tc_pack_weights(disn_ctx* c) {
  static const int Ks[4] = {64, 256, 512, 512}, Ns[4] = {256, 512, 512, 256};
  const size_t total = (size_t)2 * STAGES_PER_STREAM * 2 * W_STAGE;
  std::vector<uint8_t> img(total, 0);
  size_t stage = 0;
  for (int sidx = 0; sidx < 2; ++sidx) {
    const std::string p = sidx ? "sdfprediction_imgfeat" : "sdfprediction";
    const char* names[4] = {"/fold1/conv2/weights", "/fold1/conv3/weights", "/fold2/conv1/weights", "/fold2/conv2/weights"};
    for (int layer = 0; layer < 4; ++layer) {
      auto it = c->weights.find(p + names[layer]);
      DISN_REQUIRE(it != c->weights.end(), "missing variable " + p + names[layer]);
      const int K = Ks[layer], N = Ns[layer];
      std::vector<float> w((size_t)K * N);   // rows 0..K-1 of the [Cin,Cout] matrix (point-feature part)
      DISN_CUDA_OK(cudaMemcpyAsync(w.data(), it->second.data.get<float>(), w.size() * sizeof(float), cudaMemcpyDeviceToHost,
                                   c->stream));
      DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
      for (int t = 0; t < K / 64; ++t)
        for (int nb = 0; nb < N / 256; ++nb, ++stage)
          for (int part = 0; part < 2; ++part)
            for (int half = 0; half < 2; ++half) {
              const size_t pos = (size_t)kCyclePos[sidx][layer] + (size_t)(t * (N / 256) + nb);
              uint8_t* dst = img.data() + pos * (2 * W_STAGE) + (size_t)half * W_STAGE + (size_t)part * W_TILE;
              for (int nl = 0; nl < 128; ++nl) {
                const int n = nb * 256 + half * 128 + nl;
                for (int k = 0; k < 64; ++k) {
                  const float v = w[(size_t)fin_of(layer, t, k) * N + n];
                  const __nv_bfloat16 hi = __float2bfloat16(v);
                  const __nv_bfloat16 out = part == 0 ? hi : __float2bfloat16(v - __bfloat162float(hi));
                  memcpy(dst + tc::sw128_offset(nl, k / 8) + (k % 8) * 2, &out, 2);
                }
              }
            }
    }
  }
  DISN_REQUIRE(stage == (size_t)2 * STAGES_PER_STREAM, "internal: stage count");
  if (c->tc_weights.reserve(total) || c->tc_weights_f8.reserve(total)) return -1;
  DISN_CUDA_OK(cudaMemcpyAsync(c->tc_weights.get<void>(), img.data(), total, cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));   // ordered on the ctx stream (see conv_tc_pack)

  // ---- DISN_PREC_F16F8 images: per (stage, CTA half): [fp16 W, SW128, 16 KB | e5m2(w.2^-s1), SW64, 8 KB |
  //      e5m2((w - fp16(w)).2^s2), SW64, 8 KB].  The exponents follow the layer's weight rms (2^L) so that the
  //      e5m2 operands (normal range 2^-14 .. 2^15, 2 mantissa bits) sit mid-range for O(1) activations:
  //      s1 = 10 + L, s2 = 12 + L; the matching activation multipliers 2^s1 and 2^-s2 go to the kernel.
  std::fill(img.begin(), img.end(), 0);
  stage = 0;
  for (int sidx = 0; sidx < 2; ++sidx) {
    const std::string p = sidx ? "sdfprediction_imgfeat" : "sdfprediction";
    const char* names[4] = {"/fold1/conv2/weights", "/fold1/conv3/weights", "/fold2/conv1/weights", "/fold2/conv2/weights"};
    for (int layer = 0; layer < 4; ++layer) {
      auto it = c->weights.find(p + names[layer]);
      const int K = Ks[layer], N = Ns[layer];
      std::vector<float> w((size_t)K * N);
      DISN_CUDA_OK(cudaMemcpyAsync(w.data(), it->second.data.get<float>(), w.size() * sizeof(float), cudaMemcpyDeviceToHost,
                                   c->stream));
      DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
      double ss = 0;
      for (float v : w) ss += (double)v * v;
      const double rms = std::sqrt(ss / (double)w.size());
      const int L = rms > 0 ? (int)std::lround(std::log2(rms)) : -4;
      const int s1 = std::min(24, std::max(-8, 10 + L)), s2 = std::min(28, std::max(-8, 12 + L));
      c->tc_act_scale[sidx][layer][0] = std::ldexp(1.f, s1);
      c->tc_act_scale[sidx][layer][1] = std::ldexp(1.f, -s2);
      for (int t = 0; t < K / 64; ++t)
        for (int nb = 0; nb < N / 256; ++nb, ++stage)
          for (int half = 0; half < 2; ++half) {
            const size_t pos = (size_t)kCyclePos[sidx][layer] + (size_t)(t * (N / 256) + nb);
            uint8_t* dst = img.data() + pos * (2 * W_STAGE) + (size_t)half * W_STAGE;
            for (int nl = 0; nl < 128; ++nl) {
              const int n = nb * 256 + half * 128 + nl;
              for (int k = 0; k < 64; ++k) {
                const float v = w[(size_t)fin_of(layer, t, k) * N + n];
                const __half hv = __float2half_rn(v);
                memcpy(dst + tc::sw128_offset(nl, k / 8) + (k % 8) * 2, &hv, 2);
                const uint32_t o8 = tc::sw64_offset(nl, k / 16) + (k % 16);
                dst[W_TILE + o8] = (uint8_t)__nv_cvt_float_to_fp8(std::ldexp(v, -s1), __NV_SATFINITE, __NV_E5M2);
                dst[W_TILE + W8_TILE + o8] =
                    (uint8_t)__nv_cvt_float_to_fp8(std::ldexp(v - __half2float(hv), s2), __NV_SATFINITE, __NV_E5M2);
              }
            }
          }
    }
  }
  DISN_CUDA_OK(cudaMemcpyAsync(c->tc_weights_f8.get<void>(), img.data(), total, cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));

  // host copy of the small per-stream parameters at the SB_* offsets (the kernel's __grid_constant__ parameter table)
  for (int sidx = 0; sidx < 2; ++sidx) {
    const std::string p = sidx ? "sdfprediction_imgfeat" : "sdfprediction";
    const struct { const char* name; int off, n; } small[7] = {
        {"/fold1/conv2/biases", SB_B2, 256}, {"/fold1/conv3/biases", SB_B3, 512}, {"/fold2/conv1/biases", SB_B4, 512},
        {"/fold2/conv2/biases", SB_B5, 256}, {"/fold2/conv5/weights", SB_W6, 256}, {"/fold1/conv1/weights", SB_W1, 192},
        {"/fold1/conv1/biases", SB_B1, 64}};
    for (const auto& e : small) {
      auto it = c->weights.find(p + e.name);
      DISN_REQUIRE(it != c->weights.end() && it->second.numel == e.n, "missing or mis-shaped variable " + p + e.name);
      DISN_CUDA_OK(cudaMemcpyAsync(&c->tc_small[sidx][e.off], it->second.data.get<float>(), (size_t)e.n * sizeof(float),
                                   cudaMemcpyDeviceToHost, c->stream));
    }
  }
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}

int launch_point_tc(disn_ctx* c, const PointJob& job_in) {
  const bool f8 = c->cfg.precision == DISN_PREC_F16F8;
  const void* wpk = (f8 ? c->tc_weights_f8 : c->tc_weights).get<void>();
  DISN_REQUIRE(wpk != nullptr, "tensor-core weights not packed (call disn_finalize_weights)");
  static_assert(sizeof(SmallParams) == sizeof(c->tc_small), "small-parameter table layout");
  PointJob job = job_in;
  memcpy(job.act_scale, c->tc_act_scale, sizeof(job.act_scale));
  SmallParams sp;
  memcpy(&sp, c->tc_small, sizeof(sp));
  const int smem = (int)sizeof(TcSmem) + 1024;
  const int64_t tiles_per_img = (job.N + 2 * PTS - 1) / (2 * PTS);
  const int64_t total = tiles_per_img * job.B;
  if (total == 0) return 0;
  const int pairs = (int)std::min<int64_t>(total, c->num_sms / 2);
  const bool measure = getenv("DISN_TC_MEASURE") != nullptr;
  int corr = CORR_DEFAULT;
  if (const char* e = getenv("DISN_TC_CORR")) corr = (int)strtol(e, nullptr, 0);      // A/B: 0xFF = every correction
  int rc = -2;
  if (!f8) rc = measure ? launch_var<MODE_BF16X3, 1, 0xFF>(c, job, sp, wpk, pairs, smem, tiles_per_img)
                        : launch_var<MODE_BF16X3, 0, 0xFF>(c, job, sp, wpk, pairs, smem, tiles_per_img);
  else {
    switch (corr) {
#define DISN_CORR(m)                                                                                  \
  case m:                                                                                             \
    rc = measure ? launch_var<MODE_F16F8, 1, m>(c, job, sp, wpk, pairs, smem, tiles_per_img)           \
                 : launch_var<MODE_F16F8, 0, m>(c, job, sp, wpk, pairs, smem, tiles_per_img);          \
    break;
      DISN_CORR(0xFF) DISN_CORR(0xDF)
#undef DISN_CORR
      default: DISN_REQUIRE(false, "DISN_TC_CORR: only 0xFF (all corrections) and 0xDF (default) are built");
    }
  }
  if (rc) return rc;
  c->launches++;
  DISN_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace disn
