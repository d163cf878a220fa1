// Image encoder of the DISN hot path, fp32 CUDA-core implementation for sm_100a.
//
// Restates (not ports) models/model_normalization.py:65-77 (137->224 legacy bilinear resize, vgg_16 with
// num_classes=1024, is_training=False) and the per-image part of :171-190 after two exact algebraic folds
// (SURVEY.md 7): the global embedding enters fold2/conv1 of the global stream as a per-image bias, and the
// five VGG taps are projected through fold2/conv1 of the local stream at native resolution and then
// bilinearly resized+summed into one [img_h,img_w,512] map (resize and resampler are linear per channel).
#include <cstdio>
#include <cstring>

#include <cstdlib>

#include "common.cuh"

namespace disn {

// ------------------------------------------------------------------------------------------------
// TF-legacy bilinear resize (align_corners=False, no half-pixel centres), NHWC, any C.
// ------------------------------------------------------------------------------------------------
__global__ void resize_bilinear_tf_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int H,
                                          int W, int C, int OH, int OW) {
  const float sy = (float)H / (float)OH, sx = (float)W / (float)OW;
  int64_t total = (int64_t)B * OH * OW * C;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    int64_t p = i / C;
    int ox = (int)(p % OW); p /= OW;
    int oy = (int)(p % OH);
    int b = (int)(p / OH);
    float fy = __fmul_rn((float)oy, sy), fx = __fmul_rn((float)ox, sx);
    int y0 = (int)floorf(fy), x0 = (int)floorf(fx);
    int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
    float ly = __fsub_rn(fy, (float)y0), lx = __fsub_rn(fx, (float)x0);
    const float* base = in + (int64_t)b * H * W * C;
    float tl = base[((int64_t)y0 * W + x0) * C + c], tr = base[((int64_t)y0 * W + x1) * C + c];
    float bl = base[((int64_t)y1 * W + x0) * C + c], br = base[((int64_t)y1 * W + x1) * C + c];
    float top = __fadd_rn(tl, __fmul_rn(__fsub_rn(tr, tl), lx));
    float bot = __fadd_rn(bl, __fmul_rn(__fsub_rn(br, bl), lx));
    out[i] = __fadd_rn(top, __fmul_rn(__fsub_rn(bot, top), ly));
  }
}

// ------------------------------------------------------------------------------------------------
// fp32 GEMM  C[M,N] = act(A[M,K] * Bm[K,N] + bias[N]),  A either a plain row-major matrix or the
// implicit im2col view of an NHWC tensor under a 3x3 SAME convolution (K = 9*Cin, k = (ky*3+kx)*Cin+ci,
// which is exactly the row order of TF's HWIO weights reshaped to [9*Cin, Cout]).
// Tile 128 x BN x 8, 256 threads, TM x 8 outputs per thread.
// ------------------------------------------------------------------------------------------------
enum { A_PLAIN = 0, A_IM2COL = 1 };

struct ConvGeom { int H, W, Cin; };

template <int BN, int MODE, bool VEC>
__global__ void __launch_bounds__(256) gemm_f32_kernel(const float* __restrict__ A, const float* __restrict__ Bm,
                                                       const float* __restrict__ bias, float* __restrict__ C,
                                                       int M, int N, int K, int relu, ConvGeom g, int kper,
                                                       float* __restrict__ ws) {
  constexpr int BM = 128, BK = 8;
  constexpr int TN = 8;
  constexpr int TX = BN / TN;        // threads along N: 16 (BN=128) or 8 (BN=64)
  constexpr int TY = 256 / TX;       // threads along M: 16 or 32
  constexpr int TM = BM / TY;        // 8 or 4
  __shared__ __align__(16) float As[BK][BM];
  __shared__ __align__(16) float Bs[BK][BN];

  const int tid = threadIdx.x;
  const int tx = tid % TX, ty = tid / TX;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;

  // A loader: thread -> (row = tid/2, k-part = (tid%2)*4)
  const int a_row = tid >> 1, a_k = (tid & 1) * 4;
  const int am = m0 + a_row;
  int py = 0, px = 0;
  const float* a_img = A;
  if (MODE == A_IM2COL) {
    int hw = g.H * g.W;
    int b = am / hw, r = am % hw;
    py = r / g.W; px = r % g.W;
    a_img = A + (int64_t)b * hw * g.Cin;
  }
  // B loader: BK x BN floats as float4: (BK*BN/4) vectors
  constexpr int BVEC = BK * BN / 4;
  const int b_row = tid / (BN / 4), b_col = (tid % (BN / 4)) * 4;

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  float4 a_reg, b_reg;
  auto load_tiles = [&](int k0) {
    // ---- A ----
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (am < M) {
      int kk = k0 + a_k;
      if (MODE == A_PLAIN) {
        if (VEC) {
          if (kk < K) *reinterpret_cast<float4*>(v) = *reinterpret_cast<const float4*>(A + (int64_t)am * K + kk);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) if (kk + j < K) v[j] = A[(int64_t)am * K + kk + j];
        }
      } else {
        if (VEC) {  // Cin % 4 == 0: the 4 k's share (ky,kx) and are contiguous channels
          if (kk < K) {
            int t = kk / g.Cin, ci = kk % g.Cin;
            int yy = py + t / 3 - 1, xx = px + t % 3 - 1;
            if (yy >= 0 && yy < g.H && xx >= 0 && xx < g.W)
              *reinterpret_cast<float4*>(v) =
                  *reinterpret_cast<const float4*>(a_img + ((int64_t)yy * g.W + xx) * g.Cin + ci);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            int k = kk + j;
            if (k < K) {
              int t = k / g.Cin, ci = k % g.Cin;
              int yy = py + t / 3 - 1, xx = px + t % 3 - 1;
              if (yy >= 0 && yy < g.H && xx >= 0 && xx < g.W) v[j] = a_img[((int64_t)yy * g.W + xx) * g.Cin + ci];
            }
          }
        }
      }
    }
    a_reg = make_float4(v[0], v[1], v[2], v[3]);
    // ---- B ----
    b_reg = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tid < BVEC) {
      int k = k0 + b_row;
      if (k < K) b_reg = *reinterpret_cast<const float4*>(Bm + (int64_t)k * N + n0 + b_col);
    }
  };
  auto store_tiles = [&]() {
    As[a_k + 0][a_row] = a_reg.x; As[a_k + 1][a_row] = a_reg.y;
    As[a_k + 2][a_row] = a_reg.z; As[a_k + 3][a_row] = a_reg.w;
    if (tid < BVEC) *reinterpret_cast<float4*>(&Bs[b_row][b_col]) = b_reg;
  };

  // split-K: blockIdx.z owns k in [k_begin, k_end); partial sums go to the workspace, reduced afterwards
  const int k_begin = blockIdx.z * kper;
  const int k_end = min(K, k_begin + kper);
  load_tiles(k_begin);
  for (int k0 = k_begin; k0 < k_end; k0 += BK) {
    store_tiles();
    __syncthreads();
    if (k0 + BK < k_end) load_tiles(k0 + BK);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; i += 4)
        *reinterpret_cast<float4*>(&a[i]) = *reinterpret_cast<const float4*>(&As[k][ty * TM + i]);
      *reinterpret_cast<float4*>(&b[0]) = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      *reinterpret_cast<float4*>(&b[4]) = *reinterpret_cast<const float4*>(&Bs[k][BN / 2 + tx * 4]);
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  // epilogue: columns {n0 + tx*4 .. +3} and {n0 + BN/2 + tx*4 .. +3}
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    int m = m0 + ty * TM + i;
    if (m >= M) continue;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      int n = n0 + h * (BN / 2) + tx * 4;
      float4 o;
      float* op = reinterpret_cast<float*>(&o);
      if (ws) {
#pragma unroll
        for (int j = 0; j < 4; ++j) op[j] = acc[i][h * 4 + j];
        *reinterpret_cast<float4*>(ws + ((int64_t)blockIdx.z * M + m) * N + n) = o;
        continue;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float v = acc[i][h * 4 + j] + (bias ? bias[n + j] : 0.f);
        op[j] = relu ? fmaxf(v, 0.f) : v;
      }
      *reinterpret_cast<float4*>(C + (int64_t)m * N + n) = o;
    }
  }
}

// C[m,n] = act(bias[n] + sum_z ws[z,m,n])
__global__ void splitk_reduce_kernel(const float4* __restrict__ ws, const float* __restrict__ bias,
                                     float4* __restrict__ C, int64_t MN4, int N4, int splits, int relu) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < MN4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 s = ws[i];
    for (int z = 1; z < splits; ++z) {
      const float4 v = ws[(int64_t)z * MN4 + i];
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    if (bias) {
      const float4 b = reinterpret_cast<const float4*>(bias)[i % N4];
      s.x += b.x; s.y += b.y; s.z += b.z; s.w += b.w;
    }
    if (relu) { s.x = fmaxf(s.x, 0.f); s.y = fmaxf(s.y, 0.f); s.z = fmaxf(s.z, 0.f); s.w = fmaxf(s.w, 0.f); }
    C[i] = s;
  }
}

template <int BN>
static void gemm_dispatch(int mode, bool vec, dim3 grid, cudaStream_t st, const float* A, const float* Bm,
                          const float* bias, float* C, int M, int N, int K, int relu, ConvGeom g, int kper, float* ws) {
  dim3 block(256);
  if (mode == A_PLAIN) {
    if (vec) gemm_f32_kernel<BN, A_PLAIN, true><<<grid, block, 0, st>>>(A, Bm, bias, C, M, N, K, relu, g, kper, ws);
    else gemm_f32_kernel<BN, A_PLAIN, false><<<grid, block, 0, st>>>(A, Bm, bias, C, M, N, K, relu, g, kper, ws);
  } else {
    if (vec) gemm_f32_kernel<BN, A_IM2COL, true><<<grid, block, 0, st>>>(A, Bm, bias, C, M, N, K, relu, g, kper, ws);
    else gemm_f32_kernel<BN, A_IM2COL, false><<<grid, block, 0, st>>>(A, Bm, bias, C, M, N, K, relu, g, kper, ws);
  }
}

static int launch_gemm(disn_ctx* c, int mode, const float* A, const float* Bm, const float* bias, float* C, int M,
                       int N, int K, int relu, ConvGeom g) {
  bool vec = (mode == A_PLAIN) ? (K % 4 == 0) : (g.Cin % 4 == 0);
  const int BN = (N % 128 == 0) ? 128 : 64;
  if (N % 64 != 0) { set_error("gemm: N must be a multiple of 64"); return -2; }
  const int ctas = (N / BN) * ((M + 127) / 128);
  // split-K so that small late layers (few output tiles) still fill 148 SMs for ~2 waves
  int splits = 1;
  if (K % 8 == 0 && ctas < 148) {
    const int kchunks = K / 64 > 0 ? K / 64 : 1;             // keep >= 64 k per split
    int want = (296 + ctas - 1) / ctas;
    if (want > kchunks) want = kchunks;
    for (int d = want; d >= 1; --d)
      if ((K / 8) % d == 0) { splits = d; break; }
    if ((size_t)splits * M * N * sizeof(float) > c->splitk_ws.bytes()) splits = 1;
  }
  const int kper = (splits == 1) ? K : K / splits;
  dim3 grid(N / BN, (M + 127) / 128, splits);
  float* ws = splits > 1 ? c->splitk_ws.get<float>() : nullptr;
  if (BN == 128) gemm_dispatch<128>(mode, vec, grid, c->stream, A, Bm, bias, C, M, N, K, relu, g, kper, ws);
  else gemm_dispatch<64>(mode, vec, grid, c->stream, A, Bm, bias, C, M, N, K, relu, g, kper, ws);
  c->launches++;
  if (splits > 1) {
    const int64_t mn4 = (int64_t)M * N / 4;
    int blocks = (int)std::min<int64_t>((mn4 + 255) / 256, 148 * 8);
    splitk_reduce_kernel<<<blocks, 256, 0, c->stream>>>(reinterpret_cast<const float4*>(ws), bias,
                                                       reinterpret_cast<float4*>(C), mn4, N / 4, splits, relu);
    c->launches++;
  }
  DISN_CUDA_OK(cudaGetLastError());
  return 0;
}

// GEMM dispatcher: tcgen05 path (bf16 hi/lo split, fp32 accumulate) when the context runs in DISN_PREC_BF16X3 and
// the shapes fit (K % 64 == 0, channels % 64 == 0); fp32 CUDA-core path otherwise (conv1_1: Cin = 3).
static int gemm_any(disn_ctx* c, const std::string& wname, int mode, const float* A, const float* Bm, const float* bias,
                    float* C, int M, int N, int K, int relu, ConvGeom g) {
  const bool tc_ok = c->cfg.precision != DISN_PREC_FP32 && K % 64 == 0 && N % 32 == 0 &&
                     (mode == A_PLAIN || g.Cin % 64 == 0);
  if (!tc_ok) return launch_gemm(c, mode, A, Bm, bias, C, M, N, K, relu, g);
  DevBuf& pk = c->enc_tc_weights[wname];
  if (!pk.bytes() && conv_tc_pack(c, Bm, K, N, pk)) return -1;
  int splits = 1;
  float* ws = c->splitk_ws.get<float>();
  if (launch_conv_tc(c, A, pk.get<uint8_t>(), bias, C, ws, c->splitk_ws.bytes() / sizeof(float), M, N, K,
                     mode == A_IM2COL ? g.H : 0, g.W, g.Cin, relu, &splits))
    return -1;
  if (splits > 1) {
    const int64_t mn4 = (int64_t)M * N / 4;
    int blocks = (int)std::min<int64_t>((mn4 + 255) / 256, 148 * 8);
    splitk_reduce_kernel<<<blocks, 256, 0, c->stream>>>(reinterpret_cast<const float4*>(ws), bias,
                                                       reinterpret_cast<float4*>(C), mn4, N / 4, splits, relu);
    c->launches++;
    DISN_CUDA_OK(cudaGetLastError());
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// 2x2 / stride-2 VALID max pool, NHWC, C % 4 == 0
// ------------------------------------------------------------------------------------------------
__global__ void maxpool2_kernel(const float4* __restrict__ in, float4* __restrict__ out, int B, int H, int W, int C4) {
  int OH = H / 2, OW = W / 2;
  int64_t total = (int64_t)B * OH * OW * C4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % C4);
    int64_t p = i / C4;
    int ox = (int)(p % OW); p /= OW;
    int oy = (int)(p % OH);
    int b = (int)(p / OH);
    const float4* base = in + (((int64_t)b * H + oy * 2) * W + ox * 2) * C4 + c;
    float4 v0 = base[0], v1 = base[C4], v2 = base[(int64_t)W * C4], v3 = base[(int64_t)W * C4 + C4];
    float4 r;
    r.x = fmaxf(fmaxf(v0.x, v1.x), fmaxf(v2.x, v3.x));
    r.y = fmaxf(fmaxf(v0.y, v1.y), fmaxf(v2.y, v3.y));
    r.z = fmaxf(fmaxf(v0.z, v1.z), fmaxf(v2.z, v3.z));
    r.w = fmaxf(fmaxf(v0.w, v1.w), fmaxf(v2.w, v3.w));
    out[i] = r;
  }
}

// ------------------------------------------------------------------------------------------------
// Batched GEMV for the fc layers (M = batch <= 8): weight-streaming, split-K, deterministic 2-pass.
//   partial[s][b][n] = sum_{k in split s} x[b][k] * W[k][n];   out[b][n] = act(bias[n] + sum_s partial)
// ------------------------------------------------------------------------------------------------
constexpr int GEMV_KS = 64;     // rows of W per block
constexpr int GEMV_MAXB = 8;

__global__ void __launch_bounds__(256) gemv_partial_kernel(const float* __restrict__ x, const float* __restrict__ W,
                                                           float* __restrict__ partial, int B, int K, int N) {
  __shared__ float xs[GEMV_MAXB][GEMV_KS];
  const int n = (blockIdx.x * 256 + threadIdx.x) * 4;
  const int k0 = blockIdx.y * GEMV_KS;
  for (int i = threadIdx.x; i < B * GEMV_KS; i += 256) {
    int b = i / GEMV_KS, k = i % GEMV_KS;
    xs[b][k] = (k0 + k < K) ? x[(int64_t)b * K + k0 + k] : 0.f;
  }
  __syncthreads();
  if (n >= N) return;
  float acc[GEMV_MAXB][4];
#pragma unroll
  for (int b = 0; b < GEMV_MAXB; ++b) acc[b][0] = acc[b][1] = acc[b][2] = acc[b][3] = 0.f;
  const int kend = min(GEMV_KS, K - k0);
#pragma unroll 4
  for (int k = 0; k < kend; ++k) {
    float4 w = __ldg(reinterpret_cast<const float4*>(W + (int64_t)(k0 + k) * N + n));
#pragma unroll
    for (int b = 0; b < GEMV_MAXB; ++b) {
      if (b < B) {
        float xv = xs[b][k];
        acc[b][0] = fmaf(xv, w.x, acc[b][0]); acc[b][1] = fmaf(xv, w.y, acc[b][1]);
        acc[b][2] = fmaf(xv, w.z, acc[b][2]); acc[b][3] = fmaf(xv, w.w, acc[b][3]);
      }
    }
  }
#pragma unroll
  for (int b = 0; b < GEMV_MAXB; ++b)
    if (b < B)
      *reinterpret_cast<float4*>(partial + ((int64_t)blockIdx.y * B + b) * N + n) =
          make_float4(acc[b][0], acc[b][1], acc[b][2], acc[b][3]);
}

__global__ void gemv_reduce_kernel(const float* __restrict__ partial, const float* __restrict__ bias,
                                   float* __restrict__ out, int B, int N, int splits, int relu) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * N) return;
  int n = i % N;
  float s = 0.f;
  for (int sp = 0; sp < splits; ++sp) s += partial[(int64_t)sp * B * N + i];
  s += bias ? bias[n] : 0.f;
  out[i] = relu ? fmaxf(s, 0.f) : s;
}

static int launch_gemv(disn_ctx* c, const float* x, const float* W, const float* bias, float* out, int B, int K,
                       int N, int relu) {
  DISN_REQUIRE(B <= GEMV_MAXB && N % 4 == 0, "gemv: batch <= 8 and N % 4 == 0");
  int splits = (K + GEMV_KS - 1) / GEMV_KS;
  dim3 grid((N / 4 + 255) / 256, splits);
  float* partial = c->partial.get<float>();
  gemv_partial_kernel<<<grid, 256, 0, c->stream>>>(x, W, partial, B, K, N);
  gemv_reduce_kernel<<<(B * N + 255) / 256, 256, 0, c->stream>>>(partial, bias, out, B, N, splits, relu);
  c->launches += 2;
  DISN_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// pmap[b,y,x,:] = sum_l  tf_resize_bilinear(proj_l)[b,y,x,:]      (5 levels, 512 channels)
// ------------------------------------------------------------------------------------------------
struct PmapLevels { const float* p[5]; int h[5]; };

__global__ void pmap_accumulate_kernel(PmapLevels lv, float4* __restrict__ pmap, int B, int OH, int OW) {
  constexpr int C4 = kHidden / 4;
  int64_t total = (int64_t)B * OH * OW * C4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % C4);
    int64_t p = i / C4;
    int ox = (int)(p % OW); p /= OW;
    int oy = (int)(p % OH);
    int b = (int)(p / OH);
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int l = 0; l < 5; ++l) {
      int h = lv.h[l];
      float sy = (float)h / (float)OH, sx = (float)h / (float)OW;
      float fy = __fmul_rn((float)oy, sy), fx = __fmul_rn((float)ox, sx);
      int y0 = (int)floorf(fy), x0 = (int)floorf(fx);
      int y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, h - 1);
      float ly = __fsub_rn(fy, (float)y0), lx = __fsub_rn(fx, (float)x0);
      const float4* base = reinterpret_cast<const float4*>(lv.p[l]) + (int64_t)b * h * h * C4 + c;
      float4 tl = base[((int64_t)y0 * h + x0) * C4], tr = base[((int64_t)y0 * h + x1) * C4];
      float4 bl = base[((int64_t)y1 * h + x0) * C4], br = base[((int64_t)y1 * h + x1) * C4];
#define DISN_LERP(f)                                        \
  {                                                         \
    float top = tl.f + (tr.f - tl.f) * lx;                  \
    float bot = bl.f + (br.f - bl.f) * lx;                  \
    s.f += top + (bot - top) * ly;                          \
  }
      DISN_LERP(x) DISN_LERP(y) DISN_LERP(z) DISN_LERP(w)
#undef DISN_LERP
    }
    pmap[i] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static const int kConvCin[kNumConv] = {3, 64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512};
static const int kConvCout[kNumConv] = {64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512, 512};
static const int kConvHW[kNumConv] = {224, 224, 112, 112, 56, 56, 56, 28, 28, 28, 14, 14, 14};
static const char* kConvName[kNumConv] = {
    "vgg_16/conv1/conv1_1", "vgg_16/conv1/conv1_2", "vgg_16/conv2/conv2_1", "vgg_16/conv2/conv2_2",
    "vgg_16/conv3/conv3_1", "vgg_16/conv3/conv3_2", "vgg_16/conv3/conv3_3", "vgg_16/conv4/conv4_1",
    "vgg_16/conv4/conv4_2", "vgg_16/conv4/conv4_3", "vgg_16/conv5/conv5_1", "vgg_16/conv5/conv5_2",
    "vgg_16/conv5/conv5_3"};
static const int kTapHW[5] = {224, 112, 56, 28, 14};

int encoder_alloc(disn_ctx* c, int B) {
  if (B <= c->alloc_B) return 0;
  const int64_t Bn = B, V = c->cfg.vgg_in;
  std::vector<std::pair<DevBuf*, int64_t>> bufs = {{&c->img_in, Bn * V * V * 4}, {&c->img_rs, Bn * V * V * 3},
                                                   {&c->act[0], Bn * V * V * 64}, {&c->act[1], Bn * V * V * 64}};
  for (int i = 0; i < 5; ++i) {
    bufs.push_back({&c->taps[i], Bn * kTapHW[i] * kTapHW[i] * kTapC[i]});
    bufs.push_back({&c->proj[i], Bn * kTapHW[i] * kTapHW[i] * kHidden});
  }
  bufs.insert(bufs.end(), {{&c->fc_a, Bn * 4096}, {&c->fc_b, Bn * 4096},
                           {&c->partial, (int64_t)((25088 + GEMV_KS - 1) / GEMV_KS) * Bn * 4096},
                           {&c->emb, Bn * c->cfg.num_classes}, {&c->gbias, Bn * kHidden},
                           {&c->pmap, Bn * c->cfg.img_h * c->cfg.img_w * kHidden},
                           {&c->splitk_ws, Bn * 8 * 1024 * 1024}});     // 32 MB per image of split-K partial sums
  // all or nothing: every buffer is freed before any is allocated at the new size
  encoder_graph_reset(c);      // the captured graph holds these buffers' addresses
  for (auto& b : bufs) b.first->reset();
  c->alloc_B = 0;
  DISN_REQUIRE(V == 224, "vgg_in must be 224 (fc6 is a 7x7 VALID conv on the pool5 map)");
  for (auto& b : bufs)
    if (b.first->reserve(b.second * sizeof(float))) return -1;
  c->alloc_B = B;
  return 0;
}

}  // namespace disn
#ifdef DISN_DIAGNOSTICS
// Diagnostic: run one GEMM (plain if H == 0, else 3x3 SAME im2col of an NHWC tensor) through both the fp32
// CUDA-core kernel and the tcgen05 kernel; host pointers.  Used by the GPU test-suite to sweep shapes.
extern "C" int disn_debug_gemm(disn_ctx* c, const float* A, const float* Wt, const float* bias, int M, int N, int K,
                               int H, int Wd, int Cin, int relu, float* out_fp32, float* out_tc) {
  using namespace disn;
  DISN_REQUIRE(c && A && Wt && out_fp32 && out_tc, "null argument");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  if (encoder_alloc(c, 1)) return -1;
  const size_t a_elems = H ? (size_t)M * Cin : (size_t)M * K;
  DevBuf bA, bW, bB, bC;
  if (bA.reserve(a_elems * 4) || bW.reserve((size_t)K * N * 4) || bC.reserve((size_t)M * N * 4)) return -1;
  float *dA = bA.get<float>(), *dW = bW.get<float>(), *dC = bC.get<float>();
  DISN_CUDA_OK(cudaMemcpy(dA, A, a_elems * 4, cudaMemcpyHostToDevice));
  DISN_CUDA_OK(cudaMemcpy(dW, Wt, (size_t)K * N * 4, cudaMemcpyHostToDevice));
  if (bias) {
    if (bB.reserve((size_t)N * 4)) return -1;
    DISN_CUDA_OK(cudaMemcpy(bB.get<float>(), bias, (size_t)N * 4, cudaMemcpyHostToDevice));
  }
  const float* dB = bB.get<float>();
  DISN_CUDA_OK(cudaDeviceSynchronize());   // pageable H2D copies above are not ordered against the ctx stream
  ConvGeom g{H, Wd, Cin};
  const int mode = H ? A_IM2COL : A_PLAIN;
  const int saved = c->cfg.precision;
  int rc = 0;
  for (int pass = 0; pass < 2 && rc == 0; ++pass) {
    c->cfg.precision = pass ? DISN_PREC_BF16X3 : DISN_PREC_FP32;
    c->enc_tc_weights.erase("debug_gemm");
    DISN_CUDA_OK(cudaMemset(dC, 0xff, (size_t)M * N * 4));
    rc = gemm_any(c, "debug_gemm", mode, dA, dW, dB, dC, M, N, K, relu, g);
    if (rc == 0) {
      DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
      DISN_CUDA_OK(cudaMemcpy(pass ? out_tc : out_fp32, dC, (size_t)M * N * 4, cudaMemcpyDeviceToHost));
    }
  }
  c->cfg.precision = saved;
  c->enc_tc_weights.erase("debug_gemm");
  return rc;
}
#endif  // DISN_DIAGNOSTICS
namespace disn {

static const float* wptr(disn_ctx* c, const std::string& name) {
  auto it = c->weights.find(name);
  return it == c->weights.end() ? nullptr : it->second.data.get<float>();
}

int encoder_gemv(disn_ctx* c, const float* x, const float* W, const float* bias, float* out, int B, int K, int N, int relu) {
  return launch_gemv(c, x, W, bias, out, B, K, N, relu);
}
int encoder_gemm_plain(disn_ctx* c, const std::string& wname, const float* A, const float* Bm, const float* bias, float* C,
                       int M, int N, int K, int relu) {
  if (encoder_alloc(c, 1)) return -1;     // split-K workspace
  ConvGeom g{0, 0, 0};
  return gemm_any(c, wname, A_PLAIN, A, Bm, bias, C, M, N, K, relu, g);
}

static int encoder_body(disn_ctx* c, int B, int H, int W, int C, bool embedding_only);

// The encoder is ~50 small launches (13 convs with split-K reduces, pools, GEMVs, 5 projections, the map fold): at B = 1
// their GPU time is ~0.5 ms but the launch gaps made it ~3 ms per step.  After one eager run per shape (which also packs
// the tcgen05 weight images), the launch sequence is captured into a CUDA graph and replayed with one cudaGraphLaunch.
void encoder_graph_reset(disn_ctx* c) {
  if (c->enc_graph_exec) cudaGraphExecDestroy(c->enc_graph_exec);
  c->enc_graph_exec = nullptr;
  c->enc_graph_key.clear();
  c->enc_warm_key.clear();
}

int encoder_run(disn_ctx* c, const float* imgs, int B, int H, int W, int C, bool device_ptr, bool embedding_only) {
  DISN_REQUIRE(C == 3, "imgs must have 3 channels (FLAGS.alpha is not on the hot path)");
  DISN_REQUIRE(B >= 1 && B <= GEMV_MAXB, "batch must be in [1,8]");
  DISN_REQUIRE((int64_t)H * W <= (int64_t)c->cfg.vgg_in * c->cfg.vgg_in * 4 / 3, "input image too large");
  if (encoder_alloc(c, B)) return -1;
  DISN_CUDA_OK(cudaMemcpyAsync(c->img_in.get<float>(), imgs, (size_t)B * H * W * C * sizeof(float),
                               device_ptr ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->stream));
  const std::vector<int64_t> key = {B, H, W, C, (int64_t)embedding_only, (int64_t)c->cfg.precision};
  static const bool no_graph = getenv("DISN_NO_GRAPH") != nullptr;
  if (!no_graph && c->enc_graph_exec && key == c->enc_graph_key) {
    DISN_CUDA_OK(cudaGraphLaunch(c->enc_graph_exec, c->stream));
    c->launches += c->enc_graph_launches;
    c->enc_B = embedding_only ? 0 : B;
    return 0;
  }
  if (no_graph || key != c->enc_warm_key) {      // first time with this shape: eager (packs weights, sets attributes)
    const int rc = encoder_body(c, B, H, W, C, embedding_only);
    if (rc == 0) c->enc_warm_key = key;
    return rc;
  }
  // second time: capture, instantiate, replay
  if (c->enc_graph_exec) { cudaGraphExecDestroy(c->enc_graph_exec); c->enc_graph_exec = nullptr; c->enc_graph_key.clear(); }
  const int64_t l0 = c->launches;
  DISN_CUDA_OK(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
  const int rc = encoder_body(c, B, H, W, C, embedding_only);
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(c->stream, &graph);
  c->enc_graph_launches = c->launches - l0;
  c->launches = l0;
  if (rc != 0 || ce != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    c->enc_B = 0;
    if (rc == 0) set_error(std::string("encoder graph capture failed: ") + cudaGetErrorString(ce));
    return -1;
  }
  const cudaError_t ie = cudaGraphInstantiate(&c->enc_graph_exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ie != cudaSuccess) { c->enc_graph_exec = nullptr; set_error(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ie)); return -1; }
  c->enc_graph_key = key;
  DISN_CUDA_OK(cudaGraphLaunch(c->enc_graph_exec, c->stream));
  c->launches += c->enc_graph_launches;
  c->enc_B = embedding_only ? 0 : B;
  return 0;
}

static int encoder_body(disn_ctx* c, int B, int H, int W, int C, bool embedding_only) {
  const int V = c->cfg.vgg_in;
  for (int i = 0; i < kNumConv; ++i) {
    DISN_REQUIRE(wptr(c, std::string(kConvName[i]) + "/weights") && wptr(c, std::string(kConvName[i]) + "/biases"),
                 std::string("missing weights for ") + kConvName[i]);
  }
  for (const char* nm : {"vgg_16/fc6", "vgg_16/fc7", "vgg_16/fc8", "sdfprediction/fold2/conv1",
                         "sdfprediction_imgfeat/fold2/conv1"}) {
    if (embedding_only && std::string(nm).rfind("sdfprediction", 0) == 0) continue;
    DISN_REQUIRE(wptr(c, std::string(nm) + "/weights") && wptr(c, std::string(nm) + "/biases"),
                 std::string("missing weights for ") + nm);
  }

  float *img_in = c->img_in.get<float>(), *img_rs = c->img_rs.get<float>();
  const float* x = img_in;
  if (H != V || W != V) {  // model_normalization.py:65-72
    resize_bilinear_tf_kernel<<<592, 256, 0, c->stream>>>(img_in, img_rs, B, H, W, C, V, V);
    c->launches++;
    x = img_rs;
  } else {
    DISN_CUDA_OK(cudaMemcpyAsync(img_rs, img_in, (size_t)B * V * V * 3 * sizeof(float), cudaMemcpyDeviceToDevice, c->stream));
    x = img_rs;
  }
  // 13 convs + 5 pools (models/CNN/vgg.py:187-196)
  int pp = 0, tap = 0;
  for (int i = 0; i < kNumConv; ++i) {
    int hw = kConvHW[i];
    bool is_tap = (tap < 5 && kTapLayer[tap] == i);
    float* y = is_tap ? c->taps[tap].get<float>() : c->act[pp].get<float>();
    ConvGeom g{hw, hw, kConvCin[i]};
    if (gemm_any(c, std::string(kConvName[i]) + "/weights", A_IM2COL, x, wptr(c, std::string(kConvName[i]) + "/weights"),
                 wptr(c, std::string(kConvName[i]) + "/biases"), y, B * hw * hw, kConvCout[i], 9 * kConvCin[i], 1, g))
      return -1;
    x = y;
    if (!is_tap) pp ^= 1;
    if (is_tap) {
      float* p = c->act[pp].get<float>();
      int64_t total = (int64_t)B * (hw / 2) * (hw / 2) * (kConvCout[i] / 4);
      int blocks = (int)std::min<int64_t>((total + 255) / 256, 148 * 8);
      maxpool2_kernel<<<blocks, 256, 0, c->stream>>>(reinterpret_cast<const float4*>(x), reinterpret_cast<float4*>(p),
                                                     B, hw, hw, kConvCout[i] / 4);
      c->launches++;
      x = p;
      pp ^= 1;
      ++tap;
    }
  }
  // fc6 (7x7 VALID == dense over the (y,x,c)-flattened 7x7x512 map), fc7, fc8 (linear)
  float *fc_a = c->fc_a.get<float>(), *fc_b = c->fc_b.get<float>(), *emb = c->emb.get<float>();
  if (launch_gemv(c, x, wptr(c, "vgg_16/fc6/weights"), wptr(c, "vgg_16/fc6/biases"), fc_a, B, 7 * 7 * 512, 4096, 1))
    return -1;
  if (launch_gemv(c, fc_a, wptr(c, "vgg_16/fc7/weights"), wptr(c, "vgg_16/fc7/biases"), fc_b, B, 4096, 4096, 1))
    return -1;
  if (launch_gemv(c, fc_b, wptr(c, "vgg_16/fc8/weights"), wptr(c, "vgg_16/fc8/biases"), emb, B, 4096,
                  c->cfg.num_classes, 0))
    return -1;
  if (embedding_only) {      // camera-pose net: only the VGG embedding is needed
    c->enc_B = 0;
    return 0;
  }
  // global-feature fold: gbias = emb * Wg[512:512+nc, :] + b   (models/sdfnet.py:78-85)
  if (launch_gemv(c, emb, wptr(c, "sdfprediction/fold2/conv1/weights") + (int64_t)kHidden * kHidden,
                  wptr(c, "sdfprediction/fold2/conv1/biases"), c->gbias.get<float>(), B, c->cfg.num_classes, kHidden, 0))
    return -1;
  // local-feature fold: proj_l = tap_l * Wl[512+off_l : 512+off_l+C_l, :]   (models/sdfnet.py:180-183)
  const float* wl = wptr(c, "sdfprediction_imgfeat/fold2/conv1/weights") + (int64_t)kHidden * kHidden;
  int off = 0;
  PmapLevels lv;
  for (int l = 0; l < 5; ++l) {
    int hw = kTapHW[l];
    const float* src = c->taps[l].get<float>();
    if (hw > c->cfg.img_h && c->cfg.img_h == c->cfg.img_w) {
      // resize and projection commute (both linear per channel): where the tap is LARGER than the 137x137 target (conv1_2,
      // 224x224) resize first -- the GEMM then has 2.7x fewer rows and the [B,224,224,512] intermediate (103 MB per image)
      // never exists.  This is also the reference's own order (model_normalization.py:171-172).
      float* tmp = c->act[0].get<float>();
      const int oh = c->cfg.img_h;
      const int64_t total = (int64_t)B * oh * oh * kTapC[l];
      resize_bilinear_tf_kernel<<<(int)std::min<int64_t>((total + 255) / 256, 148 * 16), 256, 0, c->stream>>>(
          c->taps[l].get<float>(), tmp, B, hw, hw, kTapC[l], oh, oh);
      c->launches++;
      src = tmp;
      hw = oh;
    }
    ConvGeom g{0, 0, 0};
    if (gemm_any(c, "proj" + std::to_string(l), A_PLAIN, src, wl + (int64_t)off * kHidden, nullptr, c->proj[l].get<float>(),
                 B * hw * hw, kHidden, kTapC[l], 0, g))
      return -1;
    off += kTapC[l];
    lv.p[l] = c->proj[l].get<float>();
    lv.h[l] = hw;
  }
  {
    int64_t total = (int64_t)B * c->cfg.img_h * c->cfg.img_w * (kHidden / 4);
    int blocks = (int)std::min<int64_t>((total + 255) / 256, 148 * 16);
    pmap_accumulate_kernel<<<blocks, 256, 0, c->stream>>>(lv, reinterpret_cast<float4*>(c->pmap.get<float>()), B, c->cfg.img_h,
                                                          c->cfg.img_w);
    c->launches++;
  }
  DISN_CUDA_OK(cudaGetLastError());
  c->enc_B = B;
  return 0;
}

}  // namespace disn
