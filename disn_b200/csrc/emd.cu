// Approximate earth mover's distance between point sets -- the B200 replacement of the reference's custom TF ops
// ApproxMatch / MatchCost (models/tf_ops/approxmatch/tf_approxmatch.cpp:23-85 `approxmatch_cpu`, :86-107 `matchcost_cpu`;
// GPU twins in tf_approxmatch_g.cu), used by the mesh metrics (test/test_cd_emd.py:307-308).
//
// The algorithm is eleven rounds (j = 8..-2) of a soft assignment: weights expf(-4^j |p_k - q_l|^2) scaled by what point l
// can still take, normalised per row to what point k can still give, clipped per column, accumulated into `match`.
// The reference materialises the N x M weight matrix in float64 and sweeps it five times per round.  Here nothing but
// `match` is materialised: each round is four passes that RECOMPUTE the weight of a pair from the coordinates (one exp per
// pair and pass -- the work is ~2e8 exps per cloud pair, nothing next to the 16 MB of `match` traffic it saves):
//   rows A: s_k  = 1e-9 + sum_l e_kl satr_l                       cols B: c_l = min(satr_l / (1e-9 + sum_k e_kl satr_l / s_k satl_k), 1)
//   rows C: w_kl = e_kl satr_l / s_k satl_k c_l; match += w; satl'_k = max(satl_k - sum_l w_kl, 0)
//   cols D: satr'_l = max(satr_l - sum_k w_kl, 0)
// Arithmetic follows the CPU op operation for operation -- float32 coordinates widened to float64, the exponent rounded to
// float32, expf in float32 (computed as the float64 exp rounded once, which agrees with a correctly rounded expf), all else
// float64 without FMA contraction, `match` accumulated in float32 -- so the result differs from it only through the order
// of the float64 sums (~1e-16 relative) and the rare last-bit difference of expf.  Every reduction has a fixed order:
// results are reproducible run to run.
#include "common.cuh"

namespace disn {
namespace {

constexpr int EM_WARPS = 8;
constexpr int EM_THREADS = EM_WARPS * 32;

struct EmdJob {
  const float* xyz1;   // [B,N,3]
  const float* xyz2;   // [B,M,3]
  const double* satl;  // [B,N]  what point k of set 1 can still give
  const double* satr;  // [B,M]  what point l of set 2 can still take
  double* satl_next;   // rows C
  double* satr_next;   // cols D
  double* s;           // [B,N]  row normaliser of this round
  double* clip;        // [B,M]  column clip factor of this round
  float* match;        // [B,N,M]
  double level;
  int n, m;
};

__device__ __forceinline__ double pair_exp(double x1, double y1, double z1, double x2, double y2, double z2, double level) {
  const double dx = __dsub_rn(x1, x2), dy = __dsub_rn(y1, y2), dz = __dsub_rn(z1, z2);
  const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
  const float arg = __double2float_rn(__dmul_rn(level, d2));
  return (double)__double2float_rn(exp((double)arg));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// kPass 0: rows A, 2: rows C (one warp per point k of set 1, lanes over l)
template <int kPass>
__global__ void __launch_bounds__(EM_THREADS) emd_rows_kernel(EmdJob j) {
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  const int k = blockIdx.x * EM_WARPS + (threadIdx.x >> 5);
  if (k >= j.n) return;
  const float* p1 = j.xyz1 + ((size_t)b * j.n + k) * 3;
  const float* p2 = j.xyz2 + (size_t)b * j.m * 3;
  const double* satr = j.satr + (size_t)b * j.m;
  const double x1 = p1[0], y1 = p1[1], z1 = p1[2];
  double acc = 0.0;
  if (kPass == 0) {
    for (int l = lane; l < j.m; l += 32)
      acc = __dadd_rn(acc, __dmul_rn(pair_exp(x1, y1, z1, p2[l * 3], p2[l * 3 + 1], p2[l * 3 + 2], j.level), satr[l]));
    acc = warp_sum(acc);
    if (lane == 0) j.s[(size_t)b * j.n + k] = __dadd_rn(1e-9, acc);
  } else {
    const double s = j.s[(size_t)b * j.n + k], sl = j.satl[(size_t)b * j.n + k];
    const double* clip = j.clip + (size_t)b * j.m;
    float* mrow = j.match + ((size_t)b * j.n + k) * j.m;
    for (int l = lane; l < j.m; l += 32) {
      double w = __dmul_rn(pair_exp(x1, y1, z1, p2[l * 3], p2[l * 3 + 1], p2[l * 3 + 2], j.level), satr[l]);
      w = __dmul_rn(__dmul_rn(__ddiv_rn(w, s), sl), clip[l]);
      mrow[l] = __double2float_rn(__dadd_rn((double)mrow[l], w));
      acc = __dadd_rn(acc, w);
    }
    acc = warp_sum(acc);
    if (lane == 0) j.satl_next[(size_t)b * j.n + k] = fmax(__dsub_rn(sl, acc), 0.0);
  }
}

// kPass 1: cols B, 3: cols D (one warp per point l of set 2, lanes over k)
template <int kPass>
__global__ void __launch_bounds__(EM_THREADS) emd_cols_kernel(EmdJob j) {
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  const int l = blockIdx.x * EM_WARPS + (threadIdx.x >> 5);
  if (l >= j.m) return;
  const float* p1 = j.xyz1 + (size_t)b * j.n * 3;
  const float* p2 = j.xyz2 + ((size_t)b * j.m + l) * 3;
  const double* s = j.s + (size_t)b * j.n;
  const double* satl = j.satl + (size_t)b * j.n;
  const double x2 = p2[0], y2 = p2[1], z2 = p2[2];
  const double sr = j.satr[(size_t)b * j.m + l];
  const double cl = kPass == 3 ? j.clip[(size_t)b * j.m + l] : 1.0;
  double acc = 0.0;
  for (int k = lane; k < j.n; k += 32) {
    double w = __dmul_rn(pair_exp(p1[k * 3], p1[k * 3 + 1], p1[k * 3 + 2], x2, y2, z2, j.level), sr);
    w = __dmul_rn(__ddiv_rn(w, s[k]), satl[k]);
    if (kPass == 3) w = __dmul_rn(w, cl);
    acc = __dadd_rn(acc, w);
  }
  acc = warp_sum(acc);
  if (lane == 0) {
    if (kPass == 1) j.clip[(size_t)b * j.m + l] = fmin(__ddiv_rn(sr, __dadd_rn(1e-9, acc)), 1.0);
    else j.satr_next[(size_t)b * j.m + l] = fmax(__dsub_rn(sr, acc), 0.0);
  }
}

__global__ void emd_fill_kernel(double* p, int64_t n, double v) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

// MatchCost: per row k the float64 sum of the float32 products sqrtf(d2) * match (tf_approxmatch.cpp:86-107)
__global__ void __launch_bounds__(EM_THREADS) match_cost_rows_kernel(const float* __restrict__ xyz1, const float* __restrict__ xyz2,
                                                                     const float* __restrict__ match, int n, int m,
                                                                     double* __restrict__ rowcost) {
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  const int k = blockIdx.x * EM_WARPS + (threadIdx.x >> 5);
  if (k >= n) return;
  const float* p1 = xyz1 + ((size_t)b * n + k) * 3;
  const float* p2 = xyz2 + (size_t)b * m * 3;
  const float* mrow = match + ((size_t)b * n + k) * m;
  const float x1 = p1[0], y1 = p1[1], z1 = p1[2];
  double acc = 0.0;
  for (int l = lane; l < m; l += 32) {
    const float dx = __fsub_rn(p2[l * 3], x1), dy = __fsub_rn(p2[l * 3 + 1], y1), dz = __fsub_rn(p2[l * 3 + 2], z1);
    const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    acc = __dadd_rn(acc, (double)__fmul_rn(__fsqrt_rn(d2), mrow[l]));
  }
  acc = warp_sum(acc);
  if (lane == 0) rowcost[(size_t)b * n + k] = acc;
}

__global__ void __launch_bounds__(EM_THREADS) match_cost_sum_kernel(const double* __restrict__ rowcost, int n, float* __restrict__ cost) {
  __shared__ double part[EM_THREADS];
  const int b = blockIdx.x;
  double acc = 0.0;
  for (int k = threadIdx.x; k < n; k += EM_THREADS) acc = __dadd_rn(acc, rowcost[(size_t)b * n + k]);
  part[threadIdx.x] = acc;
  __syncthreads();
  for (int o = EM_THREADS / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) part[threadIdx.x] = __dadd_rn(part[threadIdx.x], part[threadIdx.x + o]);
    __syncthreads();
  }
  if (threadIdx.x == 0) cost[b] = __double2float_rn(part[0]);
}

int match_cost_device(disn_ctx* c, const float* d1, const float* d2, const float* dmatch, int B, int N, int M, double* rowcost,
                      float* dcost) {
  match_cost_rows_kernel<<<dim3((N + EM_WARPS - 1) / EM_WARPS, B), EM_THREADS, 0, c->stream>>>(d1, d2, dmatch, N, M, rowcost);
  match_cost_sum_kernel<<<B, EM_THREADS, 0, c->stream>>>(rowcost, N, dcost);
  c->launches += 2;
  DISN_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace
}  // namespace disn

using namespace disn;

extern "C" int disn_approx_match(disn_ctx* c, const float* xyz1, const float* xyz2, int32_t B, int32_t N, int32_t M,
                                 float* match_out, float* cost_out) {
  DISN_REQUIRE(c && xyz1 && xyz2 && (match_out || cost_out), "null argument");
  DISN_REQUIRE(B >= 1 && N >= 1 && M >= 1 && B <= 65535, "ApproxMatch expects (batch_size,num_points,3) point sets, batch <= 65535");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  const size_t n1 = (size_t)B * N, n2 = (size_t)B * M, nm = (size_t)B * N * M;
  DevBuf buf;       // per call: the match matrix alone is B*N*M floats
  if (buf.reserve((n1 + n2) * 12 + (3 * n1 + 3 * n2) * 8 + nm * 4 + n1 * 8 + (size_t)B * 4 + 16 * 256)) return -1;
  float* d1 = buf.take<float>(n1 * 3);
  float* d2 = buf.take<float>(n2 * 3);
  double* satl[2] = {buf.take<double>(n1), buf.take<double>(n1)};
  double* satr[2] = {buf.take<double>(n2), buf.take<double>(n2)};
  double* s = buf.take<double>(n1);
  double* clip = buf.take<double>(n2);
  float* dmatch = buf.take<float>(nm);
  double* rowcost = buf.take<double>(n1);
  float* dcost = buf.take<float>(B);
  DISN_CUDA_OK(cudaMemcpyAsync(d1, xyz1, n1 * 12, cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaMemcpyAsync(d2, xyz2, n2 * 12, cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaMemsetAsync(dmatch, 0, nm * 4, c->stream));
  const int big = N > M ? N : M;
  emd_fill_kernel<<<c->num_sms, 256, 0, c->stream>>>(satl[0], (int64_t)n1, (double)(big / N));
  emd_fill_kernel<<<c->num_sms, 256, 0, c->stream>>>(satr[0], (int64_t)n2, (double)(big / M));
  c->launches += 2;
  const dim3 grows((N + EM_WARPS - 1) / EM_WARPS, B), gcols((M + EM_WARPS - 1) / EM_WARPS, B);
  int cur = 0;
  for (int jl = 8; jl >= -2; --jl) {
    EmdJob j;
    j.xyz1 = d1; j.xyz2 = d2; j.satl = satl[cur]; j.satr = satr[cur]; j.satl_next = satl[cur ^ 1]; j.satr_next = satr[cur ^ 1];
    j.s = s; j.clip = clip; j.match = dmatch; j.n = N; j.m = M;
    j.level = jl == -2 ? 0.0 : -(double)powf(4.0f, (float)jl);
    emd_rows_kernel<0><<<grows, EM_THREADS, 0, c->stream>>>(j);
    emd_cols_kernel<1><<<gcols, EM_THREADS, 0, c->stream>>>(j);
    emd_rows_kernel<2><<<grows, EM_THREADS, 0, c->stream>>>(j);
    emd_cols_kernel<3><<<gcols, EM_THREADS, 0, c->stream>>>(j);
    c->launches += 4;
    cur ^= 1;
  }
  DISN_CUDA_OK(cudaGetLastError());
  if (cost_out) {
    if (match_cost_device(c, d1, d2, dmatch, B, N, M, rowcost, dcost)) return -1;
    DISN_CUDA_OK(cudaMemcpyAsync(cost_out, dcost, (size_t)B * 4, cudaMemcpyDeviceToHost, c->stream));
  }
  if (match_out) DISN_CUDA_OK(cudaMemcpyAsync(match_out, dmatch, nm * 4, cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" int disn_match_cost(disn_ctx* c, const float* xyz1, const float* xyz2, const float* match, int32_t B, int32_t N,
                               int32_t M, float* cost) {
  DISN_REQUIRE(c && xyz1 && xyz2 && match && cost, "null argument");
  DISN_REQUIRE(B >= 1 && N >= 1 && M >= 1 && B <= 65535, "MatchCost expects (batch_size,num_points,3) point sets, batch <= 65535");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  const size_t n1 = (size_t)B * N, n2 = (size_t)B * M, nm = (size_t)B * N * M;
  DevBuf buf;
  if (buf.reserve((n1 + n2) * 12 + nm * 4 + n1 * 8 + (size_t)B * 4 + 8 * 256)) return -1;
  float* d1 = buf.take<float>(n1 * 3);
  float* d2 = buf.take<float>(n2 * 3);
  float* dmatch = buf.take<float>(nm);
  double* rowcost = buf.take<double>(n1);
  float* dcost = buf.take<float>(B);
  DISN_CUDA_OK(cudaMemcpyAsync(d1, xyz1, n1 * 12, cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaMemcpyAsync(d2, xyz2, n2 * 12, cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaMemcpyAsync(dmatch, match, nm * 4, cudaMemcpyHostToDevice, c->stream));
  if (match_cost_device(c, d1, d2, dmatch, B, N, M, rowcost, dcost)) return -1;
  DISN_CUDA_OK(cudaMemcpyAsync(cost, dcost, (size_t)B * 4, cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}
