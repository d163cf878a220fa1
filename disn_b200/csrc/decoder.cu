// The reference's encoder/decoder split point and its graph intermediates (models/model_normalization.py:38-45,
// 169-190,223-238), for callers that fetch or feed them.  NOT the hot path: the fused kernels never materialise the
// per-point [N,1472] feature (that is the point of the design); these entry points exist so that
//   * end_points['point_img_feat'], ['pred_sdf_value_global'], ['pred_sdf_value_local'] can be fetched (Session.run), and
//   * get_decoder(num_point, input_pls, feature_pls) -- explicit [B,1,1,1024] / [B,N,1,1472] features in -- can be run:
//     global feature -> folded bias (GEMV), point features -> [N,512] through W[512:1984] (GEMM, the same linear fold the
//     encoder applies to the maps), then the ordinary point kernel with `pfeat` in place of the map gather.
#include <algorithm>

#include "common.cuh"

namespace disn {
namespace {

struct TapLevels { const float* p[5]; int h[5]; int c[5]; int coff[5]; };

// out[b,n, coff_l + c] = resampler( tf_resize_bilinear(tap_l -> OHxOW), uv[b,n] )     (model_normalization.py:171-189)
// one thread = one (point, level, float4 of channels); TF-legacy resize (scale = in/out, no half-pixel) of the four
// resampler neighbours, then the contrib resampler's four-tap sum (zero outside the map)
__global__ void point_img_feat_kernel(TapLevels lv, const float* __restrict__ uv, float* __restrict__ out, int B, int64_t N,
                                      int OH, int OW, int C4total) {
  const int64_t total = (int64_t)B * N * C4total;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c4 = (int)(i % C4total);
    const int64_t pn = i / C4total;
    const int b = (int)(pn / N);
    int l = 0;
    while (l < 4 && c4 * 4 >= lv.coff[l + 1]) ++l;
    const int ch = c4 * 4 - lv.coff[l];
    const int h = lv.h[l], C = lv.c[l];
    const float* tap = lv.p[l] + (int64_t)b * h * h * C + ch;
    const float x = uv[pn * 2], y = uv[pn * 2 + 1];
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (x > -1.f && y > -1.f && x < (float)OW && y < (float)OH) {
      const int fx = (int)floorf(x), fy = (int)floorf(y);
      const int cx = fx + 1, cy = fy + 1;
      const float dx = (float)cx - x, dy = (float)cy - y;
      const int tx[4] = {fx, cx, fx, cx}, ty[4] = {fy, cy, cy, fy};
      const float wg[4] = {dx * dy, (1.f - dx) * (1.f - dy), dx * (1.f - dy), (1.f - dx) * dy};
      const float sy = (float)h / (float)OH, sx = (float)h / (float)OW;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        if (tx[t] < 0 || tx[t] >= OW || ty[t] < 0 || ty[t] >= OH) continue;
        // pixel (ty,tx) of the resized map
        const float fyy = __fmul_rn((float)ty[t], sy), fxx = __fmul_rn((float)tx[t], sx);
        const int y0 = (int)floorf(fyy), x0 = (int)floorf(fxx);
        const int y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, h - 1);
        const float ly = __fsub_rn(fyy, (float)y0), lx = __fsub_rn(fxx, (float)x0);
        const float4 tl = *reinterpret_cast<const float4*>(tap + ((int64_t)y0 * h + x0) * C);
        const float4 tr = *reinterpret_cast<const float4*>(tap + ((int64_t)y0 * h + x1) * C);
        const float4 bl = *reinterpret_cast<const float4*>(tap + ((int64_t)y1 * h + x0) * C);
        const float4 br = *reinterpret_cast<const float4*>(tap + ((int64_t)y1 * h + x1) * C);
#define DISN_RS(f)                                           \
  {                                                          \
    const float top = tl.f + (tr.f - tl.f) * lx;             \
    const float bot = bl.f + (br.f - bl.f) * lx;             \
    acc.f += wg[t] * (top + (bot - top) * ly);               \
  }
        DISN_RS(x) DISN_RS(y) DISN_RS(z) DISN_RS(w)
#undef DISN_RS
      }
    }
    *reinterpret_cast<float4*>(out + pn * (int64_t)(C4total * 4) + c4 * 4) = acc;
  }
}

// models/model_normalization.py:241-251
__global__ void img_points_kernel(const float* __restrict__ pts, const float* __restrict__ tm, float* __restrict__ uv, int B,
                                  int64_t N, float clamp_max) {
  const int64_t total = (int64_t)B * N;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const float* T = tm + (i / N) * 12;
    const float x = pts[i * 3], y = pts[i * 3 + 1], z = pts[i * 3 + 2];
    const float q0 = fmaf(z, T[6], fmaf(y, T[3], x * T[0])) + T[9];
    const float q1 = fmaf(z, T[7], fmaf(y, T[4], x * T[1])) + T[10];
    const float q2 = fmaf(z, T[8], fmaf(y, T[5], x * T[2])) + T[11];
    uv[i * 2] = fminf(clamp_max, fmaxf(0.f, q0 / q2));
    uv[i * 2 + 1] = fminf(clamp_max, fmaxf(0.f, q1 / q2));
  }
}

}  // namespace
}  // namespace disn

using namespace disn;

extern "C" {

// end_points['point_img_feat'] (models/model_normalization.py:171-190): pts [B,N,3], trans_mat [B,4,3] host ->
// out_feat [B,N,1472] host (concat order conv1..conv5), out_uv [B,N,2] host or NULL.  Needs a prior disn_encode.
int disn_point_img_feat(disn_ctx* c, const float* pts, const float* trans_mat, int32_t B, int64_t N, float* out_feat,
                        float* out_uv) {
  DISN_REQUIRE(c && pts && trans_mat && out_feat, "null argument");
  DISN_REQUIRE(c->enc_B > 0, "disn_encode has not been called");
  DISN_REQUIRE(B == c->enc_B, "batch differs from the encoded batch");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  if (N <= 0) return 0;
  static const int tapHW[5] = {224, 112, 56, 28, 14};
  const int64_t n = (int64_t)B * N;
  if (c->staging.reserve((size_t)n * (3 + 2 + kLocalFeat) * 4 + 3 * 256)) return -1;
  float* d_pts = c->staging.take<float>(n * 3);
  float* d_uv = c->staging.take<float>(n * 2);
  float* d_feat = c->staging.take<float>(n * kLocalFeat);
  DISN_CUDA_OK(cudaMemcpyAsync(d_pts, pts, (size_t)n * 3 * 4, cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaMemcpyAsync(c->d_tm.get<float>(), trans_mat, (size_t)B * 12 * 4, cudaMemcpyHostToDevice, c->stream));
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, (int64_t)c->num_sms * 8);
  img_points_kernel<<<blocks, 256, 0, c->stream>>>(d_pts, c->d_tm.get<float>(), d_uv, B, N, c->cfg.clamp_max);
  TapLevels lv;
  int off = 0;
  for (int l = 0; l < 5; ++l) {
    lv.p[l] = c->taps[l].get<float>(); lv.h[l] = tapHW[l]; lv.c[l] = kTapC[l]; lv.coff[l] = off; off += kTapC[l];
  }
  const int64_t total = n * (kLocalFeat / 4);
  const int blocks2 = (int)std::min<int64_t>((total + 255) / 256, (int64_t)c->num_sms * 16);
  point_img_feat_kernel<<<blocks2, 256, 0, c->stream>>>(lv, d_uv, d_feat, B, N, c->cfg.img_h, c->cfg.img_w, kLocalFeat / 4);
  c->launches += 2;
  DISN_CUDA_OK(cudaGetLastError());
  DISN_CUDA_OK(cudaMemcpyAsync(out_feat, d_feat, (size_t)n * kLocalFeat * 4, cudaMemcpyDeviceToHost, c->stream));
  if (out_uv) DISN_CUDA_OK(cudaMemcpyAsync(out_uv, d_uv, (size_t)n * 2 * 4, cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}

// disn_eval_points plus the two stream outputs (end_points['pred_sdf_value_global'/'_local'], model_normalization.py:
// 194-204): out_global / out_local [B,N,1] host or NULL.  Host pointers only.
int disn_eval_points_ex(disn_ctx* c, const float* pts, const float* pts_rot, const float* trans_mat, int32_t B, int64_t N,
                        float* out_pred, float* out_uv, float* out_global, float* out_local) {
  DISN_REQUIRE(c && pts && trans_mat && out_pred, "null argument");
  DISN_REQUIRE(c->enc_B > 0, "disn_encode has not been called");
  DISN_REQUIRE(B == c->enc_B, "batch differs from the encoded batch");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  if (N <= 0) return 0;
  const int64_t n = (int64_t)B * N;
  if (ensure_point_scratch(c, n)) return -1;
  if (c->staging.reserve((size_t)n * 2 * 4 + 2 * 256)) return -1;
  float* d_g = c->staging.take<float>(n);
  float* d_l = c->staging.take<float>(n);
  PointJob job{};
  job.B = B; job.N = N; job.out_div = 1.0f;
  DISN_CUDA_OK(cudaMemcpyAsync(c->d_pts.get<float>(), pts, (size_t)n * 12, cudaMemcpyHostToDevice, c->stream));
  job.pts = c->d_pts.get<float>();
  if (pts_rot && pts_rot != pts) {
    DISN_CUDA_OK(cudaMemcpyAsync(c->d_pts_rot.get<float>(), pts_rot, (size_t)n * 12, cudaMemcpyHostToDevice, c->stream));
    job.pts_rot = c->d_pts_rot.get<float>();
  }
  DISN_CUDA_OK(cudaMemcpyAsync(c->d_tm.get<float>(), trans_mat, (size_t)B * 48, cudaMemcpyHostToDevice, c->stream));
  job.trans_mat = c->d_tm.get<float>();
  job.out_pred = c->d_out.get<float>();
  job.out_uv = out_uv ? c->d_uv.get<float>() : nullptr;
  job.out_global = out_global ? d_g : nullptr;
  job.out_local = out_local ? d_l : nullptr;
  if (run_point_job(c, job)) return -1;
  DISN_CUDA_OK(cudaMemcpyAsync(out_pred, c->d_out.get<float>(), (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (out_uv) DISN_CUDA_OK(cudaMemcpyAsync(out_uv, c->d_uv.get<float>(), (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
  if (out_global) DISN_CUDA_OK(cudaMemcpyAsync(out_global, d_g, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (out_local) DISN_CUDA_OK(cudaMemcpyAsync(out_local, d_l, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return disn_synchronize(c);      // surfaces a kernel status bit (fp16 overflow) as an error
}

// get_decoder (models/model_normalization.py:223-238): pts_rot [B,N,3], global_feat [B,1024] (the [B,1,1,1024]
// placeholder), point_feat [B,N,1472] (the [B,N,1,1472] placeholder), all host -> out_pred [B,N,1] = global + local
// (no tanh, no /sdf_weight: the reference's decoder returns the raw sum), out_global / out_local or NULL.
// Needs the weights only (no disn_encode).  B <= max_batch, B*N*512 < 2^31.
int disn_eval_features(disn_ctx* c, const float* pts_rot, const float* global_feat, const float* point_feat, int32_t B,
                       int64_t N, float* out_pred, float* out_global, float* out_local, uint32_t flags) {
  DISN_REQUIRE(c && pts_rot && global_feat && point_feat && out_pred, "null argument");
  DISN_REQUIRE(flags == 0, "host pointers only");
  DISN_REQUIRE(B >= 1 && B <= 8 && N >= 1, "B in [1,8], N >= 1");
  DISN_REQUIRE((int64_t)B * N * kHidden < ((int64_t)1 << 31), "B*N too large for the explicit-feature path");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  if (c->weights_dirty && disn_finalize_weights(c)) return -1;
  const int nc = c->cfg.num_classes;
  const int64_t n = (int64_t)B * N;
  if (ensure_point_scratch(c, n)) return -1;
  if (c->staging.reserve(((size_t)n * (kLocalFeat + kHidden + 2) + (size_t)B * (nc + kHidden)) * 4 + 6 * 256)) return -1;
  float* d_feat = c->staging.take<float>(n * kLocalFeat);
  float* d_pf = c->staging.take<float>(n * kHidden);
  float* d_gf = c->staging.take<float>((size_t)B * nc);
  float* d_gb = c->staging.take<float>((size_t)B * kHidden);
  float* d_g = c->staging.take<float>(n);
  float* d_l = c->staging.take<float>(n);
  DISN_CUDA_OK(cudaMemcpyAsync(d_feat, point_feat, (size_t)n * kLocalFeat * 4, cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaMemcpyAsync(d_gf, global_feat, (size_t)B * nc * 4, cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaMemcpyAsync(c->d_pts.get<float>(), pts_rot, (size_t)n * 12, cudaMemcpyHostToDevice, c->stream));
  const float* wg = c->weights.at("sdfprediction/fold2/conv1/weights").data.get<float>();
  const float* bg = c->weights.at("sdfprediction/fold2/conv1/biases").data.get<float>();
  const float* wl = c->weights.at("sdfprediction_imgfeat/fold2/conv1/weights").data.get<float>();
  // global stream: gbias = g . Wg[512:512+nc] + b      (models/sdfnet.py:78-85)
  if (encoder_gemv(c, d_gf, wg + (int64_t)kHidden * kHidden, bg, d_gb, B, nc, kHidden, 0)) return -1;
  // local stream: pfeat = feat . Wl[512:1984]          (models/sdfnet.py:180-183; bias added in the point kernel)
  if (encoder_gemm_plain(c, "decoder_proj", d_feat, wl + (int64_t)kHidden * kHidden, nullptr, d_pf, (int)n, kHidden,
                         kLocalFeat, 0))
    return -1;
  static const float kIdentityish[12] = {1, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1};   // q2 = 1: the unused projection stays finite
  float tm[8 * 12];
  for (int b = 0; b < B; ++b) memcpy(tm + b * 12, kIdentityish, sizeof(kIdentityish));
  DISN_CUDA_OK(cudaMemcpyAsync(c->d_tm.get<float>(), tm, (size_t)B * 48, cudaMemcpyHostToDevice, c->stream));
  PointJob job{};
  job.B = B; job.N = N; job.out_div = 1.0f;
  job.pts = c->d_pts.get<float>();
  job.trans_mat = c->d_tm.get<float>();
  job.gbias = d_gb;
  job.pmap = d_pf;            // never dereferenced in pfeat mode
  job.pfeat = d_pf;
  job.out_pred = c->d_out.get<float>();
  job.out_global = out_global ? d_g : nullptr;
  job.out_local = out_local ? d_l : nullptr;
  const int saved_tanh = c->cfg.tanh_out;
  c->cfg.tanh_out = 0;
  const int rc = run_point_job(c, job);
  c->cfg.tanh_out = saved_tanh;
  if (rc) return -1;
  DISN_CUDA_OK(cudaMemcpyAsync(out_pred, c->d_out.get<float>(), (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (out_global) DISN_CUDA_OK(cudaMemcpyAsync(out_global, d_g, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (out_local) DISN_CUDA_OK(cudaMemcpyAsync(out_local, d_l, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  return disn_synchronize(c);
}

}  // extern "C"
