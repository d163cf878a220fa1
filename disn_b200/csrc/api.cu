// C ABI of the DISN B200 hot-path library (see include/disn_b200.h for the reference call sites).
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "common.cuh"

namespace disn {
static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
}  // namespace disn

using namespace disn;

extern "C" {

const char* disn_last_error(void) { return g_err.c_str(); }

void disn_default_config(disn_config* cfg) {
  if (!cfg) return;
  cfg->device = 0;
  cfg->img_h = 137; cfg->img_w = 137;
  cfg->vgg_in = 224;
  cfg->num_classes = 1024;
  cfg->clamp_max = 136.0f;
  cfg->sdf_weight = 10.0f;
  cfg->tanh_out = 0;
  cfg->precision = DISN_PREC_FP32;
  cfg->max_batch = 1;
}

int disn_create(const disn_config* cfg, disn_ctx** out) {
  DISN_REQUIRE(cfg && out, "null config/out");
  DISN_REQUIRE(cfg->max_batch >= 1 && cfg->max_batch <= 8, "max_batch in [1,8]");
  DISN_REQUIRE(cfg->img_h > 1 && cfg->img_w > 1 && cfg->num_classes % 4 == 0, "bad image/embedding size");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error(std::string("no CUDA device: the DISN B200 path has no CPU fallback (") + cudaGetErrorString(e) + ")");
    return -1;
  }
  DISN_REQUIRE(cfg->device >= 0 && cfg->device < ndev, "device ordinal out of range");
  DISN_CUDA_OK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  DISN_CUDA_OK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) {
    set_error("this library is built for sm_100a (B200) only; device is sm_" + std::to_string(prop.major) +
              std::to_string(prop.minor));
    return -1;
  }
  disn_ctx* c = new disn_ctx();
  c->cfg = *cfg;
  c->num_sms = prop.multiProcessorCount;
  DISN_CUDA_OK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  c->own_stream = true;
  if (c->d_tm.reserve(sizeof(float) * 12 * 8) || c->d_status.reserve(sizeof(int))) return -1;
  DISN_CUDA_OK(cudaMemset(c->d_status.get<int>(), 0, sizeof(int)));
  DISN_CUDA_OK(cudaMallocHost(&c->h_status, sizeof(int)));
  *c->h_status = 0;
  *out = c;
  return 0;
}

void disn_destroy(disn_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->cfg.device);
  cudaStreamSynchronize(c->stream);
  encoder_graph_reset(c);      // the captured graph holds the addresses of buffers `delete c` frees
  if (c->h_status) cudaFreeHost(c->h_status);
  if (c->mc_totals_host) cudaFreeHost(c->mc_totals_host);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

// Call after a synchronisation of c->stream: turns failure bits the kernels raised into a loud error.
static int check_status(disn_ctx* c) {
  const int st = *c->h_status;
  if (st == 0) return 0;
  *c->h_status = 0;
  cudaMemsetAsync(c->d_status.get<int>(), 0, sizeof(int), c->stream);
  if (st & DISN_STATUS_FP16_OVERFLOW) {
    set_error("DISN_PREC_F16F8: an MLP activation exceeded the fp16 range (65504); the result is invalid -- "
              "use DISN_PREC_BF16X3 (fp32 range) for these weights");
    return -4;
  }
  set_error("kernel reported status " + std::to_string(st));
  return -4;
}

int disn_set_stream(disn_ctx* c, void* cuda_stream) {
  DISN_REQUIRE(c, "null ctx");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  if (cuda_stream) {
    c->stream = (cudaStream_t)cuda_stream;
    c->own_stream = false;
  } else {
    DISN_CUDA_OK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    c->own_stream = true;
  }
  return 0;
}

int disn_synchronize(disn_ctx* c) {
  DISN_REQUIRE(c, "null ctx");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return check_status(c);     // asynchronous (DISN_DEVICE_PTR) launches report here
}

int disn_set_precision(disn_ctx* c, int32_t precision) {
  DISN_REQUIRE(c, "null ctx");
  DISN_REQUIRE(precision == DISN_PREC_FP32 || precision == DISN_PREC_BF16X3 || precision == DISN_PREC_F16F8,
               "unknown precision");
  c->cfg.precision = precision;
  return 0;
}

int64_t disn_launch_count(disn_ctx* c) { return c ? c->launches : 0; }

int disn_load_weight(disn_ctx* c, const char* name, const float* data, const int64_t* shape, int32_t ndim) {
  DISN_REQUIRE(c && name && data && shape && ndim >= 1 && ndim <= 4, "bad load_weight arguments");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  int64_t numel = 1;
  std::vector<int64_t> shp(shape, shape + ndim);
  for (int i = 0; i < ndim; ++i) { DISN_REQUIRE(shape[i] > 0, "non-positive dim"); numel *= shape[i]; }
  DevTensor& t = c->weights[name];
  if (t.numel != numel) {
    t.data.reset();
    if (t.data.reserve(numel * sizeof(float))) return -1;
  }
  t.shape = shp;
  t.numel = numel;
  DISN_CUDA_OK(cudaMemcpyAsync(t.data.get<float>(), data, numel * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));   // caller-owned host buffer; ordered on the ctx stream
  c->weights_dirty = true;
  c->enc_B = 0;     // encoder products (taps, gbias, pmap) belong to the previous weights: force a new disn_encode
  encoder_graph_reset(c);    // the graph replays launches that read the old packed images
  c->enc_tc_weights.clear();     // packed encoder weights follow the fp32 masters
  return 0;
}

static int check_shape(disn_ctx* c, const std::string& name, std::initializer_list<int64_t> want) {
  auto it = c->weights.find(name);
  DISN_REQUIRE(it != c->weights.end(), "missing variable " + name);
  std::vector<int64_t> w(want);
  // accept [1,1,Cin,Cout] or [Cin,Cout] for 1x1 convs
  const auto& s = it->second.shape;
  int64_t nw = 1, ns = 1;
  for (auto v : w) nw *= v;
  for (auto v : s) ns *= v;
  DISN_REQUIRE(nw == ns && s.back() == w.back(), "variable " + name + " has the wrong shape");
  return 0;
}

int disn_finalize_weights(disn_ctx* c) {
  DISN_REQUIRE(c, "null ctx");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  const int nc = c->cfg.num_classes;
  for (const char* sc : {"sdfprediction", "sdfprediction_imgfeat"}) {
    std::string p(sc);
    int64_t cat = (p == "sdfprediction") ? 512 + nc : 512 + kLocalFeat;
    if (check_shape(c, p + "/fold1/conv1/weights", {3, 64})) return -2;
    if (check_shape(c, p + "/fold1/conv2/weights", {64, 256})) return -2;
    if (check_shape(c, p + "/fold1/conv3/weights", {256, 512})) return -2;
    if (check_shape(c, p + "/fold2/conv1/weights", {cat, 512})) return -2;
    if (check_shape(c, p + "/fold2/conv2/weights", {512, 256})) return -2;
    if (check_shape(c, p + "/fold2/conv5/weights", {256, 1})) return -2;
    for (const char* l : {"fold1/conv1", "fold1/conv2", "fold1/conv3", "fold2/conv1", "fold2/conv2", "fold2/conv5"})
      DISN_REQUIRE(c->weights.count(p + "/" + l + "/biases"), "missing variable " + p + "/" + l + "/biases");
  }
  if (tc_pack_weights(c)) return -1;
  c->weights_dirty = false;
  return 0;
}

int disn_encode(disn_ctx* c, const float* imgs, int32_t B, int32_t H, int32_t W, int32_t C, uint32_t flags) {
  DISN_REQUIRE(c && imgs, "null ctx/imgs");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  DISN_REQUIRE(B <= c->cfg.max_batch, "batch exceeds max_batch of the context");
  if (c->weights_dirty && disn_finalize_weights(c)) return -1;
  if (encoder_run(c, imgs, B, H, W, C, (flags & DISN_DEVICE_PTR) != 0)) return -1;
  if (!(flags & DISN_DEVICE_PTR)) DISN_CUDA_OK(cudaStreamSynchronize(c->stream));   // caller-owned host buffer
  return 0;
}

int disn_get_encoded(disn_ctx* c, int32_t what, float* out, int64_t out_elems) {
  DISN_REQUIRE(c && out, "null ctx/out");
  DISN_REQUIRE(c->enc_B > 0, "disn_encode has not been called");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  static const int tapHW[5] = {224, 112, 56, 28, 14};
  const float* src = nullptr;
  int64_t n = 0, B = c->enc_B;
  if (what == 0) { src = c->emb.get<float>(); n = B * c->cfg.num_classes; }
  else if (what >= 1 && what <= 5) {
    src = c->taps[what - 1].get<float>();
    n = B * tapHW[what - 1] * tapHW[what - 1] * kTapC[what - 1];
  }
  else if (what == 6) { src = c->pmap.get<float>(); n = B * c->cfg.img_h * c->cfg.img_w * kHidden; }
  else if (what == 7) { src = c->gbias.get<float>(); n = B * kHidden; }
  else if (what == 8) { src = c->img_rs.get<float>(); n = B * c->cfg.vgg_in * c->cfg.vgg_in * 3; }
  DISN_REQUIRE(src, "unknown `what`");
  DISN_REQUIRE(out_elems == n, "output buffer has the wrong number of elements");
  DISN_CUDA_OK(cudaMemcpyAsync(out, src, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}

static const float* W(disn_ctx* c, const std::string& n) { return c->weights.at(n).data.get<float>(); }

static void fill_stream(disn_ctx* c, const std::string& p, StreamWeights& s) {
  s.w1 = W(c, p + "/fold1/conv1/weights"); s.b1 = W(c, p + "/fold1/conv1/biases");
  s.w2 = W(c, p + "/fold1/conv2/weights"); s.b2 = W(c, p + "/fold1/conv2/biases");
  s.w3 = W(c, p + "/fold1/conv3/weights"); s.b3 = W(c, p + "/fold1/conv3/biases");
  s.w4 = W(c, p + "/fold2/conv1/weights"); s.b4 = W(c, p + "/fold2/conv1/biases");
  s.w5 = W(c, p + "/fold2/conv2/weights"); s.b5 = W(c, p + "/fold2/conv2/biases");
  s.w6 = W(c, p + "/fold2/conv5/weights"); s.b6 = W(c, p + "/fold2/conv5/biases");
}

}  // extern "C"
int disn::ensure_point_scratch(disn_ctx* c, int64_t pts) {
  const size_t n = (size_t)pts * sizeof(float);
  return (c->d_pts.reserve(n * 3) || c->d_pts_rot.reserve(n * 3) || c->d_out.reserve(n) || c->d_uv.reserve(n * 2)) ? -1 : 0;
}

// Device-visible alias of a caller buffer that is pinned (cudaHostAlloc / cudaHostRegister / torch pin_memory), else
// nullptr.  With unified addressing the kernel epilogue can store its 4 B per point straight into such memory over PCIe
// (~1 GB/s at 2.5e8 points/s), so the host result needs no device scratch and no device->host copy after the kernel.
static float* pinned_alias(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  if (a.type == cudaMemoryTypeHost && a.devicePointer) return static_cast<float*>(a.devicePointer);
  return nullptr;
}

int disn::run_point_job(disn_ctx* c, PointJob& job) {
  if (!job.gbias) job.gbias = c->gbias.get<float>();
  if (!job.pmap) job.pmap = c->pmap.get<float>();
  job.img_h = c->cfg.img_h; job.img_w = c->cfg.img_w;
  job.clamp_max = c->cfg.clamp_max;
  job.tanh_out = c->cfg.tanh_out;
  fill_stream(c, "sdfprediction", job.g);
  fill_stream(c, "sdfprediction_imgfeat", job.l);
  job.status = c->d_status.get<int>();
  if (c->cfg.precision == DISN_PREC_FP32) return launch_point_fp32(c, job);
  if (launch_point_tc(c, job)) return -1;
  // the status word travels to the pinned mirror behind the kernel; whoever synchronises next checks it
  DISN_CUDA_OK(cudaMemcpyAsync(c->h_status, c->d_status.get<int>(), sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  return 0;
}

extern "C" {

int disn_eval_points(disn_ctx* c, const float* pts, const float* pts_rot, const float* trans_mat, int32_t B,
                     int64_t N, float* out_pred, float* out_uv, uint32_t flags) {
  DISN_REQUIRE(c && pts && trans_mat && out_pred, "null argument");
  DISN_REQUIRE(c->enc_B > 0, "disn_encode has not been called");
  DISN_REQUIRE(B == c->enc_B, "batch differs from the encoded batch");
  DISN_REQUIRE(N >= 0, "negative N");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  if (N == 0) return 0;
  PointJob job{};
  job.B = B; job.N = N; job.out_div = 1.0f;
  if (flags & DISN_DEVICE_PTR) {
    job.pts = pts; job.pts_rot = (pts_rot && pts_rot != pts) ? pts_rot : nullptr;
    job.trans_mat = trans_mat; job.out_pred = out_pred; job.out_uv = out_uv;
    return run_point_job(c, job);
  }
  if (ensure_point_scratch(c, (int64_t)B * N)) return -1;
  float* pred_alias = pinned_alias(out_pred);
  float* uv_alias = out_uv ? pinned_alias(out_uv) : nullptr;
  size_t nb = (size_t)B * N * 3 * sizeof(float);
  DISN_CUDA_OK(cudaMemcpyAsync(c->d_pts.get<float>(), pts, nb, cudaMemcpyHostToDevice, c->stream));
  job.pts = c->d_pts.get<float>();
  if (pts_rot && pts_rot != pts) {
    DISN_CUDA_OK(cudaMemcpyAsync(c->d_pts_rot.get<float>(), pts_rot, nb, cudaMemcpyHostToDevice, c->stream));
    job.pts_rot = c->d_pts_rot.get<float>();
  }
  DISN_CUDA_OK(cudaMemcpyAsync(c->d_tm.get<float>(), trans_mat, (size_t)B * 12 * sizeof(float), cudaMemcpyHostToDevice,
                               c->stream));
  job.trans_mat = c->d_tm.get<float>();
  job.out_pred = pred_alias ? pred_alias : c->d_out.get<float>();
  job.out_uv = out_uv ? (uv_alias ? uv_alias : c->d_uv.get<float>()) : nullptr;
  if (run_point_job(c, job)) return -1;
  if (!pred_alias)
    DISN_CUDA_OK(cudaMemcpyAsync(out_pred, job.out_pred, (size_t)B * N * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  if (out_uv && !uv_alias)
    DISN_CUDA_OK(cudaMemcpyAsync(out_uv, job.out_uv, (size_t)B * N * 2 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return check_status(c);
}

// numpy.linspace(start, stop, num) in float64, then cast to float32 (test/create_sdf.py:247-254):
// y[i] = start + i*step with step = (stop-start)/(num-1), last element forced to stop.
static void linspace_f32(double start, double stop, int num, float* out) {
  if (num == 1) { out[0] = (float)start; return; }
  const double div = (double)(num - 1);
  const double delta = stop - start;
  volatile double step = delta / div;
  for (int i = 0; i < num; ++i) {
    volatile double prod = (double)i * step;   // volatile: no FMA contraction, match numpy's two roundings
    out[i] = (float)(prod + start);
  }
  out[num - 1] = (float)stop;
}

int disn_eval_grid(disn_ctx* c, const double* sdf_params, const float* trans_mat, int32_t B, int32_t sdf_res,
                   int32_t z0, int32_t z1, float* out_sdf, uint32_t flags) {
  DISN_REQUIRE(c && sdf_params && trans_mat && out_sdf, "null argument");
  DISN_REQUIRE(c->enc_B > 0, "disn_encode has not been called");
  DISN_REQUIRE(B == c->enc_B, "batch differs from the encoded batch");
  DISN_REQUIRE(sdf_res >= 1, "sdf_res >= 1");
  const int R = sdf_res + 1;
  DISN_REQUIRE(z0 >= 0 && z1 <= R && z0 <= z1, "z range outside [0, sdf_res+1]");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  const int64_t N = (int64_t)(z1 - z0) * R * R;
  if (N == 0) return 0;
  // axis tables (host float64 linspace -> float32), uploaded per call: B*3*R floats
  const size_t axes_bytes = (size_t)8 * 3 * R * sizeof(float);
  if (c->d_axes.bytes() < axes_bytes) {
    c->axes_key.clear();
    if (c->d_axes.reserve(axes_bytes)) return -1;
  }
  // re-upload only when the boxes / resolution change (keeps repeated calls free of host syncs)
  std::vector<double> key(sdf_params, sdf_params + (size_t)B * 6);
  key.push_back((double)R);
  if (key != c->axes_key) {
    std::vector<float> axes((size_t)B * 3 * R);
    for (int b = 0; b < B; ++b)
      for (int a = 0; a < 3; ++a)
        linspace_f32(sdf_params[b * 6 + a], sdf_params[b * 6 + 3 + a], R, &axes[((size_t)b * 3 + a) * R]);
    DISN_CUDA_OK(cudaMemcpyAsync(c->d_axes.get<float>(), axes.data(), axes.size() * sizeof(float), cudaMemcpyHostToDevice,
                                 c->stream));
    DISN_CUDA_OK(cudaStreamSynchronize(c->stream));   // `axes` is a stack-owned staging buffer
    c->axes_key = key;
  }

  PointJob job{};
  job.B = B; job.N = N; job.R = R; job.z0 = z0; job.axes = c->d_axes.get<float>();
  job.out_div = c->cfg.sdf_weight;   // correctly rounded r / 10 like the reference's float64 divide + float32 pack (create_sdf.py:285,299)
  if (flags & DISN_DEVICE_PTR) {
    job.trans_mat = trans_mat;
    job.out_pred = out_sdf;
    return run_point_job(c, job);
  }
  DISN_CUDA_OK(cudaMemcpyAsync(c->d_tm.get<float>(), trans_mat, (size_t)B * 12 * sizeof(float), cudaMemcpyHostToDevice,
                               c->stream));
  job.trans_mat = c->d_tm.get<float>();
  if (float* alias = pinned_alias(out_sdf)) {     // pinned caller buffer: the kernel writes the host grid directly
    job.out_pred = alias;
    if (run_point_job(c, job)) return -1;
    DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
    return check_status(c);
  }
  if (ensure_point_scratch(c, (int64_t)B * N)) return -1;
  job.out_pred = c->d_out.get<float>();
  if (run_point_job(c, job)) return -1;
  DISN_CUDA_OK(cudaMemcpyAsync(out_sdf, job.out_pred, (size_t)B * N * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return check_status(c);
}

int disn_write_dist(const char* path, int32_t res, const double* bbox, const float* values) {
  DISN_REQUIRE(path && bbox && values && res >= 1, "bad write_dist arguments");
  FILE* f = fopen(path, "wb");
  if (!f) { set_error(std::string("cannot open ") + path); return -3; }
  int32_t hdr[3] = {-res, res, res};
  const size_t n = (size_t)(res + 1) * (res + 1) * (res + 1);
  bool ok = fwrite(hdr, sizeof(int32_t), 3, f) == 3 && fwrite(bbox, sizeof(double), 6, f) == 6 &&
            fwrite(values, sizeof(float), n, f) == n;
  ok = (fclose(f) == 0) && ok;
  if (!ok) { set_error(std::string("short write to ") + path); return -3; }
  return 0;
}

int disn_cam_estimate(disn_ctx* c, const float* imgs, int32_t B, int32_t H, int32_t W, int32_t C, const float* K,
                      float* out_rt, float* out_trans_mat) {
  DISN_REQUIRE(c && imgs && out_trans_mat, "null argument");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  DISN_REQUIRE(B >= 1 && B <= c->cfg.max_batch, "batch exceeds max_batch of the context");
  if (encoder_run(c, imgs, B, H, W, C, false, /*embedding_only=*/true)) return -1;
  static const float kDefaultK[9] = {149.84375f, 0.f, 68.5f, 0.f, 149.84375f, 68.5f, 0.f, 0.f, 1.f};
  if (c->staging.reserve((9 + (size_t)B * 12 * 2) * 4 + 3 * 256)) return -1;
  float* dK = c->staging.take<float>(9);
  float* dRT = c->staging.take<float>((size_t)B * 12);
  float* dTM = c->staging.take<float>((size_t)B * 12);
  DISN_CUDA_OK(cudaMemcpyAsync(dK, K ? K : kDefaultK, 9 * 4, cudaMemcpyHostToDevice, c->stream));
  if (launch_cam_heads(c, B, dK, dRT, dTM)) return -1;
  if (out_rt) DISN_CUDA_OK(cudaMemcpyAsync(out_rt, dRT, (size_t)B * 12 * 4, cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaMemcpyAsync(out_trans_mat, dTM, (size_t)B * 12 * 4, cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}

int disn_nn_distance(disn_ctx* c, const float* xyz1, const float* xyz2, int32_t B, int32_t N, int32_t M, float* dist1,
                     int32_t* idx1, float* dist2, int32_t* idx2) {
  DISN_REQUIRE(c && xyz1 && xyz2 && dist1 && idx1 && dist2 && idx2, "null argument");
  DISN_REQUIRE(B >= 1 && N >= 1 && M >= 1, "NnDistance requires non-empty point sets of shape (batch,#points,3)");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  const size_t n1 = (size_t)B * N, n2 = (size_t)B * M;
  if (c->staging.reserve((n1 + n2) * (3 + 1 + 1) * 4 + 6 * 256)) return -1;
  float* d1 = c->staging.take<float>(n1 * 3);
  float* d2 = c->staging.take<float>(n2 * 3);
  float* o1 = c->staging.take<float>(n1);
  float* o2 = c->staging.take<float>(n2);
  int* i1 = c->staging.take<int>(n1);
  int* i2 = c->staging.take<int>(n2);
  DISN_CUDA_OK(cudaMemcpyAsync(d1, xyz1, n1 * 3 * 4, cudaMemcpyHostToDevice, c->stream));
  DISN_CUDA_OK(cudaMemcpyAsync(d2, xyz2, n2 * 3 * 4, cudaMemcpyHostToDevice, c->stream));
  if (nn_distance(c, d1, N, d2, M, B, o1, i1, o2, i2)) return -1;
  DISN_CUDA_OK(cudaMemcpyAsync(dist1, o1, n1 * 4, cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaMemcpyAsync(idx1, i1, n1 * 4, cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaMemcpyAsync(dist2, o2, n2 * 4, cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaMemcpyAsync(idx2, i2, n2 * 4, cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return 0;
}

int disn_write_obj(const char* path, const float* verts, int64_t n_verts, const int32_t* faces, int64_t n_faces) {
  DISN_REQUIRE(path && (verts || n_verts == 0) && (faces || n_faces == 0) && n_verts >= 0 && n_faces >= 0,
               "bad write_obj arguments");
  FILE* f = fopen(path, "w");
  if (!f) { set_error(std::string("cannot open ") + path); return -3; }
  std::vector<char> buf(1 << 20);
  setvbuf(f, buf.data(), _IOFBF, buf.size());
  fprintf(f, "# Generated by the DISN B200 marching-cubes post-pass\n# Number of vertices: %lld\n# Number of faces: %lld\n",
          (long long)n_verts, (long long)n_faces);
  for (int64_t i = 0; i < n_verts; ++i) fprintf(f, "v %g %g %g\n", verts[3 * i], verts[3 * i + 1], verts[3 * i + 2]);
  for (int64_t i = 0; i < n_faces; ++i)
    fprintf(f, "f %d %d %d\n", faces[3 * i] + 1, faces[3 * i + 1] + 1, faces[3 * i + 2] + 1);
  bool ok = !ferror(f);
  ok = (fclose(f) == 0) && ok;
  if (!ok) { set_error(std::string("short write to ") + path); return -3; }
  return 0;
}

// staging of a host SDF grid for marching cubes (persistent, grows)
static int mc_input(disn_ctx* c, const float* sdf, int32_t R, uint32_t flags, const float** d_sdf) {
  if (flags & DISN_DEVICE_PTR) { *d_sdf = sdf; return 0; }
  const size_t bytes = (size_t)R * R * R * sizeof(float);
  if (c->d_mc_in.reserve(bytes)) return -1;
  DISN_CUDA_OK(cudaMemcpyAsync(c->d_mc_in.get<float>(), sdf, bytes, cudaMemcpyHostToDevice, c->stream));
  *d_sdf = c->d_mc_in.get<float>();
  return 0;
}

int disn_mc_run(disn_ctx* c, const float* sdf, int32_t R, const double* bbox, float iso, uint32_t flags,
                int64_t* n_verts, int64_t* n_faces) {
  DISN_REQUIRE(c && sdf && bbox, "null argument");
  DISN_REQUIRE(R >= 2, "need at least 2 samples per axis");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  const float* d_sdf = nullptr;
  if (mc_input(c, sdf, R, flags, &d_sdf)) return -1;
  return mc_run(c, d_sdf, R, bbox, iso, n_verts, n_faces);
}

int disn_mc_fetch(disn_ctx* c, float* verts, int32_t* faces) {
  DISN_REQUIRE(c, "null ctx");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  return mc_fetch(c, verts, faces);
}

int disn_mc_write_obj(disn_ctx* c, const char* path) {
  DISN_REQUIRE(c && path, "null argument");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  std::vector<float> v((size_t)c->mc_nv * 3);
  std::vector<int32_t> f((size_t)c->mc_nf * 3);
  if (mc_fetch(c, v.data(), f.data())) return -1;
  return disn_write_obj(path, v.data(), c->mc_nv, f.data(), c->mc_nf);
}

int disn_marching_cubes(disn_ctx* c, const float* sdf, int32_t R, const double* bbox, float iso, float* verts,
                        int64_t* n_verts, int32_t* faces, int64_t* n_faces, uint32_t flags) {
  DISN_REQUIRE(c && sdf && bbox && n_verts && n_faces, "null argument");
  int64_t nv = 0, nf = 0;
  const int rc = disn_mc_run(c, sdf, R, bbox, iso, flags, &nv, &nf);
  if (rc) return rc;
  if (verts == nullptr || faces == nullptr) { *n_verts = nv; *n_faces = nf; return 0; }     // counting call
  if (*n_verts < nv || *n_faces < nf) { set_error("marching_cubes: output buffers too small"); return -2; }
  *n_verts = nv; *n_faces = nf;
  return mc_fetch(c, verts, faces);
}

int disn_eval_grid_resident(disn_ctx* c, const double* sdf_params, const float* trans_mat, int32_t B, int32_t sdf_res,
                            float** out_dev) {
  DISN_REQUIRE(c && sdf_params && trans_mat && out_dev, "null argument");
  DISN_REQUIRE(sdf_res >= 1 && B >= 1, "sdf_res >= 1, B >= 1");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  const int R = sdf_res + 1;
  if (c->d_grid.reserve((size_t)B * R * R * R * sizeof(float))) return -1;
  float* d_tm = c->d_tm.get<float>();
  DISN_CUDA_OK(cudaMemcpyAsync(d_tm, trans_mat, (size_t)B * 12 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  const int rc = disn_eval_grid(c, sdf_params, d_tm, B, sdf_res, 0, R, c->d_grid.get<float>(), DISN_DEVICE_PTR);
  if (rc) return rc;
  *out_dev = c->d_grid.get<float>();
  return 0;
}

// ---- cross-process device buffers (multi-GPU gather without a collective) -------------------------------------------
// Rank 0 allocates the whole-grid buffer and exports a CUDA IPC handle; the other ranks (one process per GPU) open it and
// pass `ptr + slab offset` as the DISN_DEVICE_PTR output of disn_eval_grid, so the kernel's epilogue stores every
// SDF value straight into rank 0's HBM over NVLink (peer stores) while it computes: compute and gather are one kernel.
int disn_shared_alloc(disn_ctx* c, int64_t bytes, void** dev_ptr, unsigned char* handle64) {
  DISN_REQUIRE(c && dev_ptr && handle64 && bytes > 0, "bad shared_alloc arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  void* p = nullptr;
  DISN_CUDA_OK(cudaMalloc(&p, (size_t)bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); set_error(std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e)); return -1; }
  memcpy(handle64, &h, 64);
  *dev_ptr = p;
  return 0;
}

int disn_shared_open(disn_ctx* c, const unsigned char* handle64, void** dev_ptr) {
  DISN_REQUIRE(c && handle64 && dev_ptr, "bad shared_open arguments");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  DISN_CUDA_OK(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}

int disn_shared_close(disn_ctx* c, void* dev_ptr, int32_t owner) {
  DISN_REQUIRE(c && dev_ptr, "bad shared_close arguments");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  if (owner) DISN_CUDA_OK(cudaFree(dev_ptr));
  else DISN_CUDA_OK(cudaIpcCloseMemHandle(dev_ptr));
  return 0;
}

int disn_fetch(disn_ctx* c, const void* dev, void* host, int64_t bytes) {
  DISN_REQUIRE(c && dev && host && bytes >= 0, "bad fetch arguments");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  DISN_CUDA_OK(cudaMemcpyAsync(host, dev, (size_t)bytes, cudaMemcpyDeviceToHost, c->stream));
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  return check_status(c);
}

}  // extern "C"
