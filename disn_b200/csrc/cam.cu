// Camera-pose heads of the reference's estimated-camera path (the step that produces `trans_mat` when the drivers
// run with --cam_est: demo/demo.py:195-258, cam_est/model_cam.py:47-109, models/posenet.py:22-36,91-124).
// Input: the 1024-d VGG-16 embedding of the image (same encoder kernels as the SDF path, camera checkpoint's
// weights).  One CTA per image evaluates the three tiny fully-connected heads (utils/tf_util.py:328-362:
// y = relu(x.W + b), last layer linear), builds the rotation from the 6-D ortho representation, applies the
// predicted isotropic scale, appends the translation row and right-multiplies by K^T:
//     pred_RT[4,3] = [ (s*I).R ; t ],   pred_trans_mat[4,3] = pred_RT . K^T.
#include "common.cuh"

namespace disn {
namespace {

struct CamHeadWeights {
  const float *s1w, *s1b, *s2w, *s2b, *s3w, *s3b;      // scale: 1024-64-32-1
  const float *r1w, *r1b, *r2w, *r2b, *r3w, *r3b;      // ortho6d: 1024-512-256-6
  const float *t1w, *t1b, *t2w, *t2b, *t3w, *t3b;      // translation: 1024-128-64-3
};

// out[n] = act(b[n] + sum_k in[k] * W[k][n]); threads over n (coalesced rows of W)
__device__ void fc_layer(const float* in, int K, const float* __restrict__ W, const float* __restrict__ b, float* out,
                         int N, bool relu) {
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    float acc = 0.f;
    for (int k = 0; k < K; ++k) acc = fmaf(in[k], W[(size_t)k * N + n], acc);
    acc += b[n];
    out[n] = relu ? fmaxf(acc, 0.f) : acc;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(256) cam_heads_kernel(const float* __restrict__ emb, int emb_dim, CamHeadWeights w,
                                                        const float* __restrict__ Kmat /*[3,3]*/,
                                                        float* __restrict__ out_rt, float* __restrict__ out_tm) {
  __shared__ float x[1024], h1[512], h2[256], o_scale[1], o_rot[6], o_tr[3];
  const int b = blockIdx.x;
  for (int i = threadIdx.x; i < emb_dim; i += blockDim.x) x[i] = emb[(size_t)b * emb_dim + i];
  __syncthreads();
  fc_layer(x, emb_dim, w.s1w, w.s1b, h1, 64, true);
  fc_layer(h1, 64, w.s2w, w.s2b, h2, 32, true);
  fc_layer(h2, 32, w.s3w, w.s3b, o_scale, 1, false);
  fc_layer(x, emb_dim, w.r1w, w.r1b, h1, 512, true);
  fc_layer(h1, 512, w.r2w, w.r2b, h2, 256, true);
  fc_layer(h2, 256, w.r3w, w.r3b, o_rot, 6, false);
  fc_layer(x, emb_dim, w.t1w, w.t1b, h1, 128, true);
  fc_layer(h1, 128, w.t2w, w.t2b, h2, 64, true);
  fc_layer(h2, 64, w.t3w, w.t3b, o_tr, 3, false);
  if (threadIdx.x == 0) {
    // models/posenet.py:22-36 compute_rotation_matrix_from_ortho6d
    float xr[3] = {o_rot[0], o_rot[1], o_rot[2]}, yr[3] = {o_rot[3], o_rot[4], o_rot[5]};
    float n = fmaxf(sqrtf(xr[0] * xr[0] + xr[1] * xr[1] + xr[2] * xr[2]), 1e-8f);
    float xv[3] = {xr[0] / n, xr[1] / n, xr[2] / n};
    float z[3] = {xv[1] * yr[2] - xv[2] * yr[1], xv[2] * yr[0] - xv[0] * yr[2], xv[0] * yr[1] - xv[1] * yr[0]};
    n = fmaxf(sqrtf(z[0] * z[0] + z[1] * z[1] + z[2] * z[2]), 1e-8f);
    z[0] /= n; z[1] /= n; z[2] /= n;
    float yv[3] = {z[1] * xv[2] - z[2] * xv[1], z[2] * xv[0] - z[0] * xv[2], z[0] * xv[1] - z[1] * xv[0]};
    const float s = o_scale[0];
    float rt[4][3];
    for (int i = 0; i < 3; ++i) { rt[i][0] = s * xv[i]; rt[i][1] = s * yv[i]; rt[i][2] = s * z[i]; }   // columns x,y,z
    // models/posenet.py:118 translation offset constant
    rt[3][0] = o_tr[0] + (-0.00193892f); rt[3][1] = o_tr[1] + 0.00169222f; rt[3][2] = o_tr[2] + 1.3949631f;
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 3; ++j) {
        if (out_rt) out_rt[(size_t)b * 12 + i * 3 + j] = rt[i][j];
        float a = 0.f;                                       // (RT . K^T)[i][j] = sum_k RT[i][k] * K[j][k]
        for (int k = 0; k < 3; ++k) a = fmaf(rt[i][k], Kmat[j * 3 + k], a);
        out_tm[(size_t)b * 12 + i * 3 + j] = a;
      }
  }
}

}  // namespace

int launch_cam_heads(disn_ctx* c, int B, const float* d_K, float* d_rt, float* d_tm) {
  CamHeadWeights w;
  auto get = [&](const char* n, const float*& p) -> int {
    auto it = c->weights.find(std::string("cameraprediction/") + n);
    DISN_REQUIRE(it != c->weights.end(), std::string("missing variable cameraprediction/") + n);
    p = it->second.data.get<float>();
    return 0;
  };
  if (get("scale/fc1/weights", w.s1w) || get("scale/fc1/biases", w.s1b) || get("scale/fc2/weights", w.s2w) ||
      get("scale/fc2/biases", w.s2b) || get("scale/fc3/weights", w.s3w) || get("scale/fc3/biases", w.s3b) ||
      get("ortho6d/fc1/weights", w.r1w) || get("ortho6d/fc1/biases", w.r1b) || get("ortho6d/fc2/weights", w.r2w) ||
      get("ortho6d/fc2/biases", w.r2b) || get("ortho6d/fc3/weights", w.r3w) || get("ortho6d/fc3/biases", w.r3b) ||
      get("translation/fc1/weights", w.t1w) || get("translation/fc1/biases", w.t1b) ||
      get("translation/fc2/weights", w.t2w) || get("translation/fc2/biases", w.t2b) ||
      get("translation/fc3/weights", w.t3w) || get("translation/fc3/biases", w.t3b))
    return -2;
  DISN_REQUIRE(c->cfg.num_classes <= 1024, "camera heads expect an embedding of at most 1024");
  cam_heads_kernel<<<B, 256, 0, c->stream>>>(c->emb.get<float>(), c->cfg.num_classes, w, d_K, d_rt, d_tm);
  c->launches++;
  DISN_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace disn
