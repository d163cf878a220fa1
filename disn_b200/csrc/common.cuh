// Shared declarations for the DISN B200 library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <set>
#include <string>
#include <utility>
#include <vector>

#include "../../include/disn_b200.h"

namespace disn {

void set_error(const std::string& msg);

#define DISN_CUDA_OK(expr)                                                                   \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      ::disn::set_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + " at " + \
                        __FILE__ + ":" + std::to_string(__LINE__));                          \
      return -1;                                                                             \
    }                                                                                        \
  } while (0)

#define DISN_REQUIRE(cond, msg)                          \
  do {                                                   \
    if (!(cond)) {                                       \
      ::disn::set_error(std::string("invalid argument: ") + (msg)); \
      return -2;                                         \
    }                                                    \
  } while (0)

// Sole owner of one cudaMalloc block (move-only; freed by the destructor).  take<T>() carves consecutive 256-byte-aligned
// arrays off the block, starting at its base after every reserve(); each array wastes under 256 bytes of padding, so a
// block carved into k arrays needs their total size plus k * 256 bytes.
class DevBuf {
 public:
  DevBuf() = default;
  DevBuf(DevBuf&& o) noexcept { *this = std::move(o); }
  DevBuf& operator=(DevBuf&& o) noexcept {
    std::swap(p_, o.p_); std::swap(bytes_, o.bytes_); std::swap(used_, o.used_);
    return *this;
  }
  ~DevBuf() { reset(); }

  // Grow-only: a block of at least `bytes` keeps its contents, a smaller one is replaced by exactly `bytes` (contents
  // lost).  On failure the buffer is left empty, the error recorded, and -1 returned.
  int reserve(size_t bytes) {
    used_ = 0;
    if (bytes <= bytes_) return 0;
    reset();
    const cudaError_t e = cudaMalloc(&p_, bytes);
    if (e != cudaSuccess) {
      p_ = nullptr;
      set_error("cudaMalloc of " + std::to_string(bytes) + " bytes failed: " + cudaGetErrorString(e));
      return -1;
    }
    bytes_ = bytes;
    return 0;
  }
  void reset() {
    if (p_) cudaFree(p_);
    p_ = nullptr;
    bytes_ = used_ = 0;
  }
  size_t bytes() const { return bytes_; }
  template <class T> T* get() const { return static_cast<T*>(p_); }
  template <class T> T* take(size_t count) {
    T* r = reinterpret_cast<T*>(static_cast<char*>(p_) + used_);
    used_ += (count * sizeof(T) + 255) / 256 * 256;
    return r;
  }

 private:
  void* p_ = nullptr;
  size_t bytes_ = 0, used_ = 0;
};

struct DevTensor {
  DevBuf data;
  std::vector<int64_t> shape;
  int64_t numel = 0;
};

// VGG-16 topology (reference spec: models/CNN/vgg.py:187-196)
static const int kNumConv = 13;
static const int kTapLayer[5] = {1, 3, 6, 9, 12};  // conv1_2, conv2_2, conv3_3, conv4_3, conv5_3
static const int kTapC[5] = {64, 128, 256, 512, 512};
static const int kLocalFeat = 1472;
static const int kHidden = 512;

// One stream of the point MLP (models/sdfnet.py:69-92 / :171-190) after the algebraic folds.
struct StreamWeights {
  const float* w1; const float* b1;   // fold1/conv1 [3,64]
  const float* w2; const float* b2;   // fold1/conv2 [64,256]
  const float* w3; const float* b3;   // fold1/conv3 [256,512]
  const float* w4;                    // fold2/conv1 rows 0..511 [512,512] (point-feature part)
  const float* b4;                    // fold2/conv1 biases [512] (local stream; global uses gbias)
  const float* w5; const float* b5;   // fold2/conv2 [512,256]
  const float* w6; const float* b6;   // fold2/conv5 [256,1]
};

struct PointJob {
  // inputs
  const float* pts;       // [B,N,3] or nullptr (grid mode)
  const float* pts_rot;   // [B,N,3] or nullptr (= pts)
  const float* trans_mat; // [B,4,3] device
  const float* axes;      // grid mode: [B,3,R] float32 linspace tables (x,y,z)
  int32_t R;              // grid mode: points per axis
  int32_t z0;             // grid mode: first z plane
  int64_t N;              // points per image in this call
  int32_t B;
  // per-image encoder products
  const float* gbias;     // [B,512]
  const float* pmap;      // [B,img_h,img_w,512]
  const float* pfeat;     // explicit-feature decoder (get_decoder): [B,N,512] per-point folded local features replace the
                          // gather of pmap; nullptr on the fused path
  int32_t img_h, img_w;
  float clamp_max;
  float out_div;          // result divisor: 1 (eval_points) or sdf_weight (eval_grid)
  int32_t tanh_out;
  StreamWeights g, l;
  // DISN_PREC_F16F8: power-of-two multipliers of the e5m2 correction operands, [stream][layer]{(a-h(a)) scale, a scale}
  float act_scale[2][4][2];
  // outputs
  float* out_pred;        // [B,N]
  float* out_uv;          // [B,N,2] or nullptr
  float* out_global;      // [B,N] pred_sdf_value_global (raw stream output) or nullptr
  float* out_local;       // [B,N] pred_sdf_value_local or nullptr
  int* status;            // device word the kernels OR failure bits into (DISN_STATUS_*), or nullptr
};

constexpr int DISN_STATUS_FP16_OVERFLOW = 1;   // DISN_PREC_F16F8: an activation exceeded fp16's range

}  // namespace disn

struct disn_ctx {
  disn_config cfg;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  std::map<std::string, disn::DevTensor> weights;
  bool weights_dirty = true;
  int64_t launches = 0;
  int num_sms = 148;            // cudaDevAttrMultiProcessorCount of cfg.device, read once in disn_create
  bool attr_conv_tc = false, attr_point_fp32 = false;   // cudaFuncSetAttribute done on this device
  std::set<const void*> attr_done;                      // ... for the point_tc_kernel instantiations

  // encoder state
  int32_t enc_B = 0;
  int32_t alloc_B = 0;          // batch the encoder buffers below are sized for
  disn::DevBuf img_in;          // [B,H,W,3] as uploaded
  disn::DevBuf img_rs;          // [B,224,224,3]
  disn::DevBuf act[2];          // ping-pong activations
  disn::DevBuf taps[5];
  disn::DevBuf proj[5];         // per-level projected maps [B,h,h,512]
  disn::DevBuf fc_a, fc_b;      // [B,4096]
  disn::DevBuf partial;         // split-K partials (fc layers)
  disn::DevBuf splitk_ws;       // split-K partials (conv / projection GEMMs)
  disn::DevBuf emb;             // [B,num_classes]
  disn::DevBuf gbias;           // [B,512]
  disn::DevBuf pmap;            // [B,img_h,img_w,512]
  cudaGraphExec_t enc_graph_exec = nullptr;   // captured encoder launch sequence (encoder_run)
  std::vector<int64_t> enc_graph_key, enc_warm_key;
  int64_t enc_graph_launches = 0;
  // scratch for host-pointer calls (ensure_point_scratch)
  disn::DevBuf d_pts, d_pts_rot, d_out, d_uv;
  disn::DevBuf d_tm;            // [max_batch,4,3]
  disn::DevBuf d_status;        // device status word (PointJob::status)
  int* h_status = nullptr;      // pinned host mirror, copied behind every point-kernel launch
  disn::DevBuf d_axes;          // [max_batch,3,R]
  std::vector<double> axes_key; // (sdf_params, R) the tables in d_axes were built from
  // bf16x3 packed weights (tcgen05 path)
  disn::DevBuf tc_weights;             // bf16 hi/lo stage images of the point MLP (DISN_PREC_BF16X3)
  disn::DevBuf tc_weights_f8;          // fp16 + e5m2 stage images (DISN_PREC_F16F8)
  float tc_act_scale[2][4][2] = {};
  float tc_small[2][2048] = {};         // host copy of the per-stream small parameters (the point kernel's __grid_constant__ table)
  std::map<std::string, disn::DevBuf> enc_tc_weights;   // packed bf16 hi/lo stage images of the encoder GEMMs
  // marching cubes: persistent scratch + the device-resident mesh of the last run (mc.cu)
  disn::DevBuf mc_code, mc_vbase, mc_chunk, mc_sums, mc_totals;
  uint32_t* mc_totals_host = nullptr;   // pinned
  disn::DevBuf mc_verts, mc_faces;
  int64_t mc_nv = 0, mc_nf = 0;
  // device-resident SDF grid of disn_eval_grid_resident and host staging for the marching-cubes input
  disn::DevBuf d_grid;
  disn::DevBuf d_mc_in;
  // staging of the host-pointer calls that synchronise before they return (nn_distance, cam, explicit-feature decoder)
  disn::DevBuf staging;
};

namespace disn {
// encoder.cu
int encoder_alloc(disn_ctx* c, int B);
int encoder_run(disn_ctx* c, const float* imgs, int B, int H, int W, int C, bool device_ptr,
                bool embedding_only = false);
void encoder_graph_reset(disn_ctx* c);
// api.cu
int run_point_job(disn_ctx* c, PointJob& job);    // fills weights / encoder products / status and launches per cfg.precision
int ensure_point_scratch(disn_ctx* c, int64_t pts);
// encoder.cu helpers reused by the explicit-feature decoder
int encoder_gemv(disn_ctx* c, const float* x, const float* W, const float* bias, float* out, int B, int K, int N, int relu);
int encoder_gemm_plain(disn_ctx* c, const std::string& wname, const float* A, const float* Bm, const float* bias, float* C,
                       int M, int N, int K, int relu);
// point_fp32.cu
int launch_point_fp32(disn_ctx* c, const PointJob& job);
// point_tc.cu
int tc_pack_weights(disn_ctx* c);
int launch_point_tc(disn_ctx* c, const PointJob& job);
// conv_tc.cu
int conv_tc_pack(disn_ctx* c, const float* d_w, int K, int N, DevBuf& out);
int launch_conv_tc(disn_ctx* c, const float* A, const uint8_t* wpk, const float* bias, float* C, float* ws,
                   int64_t ws_elems, int M, int N, int K, int H, int W, int Cin, int relu, int* splits_out);
// cam.cu
int launch_cam_heads(disn_ctx* c, int B, const float* d_K, float* d_rt, float* d_tm);
// chamfer.cu
int nn_distance(disn_ctx* c, const float* d_xyz1, int n, const float* d_xyz2, int m, int B, float* d_dist1,
                int* d_idx1, float* d_dist2, int* d_idx2);
// mc.cu
int mc_run(disn_ctx* c, const float* d_sdf, int R, const double* bbox, float iso, int64_t* n_verts, int64_t* n_faces);
int mc_fetch(disn_ctx* c, float* verts, int32_t* faces);
}  // namespace disn
