// IoU evaluator of the reference (test/test_iou.py:208-233, `iou_pymesh`): both meshes are voxelised with
// pymesh.VoxelGrid(2/dim), the VERTICES of the resulting voxel meshes are binned with ((v + 1.1) / 2.4 * dim).astype(int)
// into dim^3 occupancy grids, IoU = |A and B| / |A or B|.
//
// PyMesh is an un-vendored third-party dependency of the reference (no version pinned; README asks for a source build) and
// cannot be loaded here, so its voxeliser is RESTATED (parity unpinned against PyMesh itself):
//   * cells are indexed by integer triples k; cell k is the cube centred at k * cell with half-size cell / 2
//     (PyMesh's HashGrid keys are round(x / cell_size));
//   * a cell is occupied iff it overlaps at least one triangle (closed separating-axis test, 13 axes);
//   * the voxel mesh's vertices are the 8 corners (k +- 1/2) * cell of every occupied cell.
// The binning is the reference's expression; bins outside [0, dim) are dropped (numpy would wrap negatives and raise on
// >= dim; ShapeNet meshes are normalised into the unit sphere so neither happens).  The CPU twin
// oracle/metrics_oracle.py:iou_voxel does the same float64 operations in the same order; this file is compiled with
// --fmad=false so that the classification is identical (tests assert equal occupancy grids).
#include <algorithm>
#include <cstring>

#include "common.cuh"

namespace disn {
namespace {

constexpr int VG = 160;          // voxel index range [-80, 80) per axis: |coordinate| < 80 * 2/dim (1.45 for dim 110)
constexpr int VOFF = 80;

__device__ __forceinline__ bool axis_sep(double ax, double ay, double az, const double v[3][3], double half) {
  const double p0 = ax * v[0][0] + ay * v[0][1] + az * v[0][2];
  const double p1 = ax * v[1][0] + ay * v[1][1] + az * v[1][2];
  const double p2 = ax * v[2][0] + ay * v[2][1] + az * v[2][2];
  const double r = half * (fabs(ax) + fabs(ay) + fabs(az));
  return fmin(p0, fmin(p1, p2)) > r || fmax(p0, fmax(p1, p2)) < -r;
}

// closed triangle / axis-aligned cube overlap (separating axes: 3 cube normals, triangle normal, 9 edge cross products)
__device__ bool tri_cube_overlap(const double c[3], double half, const double t[3][3]) {
  double v[3][3];
  for (int k = 0; k < 3; ++k)
    for (int a = 0; a < 3; ++a) v[k][a] = t[k][a] - c[a];
  for (int a = 0; a < 3; ++a) {
    if (fmin(v[0][a], fmin(v[1][a], v[2][a])) > half || fmax(v[0][a], fmax(v[1][a], v[2][a])) < -half) return false;
  }
  double e[3][3];
  for (int a = 0; a < 3; ++a) { e[0][a] = v[1][a] - v[0][a]; e[1][a] = v[2][a] - v[1][a]; e[2][a] = v[0][a] - v[2][a]; }
  const double nx = e[0][1] * e[1][2] - e[0][2] * e[1][1];
  const double ny = e[0][2] * e[1][0] - e[0][0] * e[1][2];
  const double nz = e[0][0] * e[1][1] - e[0][1] * e[1][0];
  {
    const double d = nx * v[0][0] + ny * v[0][1] + nz * v[0][2];
    const double r = half * (fabs(nx) + fabs(ny) + fabs(nz));
    if (fabs(d) > r) return false;
  }
  for (int i = 0; i < 3; ++i) {
    if (axis_sep(0.0, -e[i][2], e[i][1], v, half)) return false;     // x cross e
    if (axis_sep(e[i][2], 0.0, -e[i][0], v, half)) return false;     // y cross e
    if (axis_sep(-e[i][1], e[i][0], 0.0, v, half)) return false;     // z cross e
  }
  return true;
}

__global__ void voxelize_kernel(const float* __restrict__ verts, const int32_t* __restrict__ faces, int64_t nf, double cell,
                                uint32_t* __restrict__ vox) {
  for (int64_t f = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; f < nf; f += (int64_t)gridDim.x * blockDim.x) {
    double t[3][3];
    double lo[3], hi[3];
    for (int k = 0; k < 3; ++k) {
      const float* p = verts + (int64_t)faces[f * 3 + k] * 3;
      for (int a = 0; a < 3; ++a) t[k][a] = (double)p[a];
    }
    int k0[3], k1[3];
    for (int a = 0; a < 3; ++a) {
      lo[a] = fmin(t[0][a], fmin(t[1][a], t[2][a]));
      hi[a] = fmax(t[0][a], fmax(t[1][a], t[2][a]));
      k0[a] = max(-VOFF, (int)floor(lo[a] / cell - 0.5));
      k1[a] = min(VOFF - 1, (int)ceil(hi[a] / cell + 0.5));
    }
    for (int kz = k0[2]; kz <= k1[2]; ++kz)
      for (int ky = k0[1]; ky <= k1[1]; ++ky)
        for (int kx = k0[0]; kx <= k1[0]; ++kx) {
          const double c[3] = {(double)kx * cell, (double)ky * cell, (double)kz * cell};
          if (!tri_cube_overlap(c, cell * 0.5, t)) continue;
          const int64_t id = ((int64_t)(kz + VOFF) * VG + (ky + VOFF)) * VG + (kx + VOFF);
          atomicOr(&vox[id >> 5], 1u << (id & 31));
        }
  }
}

// corners of occupied cells -> ((c + 1.1) / 2.4 * dim) truncated -> occupancy bits
__global__ void corners_kernel(const uint32_t* __restrict__ vox, double cell, int dim, uint32_t* __restrict__ occ) {
  const int64_t nwords = (int64_t)VG * VG * VG / 32;
  for (int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w < nwords; w += (int64_t)gridDim.x * blockDim.x) {
    uint32_t bits = vox[w];
    while (bits) {
      const int b = __ffs(bits) - 1;
      bits &= bits - 1;
      const int64_t id = w * 32 + b;
      const int kx = (int)(id % VG) - VOFF, ky = (int)((id / VG) % VG) - VOFF, kz = (int)(id / ((int64_t)VG * VG)) - VOFF;
      for (int cz = 0; cz < 2; ++cz)
        for (int cy = 0; cy < 2; ++cy)
          for (int cx = 0; cx < 2; ++cx) {
            const double p[3] = {((double)kx + (cx ? 0.5 : -0.5)) * cell, ((double)ky + (cy ? 0.5 : -0.5)) * cell,
                                 ((double)kz + (cz ? 0.5 : -0.5)) * cell};
            int ind[3];
            bool ok = true;
            for (int a = 0; a < 3; ++a) {
              const double q = (p[a] + 1.1) / 2.4 * (double)dim;
              ind[a] = (int)q;                       // astype(int): truncation toward zero
              ok = ok && ind[a] >= 0 && ind[a] < dim;   // q in (-1, 0) truncates to bin 0, exactly like numpy
            }
            if (!ok) continue;
            const int64_t o = ((int64_t)ind[0] * dim + ind[1]) * dim + ind[2];     // v[ind[:,0], ind[:,1], ind[:,2]]
            atomicOr(&occ[o >> 5], 1u << (o & 31));
          }
    }
  }
}

__global__ void iou_count_kernel(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, int64_t nwords,
                                 unsigned long long* __restrict__ out) {
  unsigned long long inter = 0, uni = 0;
  for (int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w < nwords; w += (int64_t)gridDim.x * blockDim.x) {
    inter += __popc(a[w] & b[w]);
    uni += __popc(a[w] | b[w]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    inter += __shfl_xor_sync(0xffffffffu, inter, o);
    uni += __shfl_xor_sync(0xffffffffu, uni, o);
  }
  if ((threadIdx.x & 31) == 0) { atomicAdd(&out[0], inter); atomicAdd(&out[1], uni); }
}

__global__ void unpack_bits_kernel(const uint32_t* __restrict__ bits, int64_t n, uint8_t* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (bits[i >> 5] >> (i & 31)) & 1u;
}

}  // namespace
}  // namespace disn

using namespace disn;

extern "C" int disn_iou(disn_ctx* c, const float* verts1, int64_t nv1, const int32_t* faces1, int64_t nf1,
                        const float* verts2, int64_t nv2, const int32_t* faces2, int64_t nf2, int32_t dim,
                        int64_t* intersection, int64_t* uni, uint8_t* occ1_out, uint8_t* occ2_out) {
  DISN_REQUIRE(c && verts1 && faces1 && verts2 && faces2 && intersection && uni, "null argument");
  DISN_REQUIRE(dim >= 2 && dim <= 512 && nv1 > 0 && nf1 > 0 && nv2 > 0 && nf2 > 0, "dim in [2,512], non-empty meshes");
  DISN_CUDA_OK(cudaSetDevice(c->cfg.device));
  for (int m = 0; m < 2; ++m) {       // reject out-of-range vertex ids up front (device reads are unchecked)
    const int32_t* f = m ? faces2 : faces1;
    const int64_t nf = m ? nf2 : nf1, nv = m ? nv2 : nv1;
    for (int64_t i = 0; i < nf * 3; ++i) DISN_REQUIRE(f[i] >= 0 && f[i] < nv, "face index out of range");
  }
  const int64_t vox_words = (int64_t)VG * VG * VG / 32, n_occ = (int64_t)dim * dim * dim, occ_words = (n_occ + 31) / 32;
  const size_t bytes = (size_t)(nv1 + nv2) * 12 + (size_t)(nf1 + nf2) * 12 + (size_t)(vox_words + 2 * occ_words) * 4 + 16 +
                       (size_t)n_occ + 4096;
  DevBuf buf;
  if (buf.reserve(bytes)) return -1;
  uint32_t* vox = buf.take<uint32_t>(vox_words);
  uint32_t* occ[2] = {buf.take<uint32_t>(occ_words), buf.take<uint32_t>(occ_words)};
  unsigned long long* cnt = buf.take<unsigned long long>(2);
  uint8_t* unp = buf.take<uint8_t>(n_occ);
  const double cell = 2.0 / (double)dim;                 // pymesh.VoxelGrid(2./dim)
  const int grid = c->num_sms * 8;
  DISN_CUDA_OK(cudaMemsetAsync(occ[0], 0, occ_words * 4, c->stream));
  DISN_CUDA_OK(cudaMemsetAsync(occ[1], 0, occ_words * 4, c->stream));
  DISN_CUDA_OK(cudaMemsetAsync(cnt, 0, 16, c->stream));
  for (int m = 0; m < 2; ++m) {
    const float* hv = m ? verts2 : verts1;
    const int32_t* hf = m ? faces2 : faces1;
    const int64_t nv = m ? nv2 : nv1, nf = m ? nf2 : nf1;
    float* dv = buf.take<float>((size_t)nv * 3);
    int32_t* df = buf.take<int32_t>((size_t)nf * 3);
    DISN_CUDA_OK(cudaMemcpyAsync(dv, hv, (size_t)nv * 12, cudaMemcpyHostToDevice, c->stream));
    DISN_CUDA_OK(cudaMemcpyAsync(df, hf, (size_t)nf * 12, cudaMemcpyHostToDevice, c->stream));
    DISN_CUDA_OK(cudaMemsetAsync(vox, 0, vox_words * 4, c->stream));
    voxelize_kernel<<<grid, 128, 0, c->stream>>>(dv, df, nf, cell, vox);
    corners_kernel<<<grid, 256, 0, c->stream>>>(vox, cell, dim, occ[m]);
    c->launches += 2;
  }
  iou_count_kernel<<<grid, 256, 0, c->stream>>>(occ[0], occ[1], occ_words, cnt);
  c->launches++;
  DISN_CUDA_OK(cudaGetLastError());
  unsigned long long h[2] = {0, 0};
  DISN_CUDA_OK(cudaMemcpyAsync(h, cnt, 16, cudaMemcpyDeviceToHost, c->stream));
  for (int m = 0; m < 2; ++m) {
    uint8_t* out = m ? occ2_out : occ1_out;
    if (!out) continue;
    unpack_bits_kernel<<<grid, 256, 0, c->stream>>>(occ[m], n_occ, unp);
    DISN_CUDA_OK(cudaMemcpyAsync(out, unp, (size_t)n_occ, cudaMemcpyDeviceToHost, c->stream));
    DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  }
  DISN_CUDA_OK(cudaStreamSynchronize(c->stream));
  *intersection = (int64_t)h[0];
  *uni = (int64_t)h[1];
  return 0;
}
