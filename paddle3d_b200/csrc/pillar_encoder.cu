// PillarFeatureNet with one PFNLayer (models/voxel_encoders/pillar_encoder.py:156-210, :81-106; SURVEY.md §8f-2):
// decorate the <= M points of a pillar (xyz - pillar mean, xy - pillar centre), zero the padding rows, Linear(F+5 -> C,
// no bias) + BatchNorm1D(eval) + ReLU, max over the M rows — one block per pillar, one thread per output channel, the
// decorated rows staged in shared memory.  The reference runs this as ~15 elementwise / matmul / argmax launches over
// the [N, M, F+5] and [N, M, C] intermediates; here only voxels [N, M, F] is read and [N, C] written.
// Parity-green on a B200 (tests/test_gpu_voxelize.py::test_pillar_feature_net, 1e-4 vs the oracle restatement).
//
// p3d_pillar_feature_net_pixel_h16 runs the same arithmetic and writes each pillar's C channels straight into the pixel
// fp16-pair image the dense RPN reads (PointPillarsScatter + the NCHW -> pixel H16 conversion folded into the epilogue):
// no [N, C] rows and no fp32 NCHW canvas in between.
#include "common.cuh"
#include "h16.cuh"
#include "p3d_b200.h"

namespace p3d {
namespace {

constexpr int kMaxM = 64, kMaxF = 8;

// kPixel = false: out_rows[i * C + c].  kPixel = true: pixel H16 image [batch * ny * nx][C / 32][hi 32 | lo' 32], row
// (b * ny + y) * nx + x of the pillar's coors (b, z, y, x); z is ignored as in PointPillarsScatter.  Pillars outside
// the grid or with b >= batch are skipped.  Cells are unique (hard_voxelize emits one row per cell), so no two blocks
// write the same pixel.  The fp32 arithmetic is the same in both forms, so the image equals
// nchw_to_pixel_h16(pillar_scatter(rows)) bit for bit.
template <bool kPixel>
__global__ void pfn_kernel(const float *__restrict__ voxels, const int32_t *__restrict__ npv,
                           const int32_t *__restrict__ coors, const int32_t *__restrict__ num_dev, int n_cap, int M, int F,
                           int C, const float *__restrict__ weight, const float *__restrict__ scale,
                           const float *__restrict__ shift, float vx, float vy, float x_off, float y_off,
                           float *__restrict__ out_rows, int batch, int ny, int nx, __half *__restrict__ out_img,
                           int32_t *__restrict__ status) {
  __shared__ float s_f[kMaxM][kMaxF + 5];
  __shared__ float s_mean[3];
  const int n = num_dev ? min(num_dev[0], n_cap) : n_cap;
  const int i = blockIdx.x;
  if (i >= n) return;
  const int cb = coors[i * 4], cy_i = coors[i * 4 + 2], cx_i = coors[i * 4 + 3];
  if (kPixel && (cb < 0 || cb >= batch || cy_i < 0 || cy_i >= ny || cx_i < 0 || cx_i >= nx)) return;
  const int cnt = npv[i];
  const int D = F + 5;
  const float *v = voxels + static_cast<size_t>(i) * M * F;
  if (threadIdx.x < 3) {  // mean over ALL M rows' sum (padding rows are zero) divided by the point count (:172-175)
    float s = 0.f;
    for (int m = 0; m < M; ++m) s += v[m * F + threadIdx.x];
    s_mean[threadIdx.x] = s / static_cast<float>(cnt);
  }
  __syncthreads();
  const float cx = static_cast<float>(cx_i) * vx + x_off, cy = static_cast<float>(cy_i) * vy + y_off;
  for (int e = threadIdx.x; e < M * D; e += blockDim.x) {
    const int m = e / D, d = e - m * D;
    float val;
    if (d < F)
      val = v[m * F + d];
    else if (d < F + 3)
      val = v[m * F + (d - F)] - s_mean[d - F];
    else
      val = v[m * F + (d - F - 3)] - (d == F + 3 ? cx : cy);
    s_f[m][d] = (m < cnt) ? val : 0.f;  // padding rows zeroed after the decoration (:193-198)
  }
  __syncthreads();
  bool ovf = false;
  __half *px = kPixel ? out_img + ((static_cast<size_t>(cb) * ny + cy_i) * nx + cx_i) * (2 * static_cast<size_t>(C)) : nullptr;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float w[kMaxF + 5];
    for (int d = 0; d < D; ++d) w[d] = __ldg(weight + d * C + c);
    const float sc = __ldg(scale + c), sh = __ldg(shift + c);
    float best = -INFINITY;
    for (int m = 0; m < M; ++m) {
      float acc = 0.f;
      for (int d = 0; d < D; ++d) acc = fmaf(s_f[m][d], w[d], acc);
      best = fmaxf(best, fmaxf(fmaf(acc, sc, sh), 0.f));
    }
    if (kPixel) {
      __half hi, lo;
      split_h16(best, hi, lo, ovf);
      __half *grp = px + (c >> 5) * 64;  // 32-channel group [hi 32 | lo' 32]
      grp[c & 31] = hi;
      grp[32 + (c & 31)] = lo;
    } else {
      out_rows[static_cast<size_t>(i) * C + c] = best;
    }
  }
  if (kPixel && ovf && status) atomicOr(status, 1);
}

struct Decor {
  float vx, vy, x_off, y_off;
};

int check_pfn_args(const float *voxels, const int32_t *npv, const int32_t *coors, int64_t n_cap, int M, int F, int C,
                   const float *weight, const float *scale, const float *shift, const float *vs, const float *pcr) {
  if (!voxels || !npv || !coors || !weight || !scale || !shift || !vs || !pcr || n_cap < 0 || C < 1)
    return P3D_ERR_INVALID_ARG;
  if (M < 1 || M > kMaxM || F < 3 || F > kMaxF) return P3D_ERR_UNSUPPORTED;
  if (n_cap > 0x7fffffff) return P3D_ERR_UNSUPPORTED;  // one block per pillar
  return P3D_OK;
}

Decor decor(const float *vs, const float *pcr) {
  const float vx = vs[0], vy = vs[1];
  return {vx, vy, vx / 2 + pcr[0], vy / 2 + pcr[1]};  // :147-148
}

}  // namespace
}  // namespace p3d

using namespace p3d;

extern "C" int p3d_pillar_feature_net(const float *voxels, const int32_t *num_points_per_voxel, const int32_t *coors,
                                      const int32_t *num_voxels_dev, int64_t n_cap, int max_points, int num_point_dim,
                                      int out_channels, const float *weight, const float *bn_scale,
                                      const float *bn_shift, const float *voxel_size_host,
                                      const float *point_cloud_range_host, float *out, p3d_stream_t stream) {
  if (!out) return P3D_ERR_INVALID_ARG;
  const int rc = check_pfn_args(voxels, num_points_per_voxel, coors, n_cap, max_points, num_point_dim, out_channels,
                                weight, bn_scale, bn_shift, voxel_size_host, point_cloud_range_host);
  if (rc != P3D_OK) return rc;
  if (n_cap == 0) return P3D_OK;
  const Decor dc = decor(voxel_size_host, point_cloud_range_host);
  const int threads = out_channels <= 64 ? 64 : 128;
  pfn_kernel<false><<<static_cast<unsigned int>(n_cap), threads, 0, static_cast<cudaStream_t>(stream)>>>(
      voxels, num_points_per_voxel, coors, num_voxels_dev, static_cast<int>(n_cap), max_points, num_point_dim,
      out_channels, weight, bn_scale, bn_shift, dc.vx, dc.vy, dc.x_off, dc.y_off, out, 0, 0, 0, nullptr, nullptr);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

extern "C" int p3d_pillar_feature_net_pixel_h16(const float *voxels, const int32_t *num_points_per_voxel,
                                                const int32_t *coors, const int32_t *num_voxels_dev, int64_t n_cap,
                                                int max_points, int num_point_dim, int out_channels, const float *weight,
                                                const float *bn_scale, const float *bn_shift, const float *voxel_size_host,
                                                const float *point_cloud_range_host, int batch, int ny, int nx,
                                                void *out_pixel_h16, int32_t *status_dev, p3d_stream_t stream) {
  if (!out_pixel_h16 || batch < 1 || ny < 1 || nx < 1) return P3D_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(out_pixel_h16) & 15) || (reinterpret_cast<uintptr_t>(coors) & 15) ||
      (reinterpret_cast<uintptr_t>(voxels) & 3))
    return P3D_ERR_INVALID_ARG;
  const int rc = check_pfn_args(voxels, num_points_per_voxel, coors, n_cap, max_points, num_point_dim, out_channels,
                                weight, bn_scale, bn_shift, voxel_size_host, point_cloud_range_host);
  if (rc != P3D_OK) return rc;
  if (out_channels % 32) return P3D_ERR_UNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t bytes = static_cast<size_t>(batch) * ny * nx * out_channels * 4;
  P3D_CUDA_CHECK(cudaMemsetAsync(out_pixel_h16, 0, bytes, st));  // (hi, lo') = (0, 0) is the value 0: empty pixels
  if (n_cap == 0) return P3D_OK;
  const Decor dc = decor(voxel_size_host, point_cloud_range_host);
  const int threads = out_channels <= 64 ? 64 : 128;
  pfn_kernel<true><<<static_cast<unsigned int>(n_cap), threads, 0, st>>>(
      voxels, num_points_per_voxel, coors, num_voxels_dev, static_cast<int>(n_cap), max_points, num_point_dim,
      out_channels, weight, bn_scale, bn_shift, dc.vx, dc.vy, dc.x_off, dc.y_off, nullptr, batch, ny, nx,
      static_cast<__half *>(out_pixel_h16), status_dev);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}
