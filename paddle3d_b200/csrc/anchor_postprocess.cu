// Anchor-based SSD head post-processing (PointPillars / SECOND) for sm_100a: batch 1, no host synchronisation.
//
// Replaces the Python post-processing of the reference's SSD head (detection/pointpillars/pointpillars.py:105-129 and
// rotate_nms_pcdet): masked_select of the candidates, argsort, and nms_gpu's host greedy step each synchronise with
// the host.  Here every stage runs on the device and the whole call can be captured into a CUDA graph:
//   K1 ap_occupancy   pillar occupancy [ny, nx] of the frame's coors (after a memset), for the anchor mask
//   K2 ap_row_scan    inclusive prefix sums along x, one CTA per row (block scan in registers / shared memory)
//   K3 ap_col_scan    inclusive prefix sums along y: 32 columns x 32 row segments per CTA, segment sums, then a
//                     scan over the segments: the integral image I of fused_get_anchors_area
//   K4 ap_score       per anchor: mask (area of its static cell box > anchor_area_threshold), sigmoid / max / first
//                     argmax over the C class logits, candidate iff score >= score_threshold; 64-bit sort key
//                     (~score_bits << ab | anchor), non-candidates get the all-ones sentinel
//   sort              cub::DeviceRadixSort over all H*W*A keys: descending score, ties by ascending anchor index
//   K5 ap_gather      the first pre_max candidates: second_box_decode (fp32, no FMA contraction), direction label,
//                     and the box re-laid as rotate_nms_pcdet hands it to nms_gpu (fp32 angle -r - pi/2)
//   K6 ap_nms_mask    rotated-IoU suppression bit-matrix (nms_rotated_tile, upper triangle)
//   K7 ap_greedy      greedy reduction on the device (nms_greedy_cta), stops after post_max kept boxes
//   K8 ap_emit        direction fix, post_center_range filter (order kept), outputs and counts
#include <cub/cub.cuh>

#include "common.cuh"
#include "nms_reduce.cuh"

namespace p3d {
namespace {

constexpr int kScoreThreads = 256;
constexpr int kRowThreads = 512;
constexpr int kEmitThreads = 256;

struct ApAttrs {
  int H, W, A, C, HW, N;   // feature map, anchors per location, classes, H*W, H*W*A
  int ab;                  // bits of the anchor index in a sort key
  int ny, nx, use_mask;
  float area_thr, score_thr, iou_thr;
  int pre_max, post_max, cbmax;
  int use_range;
  float range[6];
};

struct ApWs {
  int32_t *cnt;                 // [0] candidates, [1] boxes kept by the greedy pass
  int32_t *integral;            // [ny, nx]
  unsigned long long *keys;     // [N]
  unsigned long long *sorted;   // [N]
  void *cub_tmp;
  size_t cub_bytes;
  float *boxes;                 // [pre_max, 7] decoded, in score order
  float *nms_boxes;             // [pre_max, 7] as rotate_nms_pcdet re-lays them
  float *score;                 // [pre_max]
  int32_t *label;               // [pre_max] class | (direction label << 16)
  int32_t *anchor;              // [pre_max]
  unsigned long long *mask;     // [pre_max, cbmax]
  int32_t *keep;                // [pre_max]
  size_t bytes;
};

int key_bits(int n) {
  int b = 1;
  while ((1ll << b) <= n) ++b;  // every anchor index < 2^b - 1: the sentinel stays above every candidate key
  return b;
}

ApWs carve(void *p, int N, int ny, int nx, int pre_max) {
  ApWs w;
  Carver c(p);
  const int cbmax = (pre_max + 63) / 64;
  w.cnt = c.take<int32_t>(4);
  w.integral = c.take<int32_t>(static_cast<size_t>(ny) * nx > 0 ? static_cast<size_t>(ny) * nx : 1);
  w.keys = c.take<unsigned long long>(N);
  w.sorted = c.take<unsigned long long>(N);
  size_t a = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, a, static_cast<const unsigned long long *>(nullptr),
                                 static_cast<unsigned long long *>(nullptr), N, 0, 32 + key_bits(N));
  w.cub_bytes = a;
  w.cub_tmp = c.take<char>(a);
  w.boxes = c.take<float>(static_cast<size_t>(pre_max) * 7);
  w.nms_boxes = c.take<float>(static_cast<size_t>(pre_max) * 7);
  w.score = c.take<float>(pre_max);
  w.label = c.take<int32_t>(pre_max);
  w.anchor = c.take<int32_t>(pre_max);
  w.mask = c.take<unsigned long long>(static_cast<size_t>(pre_max) * cbmax);
  w.keep = c.take<int32_t>(pre_max);
  w.bytes = c.off;
  return w;
}

__global__ void __launch_bounds__(256) ap_occupancy_kernel(const int32_t *__restrict__ coors,
                                                           const int32_t *__restrict__ num_voxels, int ny, int nx,
                                                           int32_t *__restrict__ occ) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num_voxels[0]) return;
  const int4 c = reinterpret_cast<const int4 *>(coors)[i];  // (b, z, y, x)
  if (c.z >= 0 && c.z < ny && c.w >= 0 && c.w < nx) occ[c.z * nx + c.w] = 1;  // pillars are unique per cell
}

__global__ void __launch_bounds__(kRowThreads) ap_row_scan_kernel(int nx, int32_t *__restrict__ img) {
  using Scan = cub::BlockScan<int, kRowThreads>;
  __shared__ typename Scan::TempStorage tmp;
  int32_t *row = img + static_cast<size_t>(blockIdx.x) * nx;
  int carry = 0;
  for (int c0 = 0; c0 < nx; c0 += kRowThreads) {
    const int x = c0 + threadIdx.x;
    int v = x < nx ? row[x] : 0, total;
    Scan(tmp).InclusiveSum(v, v, total);
    if (x < nx) row[x] = v + carry;
    carry += total;
    __syncthreads();
  }
}

// 32 columns per CTA; thread (tx, ty) owns rows [ty * seg, (ty + 1) * seg) of column blockIdx.x * 32 + tx
__global__ void __launch_bounds__(1024) ap_col_scan_kernel(int ny, int nx, int32_t *__restrict__ img) {
  __shared__ int s_sum[32][33];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int x = blockIdx.x * 32 + tx;
  const int seg = (ny + 31) / 32;
  const int y0 = ty * seg, y1 = min(y0 + seg, ny);
  int s = 0;
  if (x < nx)
    for (int y = y0; y < y1; ++y) s += img[static_cast<size_t>(y) * nx + x];
  s_sum[ty][tx] = s;
  __syncthreads();
  int run = 0;
  for (int k = 0; k < ty; ++k) run += s_sum[k][tx];
  if (x < nx)
    for (int y = y0; y < y1; ++y) {
      run += img[static_cast<size_t>(y) * nx + x];
      img[static_cast<size_t>(y) * nx + x] = run;
    }
}

__device__ __forceinline__ float ap_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }  // paddle / torch sigmoid, fp32

__device__ __forceinline__ void ap_best_class(const float *__restrict__ cls, int p, int a, const ApAttrs &at, float &best,
                                              int &label) {
  best = ap_sigmoid(__ldg(cls + static_cast<size_t>(a * at.C) * at.HW + p));
  label = 0;
  for (int c = 1; c < at.C; ++c) {
    const float s = ap_sigmoid(__ldg(cls + static_cast<size_t>(a * at.C + c) * at.HW + p));
    if (s > best) {  // max / argmax: the first maximal class wins
      best = s;
      label = c;
    }
  }
}

__global__ void __launch_bounds__(kScoreThreads) ap_score_kernel(const float *__restrict__ cls, const int4 *__restrict__ cells,
                                                                 ApAttrs at, ApWs w) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  bool cand = false;
  unsigned long long key = ~0ull >> (32 - at.ab);  // sentinel: all ones over the 32 + ab sorted bits
  if (i < at.N) {
    const int a = i % at.A, p = i / at.A;
    bool keep = true;
    if (at.use_mask) {
      // fused_get_anchors_area: I[y1, x1] - I[y1, x0] - I[y0, x1] + I[y0, x0] (the min row / column is excluded)
      const int4 c = __ldg(cells + i);
      const int x0 = min(max(c.x, 0), at.nx - 1), y0 = min(max(c.y, 0), at.ny - 1);
      const int x1 = min(max(c.z, 0), at.nx - 1), y1 = min(max(c.w, 0), at.ny - 1);
      const int32_t *I = w.integral;
      const int area = I[y1 * at.nx + x1] - I[y1 * at.nx + x0] - I[y0 * at.nx + x1] + I[y0 * at.nx + x0];
      keep = static_cast<float>(area) > at.area_thr;
    }
    if (keep) {
      float best;
      int label;
      ap_best_class(cls, p, a, at, best, label);
      cand = best >= at.score_thr;  // SECOND's predict keeps top_scores >= threshold
      if (cand) key = (static_cast<unsigned long long>(~__float_as_uint(best)) << at.ab) | static_cast<unsigned int>(i);
    }
    w.keys[i] = key;
  }
  const int n = __syncthreads_count(cand);
  if (threadIdx.x == 0 && n) atomicAdd(w.cnt, n);
}

__global__ void __launch_bounds__(128) ap_gather_kernel(const float *__restrict__ cls, const float *__restrict__ box,
                                                        const float *__restrict__ dir, const float *__restrict__ anchors,
                                                        ApAttrs at, ApWs w) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = min(w.cnt[0], at.pre_max);
  if (r >= n) return;
  const unsigned long long key = w.sorted[r];
  const int i = static_cast<int>(key & ((1ull << at.ab) - 1));
  const int a = i % at.A, p = i / at.A;
  float best;
  int label;
  ap_best_class(cls, p, a, at, best, label);
  // direction label: argmax over the 2 logits, the first maximal one wins
  const float d0 = __ldg(dir + static_cast<size_t>(a * 2) * at.HW + p), d1 = __ldg(dir + static_cast<size_t>(a * 2 + 1) * at.HW + p);
  const int dl = d1 > d0 ? 1 : 0;
  // second_box_decode, (x, y, z, w, l, h, r), in the reference's operation order
  const float *an = anchors + static_cast<size_t>(i) * 7;
  float t[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) t[k] = __ldg(box + static_cast<size_t>(a * 7 + k) * at.HW + p);
  const float xa = __ldg(an), ya = __ldg(an + 1), wa = __ldg(an + 3), la = __ldg(an + 4), ha = __ldg(an + 5),
              ra = __ldg(an + 6);
  const float za = __fadd_rn(__ldg(an + 2), __fdiv_rn(ha, 2.0f));
  const float diag = sqrtf(__fadd_rn(__fmul_rn(la, la), __fmul_rn(wa, wa)));
  float b[7];
  b[0] = __fadd_rn(__fmul_rn(t[0], diag), xa);
  b[1] = __fadd_rn(__fmul_rn(t[1], diag), ya);
  const float zg = __fadd_rn(__fmul_rn(t[2], ha), za);
  b[3] = __fmul_rn(expf(t[3]), wa);
  b[4] = __fmul_rn(expf(t[4]), la);
  b[5] = __fmul_rn(expf(t[5]), ha);
  b[6] = __fadd_rn(t[6], ra);
  b[2] = __fsub_rn(zg, __fdiv_rn(b[5], 2.0f));
  float *ob = w.boxes + static_cast<size_t>(r) * 7, *nb = w.nms_boxes + static_cast<size_t>(r) * 7;
#pragma unroll
  for (int k = 0; k < 7; ++k) ob[k] = b[k];
  // rotate_nms_pcdet: columns [0, 1, 2, 4, 3, 5, 6], angle -r - pi/2 evaluated in fp32 like the tensor expression
  nb[0] = b[0];
  nb[1] = b[1];
  nb[2] = b[2];
  nb[3] = b[4];
  nb[4] = b[3];
  nb[5] = b[5];
  nb[6] = __fsub_rn(-b[6], 1.57079632679489662f);
  w.score[r] = best;
  w.label[r] = label | (dl << 16);
  w.anchor[r] = i;
}

__global__ void __launch_bounds__(64) ap_nms_mask_kernel(ApAttrs at, ApWs w) {
  const int rb = blockIdx.y, cb = blockIdx.x;
  if (cb < rb) return;
  const int n = min(w.cnt[0], at.pre_max);
  if (rb * 64 >= n || cb * 64 >= n) return;
  const int rows = min(n - rb * 64, 64), cols = min(n - cb * 64, 64);
  __shared__ float s_col[64 * 7], s_row[64 * 7];
  __shared__ unsigned short s_pairs[64 * 64];
  __shared__ unsigned long long s_bits[64];
  __shared__ int s_cnt[3];
  for (int k = threadIdx.x; k < cols * 7; k += 64) s_col[k] = w.nms_boxes[static_cast<size_t>(cb) * 64 * 7 + k];
  for (int k = threadIdx.x; k < rows * 7; k += 64) s_row[k] = w.nms_boxes[static_cast<size_t>(rb) * 64 * 7 + k];
  __syncthreads();
  const unsigned long long bits = nms_rotated_tile(s_row, s_col, rows, cols, rb == cb, at.iou_thr, s_pairs, s_bits, s_cnt);
  if (threadIdx.x < rows) w.mask[static_cast<size_t>(rb * 64 + threadIdx.x) * at.cbmax + cb] = bits;
}

__global__ void __launch_bounds__(256) ap_greedy_kernel(ApAttrs at, ApWs w) {
  extern __shared__ unsigned long long s_dyn[];
  __shared__ unsigned long long s_misc[2];
  const int n = min(w.cnt[0], at.pre_max);
  const int k = nms_greedy_cta(w.mask, n, at.cbmax, w.keep, s_dyn, s_misc, at.post_max);
  if (threadIdx.x == 0) w.cnt[1] = min(k, at.post_max);
}

__global__ void __launch_bounds__(kEmitThreads) ap_emit_kernel(ApAttrs at, ApWs w, float *__restrict__ boxes_out,
                                                               float *__restrict__ scores_out, long long *__restrict__ labels_out,
                                                               int32_t *__restrict__ index_out, int32_t *__restrict__ counts) {
  using Scan = cub::BlockScan<int, kEmitThreads>;
  __shared__ typename Scan::TempStorage tmp;
  const int kept = w.cnt[1];
  int base = 0;
  for (int r0 = 0; r0 < kept; r0 += kEmitThreads) {
    const int r = r0 + threadIdx.x;
    float b[7];
    bool ok = false;
    int src = 0;
    if (r < kept) {
      src = w.keep[r];
      const float *s = w.boxes + static_cast<size_t>(src) * 7;
#pragma unroll
      for (int k = 0; k < 7; ++k) b[k] = s[k];
      // direction fix: (r > 0) XOR dir_label -> r += pi (fp32)
      const int dl = w.label[src] >> 16;
      if ((b[6] > 0.f) != (dl != 0)) b[6] = __fadd_rn(b[6], 3.14159265358979324f);
      ok = true;
      if (at.use_range)
        ok = b[0] >= at.range[0] && b[1] >= at.range[1] && b[2] >= at.range[2] && b[0] <= at.range[3] &&
             b[1] <= at.range[4] && b[2] <= at.range[5];
    }
    int pos, total;
    Scan(tmp).ExclusiveSum(ok ? 1 : 0, pos, total);
    if (ok) {
      const int o = base + pos;
      float *ob = boxes_out + static_cast<size_t>(o) * 7;
#pragma unroll
      for (int k = 0; k < 7; ++k) ob[k] = b[k];
      scores_out[o] = w.score[src];
      labels_out[o] = static_cast<long long>(w.label[src] & 0xffff);
      if (index_out) index_out[o] = w.anchor[src];
    }
    base += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    counts[0] = w.cnt[0];
    counts[1] = base;
  }
}

}  // namespace
}  // namespace p3d

using namespace p3d;

extern "C" size_t p3d_anchor_head_postprocess_workspace_bytes(int num_anchors, int grid_ny, int grid_nx,
                                                               int nms_pre_max_size) {
  if (num_anchors < 1 || num_anchors >= (1 << 30) || grid_ny < 0 || grid_nx < 0 || nms_pre_max_size < 1 ||
      static_cast<long long>(grid_ny) * grid_nx >= (1ll << 31))
    return 0;
  return carve(nullptr, num_anchors, grid_ny, grid_nx, nms_pre_max_size).bytes;
}

extern "C" int p3d_anchor_head_postprocess(const float *cls, const float *box, const float *dir, int H, int W, int A, int C,
                                           const float *anchors, const int32_t *anchor_cells, const int32_t *coors,
                                           const int32_t *num_voxels_dev, int grid_ny, int grid_nx,
                                           float anchor_area_threshold, float score_threshold, float iou_threshold,
                                           int nms_pre_max_size, int nms_post_max_size,
                                           const float *post_center_range_host, float *boxes_out, float *scores_out,
                                           int64_t *labels_out, int32_t *anchor_index_out, int32_t *counts_out, void *workspace,
                                           size_t workspace_bytes, p3d_stream_t stream) {
  if (!cls || !box || !dir || !anchors || !boxes_out || !scores_out || !labels_out || !counts_out || !workspace || H < 1 ||
      W < 1 || A < 1 || C < 1 || C > 0xffff || nms_pre_max_size < 1 || nms_post_max_size < 0)
    return P3D_ERR_INVALID_ARG;
  const long long N = static_cast<long long>(H) * W * A;
  if (N >= (1 << 30)) return P3D_ERR_UNSUPPORTED;
  const bool use_mask = anchor_cells != nullptr && anchor_area_threshold >= 0.f;
  if (use_mask && (!coors || !num_voxels_dev || grid_ny < 1 || grid_nx < 1 ||
                   (reinterpret_cast<uintptr_t>(coors) & 15) || (reinterpret_cast<uintptr_t>(anchor_cells) & 15)))
    return P3D_ERR_INVALID_ARG;
  const int ny = use_mask ? grid_ny : 0, nx = use_mask ? grid_nx : 0;
  const size_t need = p3d_anchor_head_postprocess_workspace_bytes(static_cast<int>(N), ny, nx, nms_pre_max_size);
  if (!need) return P3D_ERR_INVALID_ARG;
  if (workspace_bytes < need) return P3D_ERR_WORKSPACE;
  ApWs w = carve(workspace, static_cast<int>(N), ny, nx, nms_pre_max_size);
  ApAttrs at;
  at.H = H;
  at.W = W;
  at.A = A;
  at.C = C;
  at.HW = H * W;
  at.N = static_cast<int>(N);
  at.ab = key_bits(at.N);
  at.ny = ny;
  at.nx = nx;
  at.use_mask = use_mask ? 1 : 0;
  at.area_thr = anchor_area_threshold;
  at.score_thr = score_threshold;
  at.iou_thr = iou_threshold;
  at.pre_max = nms_pre_max_size;
  at.post_max = nms_post_max_size;
  at.cbmax = (nms_pre_max_size + 63) / 64;
  at.use_range = post_center_range_host ? 1 : 0;
  for (int k = 0; k < 6; ++k) at.range[k] = post_center_range_host ? post_center_range_host[k] : 0.f;
  if (static_cast<size_t>(at.cbmax) * 8 > 48 * 1024 || at.cbmax > 65535) return P3D_ERR_UNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  P3D_CUDA_CHECK(cudaMemsetAsync(w.cnt, 0, 4 * sizeof(int32_t), st));
  if (use_mask) {
    P3D_CUDA_CHECK(cudaMemsetAsync(w.integral, 0, static_cast<size_t>(ny) * nx * sizeof(int32_t), st));
    // every row of coors may be live: num_voxels_dev bounds the launch's work, the grid covers the capacity ny * nx
    // (hard_voxelize emits at most one row per cell)
    ap_occupancy_kernel<<<div_up(static_cast<long long>(ny) * nx, 256), 256, 0, st>>>(coors, num_voxels_dev, ny, nx,
                                                                                      w.integral);
    P3D_LAUNCH_CHECK();
    ap_row_scan_kernel<<<ny, kRowThreads, 0, st>>>(nx, w.integral);
    P3D_LAUNCH_CHECK();
    ap_col_scan_kernel<<<div_up(nx, 32), dim3(32, 32), 0, st>>>(ny, nx, w.integral);
    P3D_LAUNCH_CHECK();
  }
  ap_score_kernel<<<div_up(N, kScoreThreads), kScoreThreads, 0, st>>>(cls, reinterpret_cast<const int4 *>(anchor_cells), at, w);
  P3D_LAUNCH_CHECK();
  size_t tmp = w.cub_bytes;
  P3D_CUDA_CHECK(cub::DeviceRadixSort::SortKeys(w.cub_tmp, tmp, w.keys, w.sorted, at.N, 0, 32 + at.ab, st));
  ap_gather_kernel<<<div_up(nms_pre_max_size, 128), 128, 0, st>>>(cls, box, dir, anchors, at, w);
  P3D_LAUNCH_CHECK();
  ap_nms_mask_kernel<<<dim3(at.cbmax, at.cbmax), 64, 0, st>>>(at, w);
  P3D_LAUNCH_CHECK();
  ap_greedy_kernel<<<1, 256, static_cast<size_t>(at.cbmax) * 8, st>>>(at, w);
  P3D_LAUNCH_CHECK();
  ap_emit_kernel<<<1, kEmitThreads, 0, st>>>(at, w, boxes_out, scores_out, reinterpret_cast<long long *>(labels_out),
                                             anchor_index_out, counts_out);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}
