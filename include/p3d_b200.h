/*
 * p3d_b200.h — C ABI of libp3d_b200.so: the B200 (sm_100a) implementation of Paddle3D's
 * point-cloud-to-BEV hot path.  This is the drop-in boundary: every entry point below is what a
 * Paddle custom-op kernel function (PD_BUILD_OP ... SetKernelFn) for this path binds to; the
 * reference interface each one replaces is cited as file:line under PaddlePaddle/Paddle3D @ 3259dabe.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch/paddle types.
 *   - unless a name ends in `_host`, every data pointer is a DEVICE pointer; attribute arrays
 *     (voxel_size, point_cloud_range, ...) are HOST pointers read before the launch.
 *   - `stream` is a cudaStream_t passed as void*.  Calls only enqueue work: they never allocate,
 *     never synchronise and never touch the default stream.  Data-dependent counts are written to
 *     device scalars; the caller reads them back when (and if) it needs them.
 *   - scratch memory is caller-provided: `p3d_<op>_workspace_bytes(...)` gives the size, any
 *     256-byte aligned device buffer of at least that size works, contents need not be preserved.
 *   - return value: 0 on success, negative p3d_status on failure (never throws).
 *     p3d_status_string() gives the message a PD_THROW would carry.
 */
#ifndef P3D_B200_H_
#define P3D_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void *p3d_stream_t; /* cudaStream_t */

enum p3d_status {
  P3D_OK = 0,
  P3D_ERR_INVALID_ARG = -1,   /* bad shape / null pointer / unsupported attribute */
  P3D_ERR_WORKSPACE = -2,     /* workspace_bytes smaller than p3d_*_workspace_bytes() */
  P3D_ERR_CUDA = -3,          /* a CUDA runtime call or launch failed (see p3d_last_cuda_error) */
  P3D_ERR_UNSUPPORTED = -4    /* valid in the reference but outside this build's limits */
};

const char *p3d_status_string(int status);
int p3d_last_cuda_error(void); /* cudaError_t of the last P3D_ERR_CUDA on this thread */
int p3d_abi_version(void);

/* ---------------------------------------------------------------------------------------------
 * hard_voxelize      replaces paddle3d/ops/voxel/voxelize_op.cc:149-166 (op `hard_voxelize`,
 *                    registration :183-191; CUDA path voxelize_op.cu:208-346).
 * Semantics are those of the reference CPU kernel (voxelize_op.cc:19-82), deterministically:
 * voxels numbered in first-appearance order of their first point, capped at max_voxels; each voxel
 * keeps its first max_points points in input order.
 *   points               [num_points, num_point_dim] fp32 (num_point_dim >= 3)
 *   voxel_size_host[3], point_cloud_range_host[6]     attrs
 *   voxels               [max_voxels, max_points, num_point_dim] fp32, fully written (zero padded)
 *   coords               [max_voxels, 3] int32 (z, y, x), zero beyond num_voxels
 *   num_points_per_voxel [max_voxels] int32, zero beyond num_voxels
 *   num_voxels           [1] int32
 * ------------------------------------------------------------------------------------------- */
size_t p3d_hard_voxelize_workspace_bytes(int64_t num_points, int max_points, int max_voxels);
int p3d_hard_voxelize(const float *points, int64_t num_points, int num_point_dim, const float *voxel_size_host,
                      const float *point_cloud_range_host, int max_points, int max_voxels, float *voxels,
                      int32_t *coords, int32_t *num_points_per_voxel, int32_t *num_voxels, void *workspace,
                      size_t workspace_bytes, p3d_stream_t stream);

/* Fused front end used by the CenterPoint pipeline: hard_voxelize + VoxelMean
 * (paddle3d/models/voxel_encoders/voxel_encoder.py:49-57) + HardVoxelizer's batch-id pad
 * (paddle3d/models/voxelizers/voxelize.py:39-58) without materialising the padded voxels tensor.
 *   mean   [max_voxels, num_point_dim] fp32 (rows >= num_voxels zero)
 *   coors4 [max_voxels, 4] int32 (batch_id, z, y, x)  */
int p3d_voxelize_mean(const float *points, int64_t num_points, int num_point_dim, const float *voxel_size_host,
                      const float *point_cloud_range_host, int max_points, int max_voxels, int batch_id,
                      float *mean, int32_t *coors4, int32_t *num_points_per_voxel, int32_t *num_voxels,
                      void *workspace, size_t workspace_bytes, p3d_stream_t stream);

/* VoxelMean alone: voxels [num_voxels_cap, max_points, F] -> mean [num_voxels_cap, F]; rows whose
 * index >= *num_voxels_dev (device scalar, may be NULL = all rows) are written as zero. */
int p3d_voxel_mean(const float *voxels, const int32_t *num_points_per_voxel, const int32_t *num_voxels_dev,
                   int num_voxels_cap, int max_points, int num_point_dim, float *mean, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * pillar_scatter / sparse to_dense     replaces PointPillarsScatter.forward_batch
 *   (paddle3d/models/middle_encoders/pillar_scatter.py:57-105: zeros + paddle.scatter + transpose)
 *   and SparseResNet3D's to_dense + transpose + reshape (sparse_resnet.py:202-206).
 *   feats  [n, C] fp32;  coords [n, 4] int32 (batch, z, y, x);  n_dev: device count (NULL = n_cap)
 *   out    [batch, C, D, ny, nx] fp32 fully written; a pillar canvas is the D == 1 case and uses
 *          index y*nx + x (z ignored), later rows win on duplicate cells.
 * ------------------------------------------------------------------------------------------- */
size_t p3d_scatter_dense_workspace_bytes(int batch, int D, int ny, int nx);
int p3d_scatter_dense(const float *feats, const int32_t *coords, const int32_t *n_dev, int n_cap, int C,
                      int batch, int D, int ny, int nx, int use_z, float *out, void *workspace,
                      size_t workspace_bytes, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * bev_pool_v2 / bev_pool_v2_bkwd      replace paddle3d/ops/bev_pool_v2/bev_pool.cc:30-54, :56-96
 *   (registrations :111-118 and ops/bev_pool_v2_backward/bev_pool_bkwd.cc:75-80; kernels
 *   bev_pool_cuda.cu:18-96).  NOTE the reference argument order: lengths before starts.
 *   depth [B*N, D, H, W] fp32 (flat-indexed by ranks_depth); feat [B*N, H, W, C] fp32;
 *   ranks_* [n_points] int32; interval_* [n_intervals] int32; out [out_numel] fp32 zero-filled here.
 * ------------------------------------------------------------------------------------------- */
int p3d_bev_pool_v2(const float *depth, const float *feat, const int32_t *ranks_depth, const int32_t *ranks_feat,
                    const int32_t *ranks_bev, const int32_t *interval_lengths, const int32_t *interval_starts,
                    int n_intervals, int c, float *out, int64_t out_numel, p3d_stream_t stream);
int p3d_bev_pool_v2_bkwd(const float *out_grad, const float *depth, const float *feat, const int32_t *ranks_depth,
                         const int32_t *ranks_feat, const int32_t *ranks_bev, const int32_t *interval_lengths,
                         const int32_t *interval_starts, int n_intervals, int c, float *depth_grad,
                         int64_t depth_numel, float *feat_grad, int64_t feat_numel, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * iou3d_nms      replaces paddle3d/ops/iou3d_nms/iou3d_nms.cpp:44-204 (registrations
 *                iou3d_nms_api.cpp:73-108).  boxes are [n, 7] = x, y, z, dx, dy, dz, heading.
 * ------------------------------------------------------------------------------------------- */
int p3d_boxes_overlap_bev(const float *boxes_a, int num_a, const float *boxes_b, int num_b, float *overlap,
                          p3d_stream_t stream);
int p3d_boxes_iou_bev(const float *boxes_a, int num_a, const float *boxes_b, int num_b, float *iou,
                      p3d_stream_t stream);
/* nms_gpu / nms_normal_gpu: boxes already sorted by score.  keep [n] int32 (first *num_keep valid),
 * num_keep [1] int32 — both on the DEVICE (the reference finishes on the host; here the greedy
 * reduction runs on the GPU with no sync).  normal != 0 selects the axis-aligned IoU. */
size_t p3d_nms_workspace_bytes(int n);
int p3d_nms(const float *boxes, int n, float nms_overlap_thresh, int normal, int32_t *keep, int32_t *num_keep,
            void *workspace, size_t workspace_bytes, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * centerpoint_postprocess      replaces paddle3d/ops/centerpoint_postprocess/postprocess.cc:34-104
 *                              (postprocess_gpu, postprocess.cu:104-280), batch size 1.
 *   hm/reg/height/dim/vel/rot: HOST arrays of T device pointers to the per-task NCHW tensors
 *   hm_channels_host[T]; attrs as in the op.  num_classes_host[T] are the label offsets.
 *   Outputs (device), sized for the worst case rows_cap = T * max(nms_post_max_size, 1):
 *     bboxes [rows_cap, 9 or 7], scores [rows_cap], labels [rows_cap] int64,
 *     counts [T + 1] int32: rows per task, then the total number of valid rows.
 *   Score-sort tie order is defined as ascending cell index.
 * ------------------------------------------------------------------------------------------- */
size_t p3d_centerpoint_postprocess_workspace_bytes(int num_tasks, int feat_h, int feat_w, int nms_pre_max_size,
                                                    int nms_post_max_size);
int p3d_centerpoint_postprocess(int num_tasks, const float *const *hm, const int32_t *hm_channels_host,
                                const float *const *reg, const float *const *height, const float *const *dim,
                                const float *const *vel, const float *const *rot, int feat_h, int feat_w,
                                const float *voxel_size_host, const float *point_cloud_range_host,
                                const float *post_center_range_host, const int32_t *num_classes_host,
                                int down_ratio, float score_threshold, float nms_iou_threshold,
                                int nms_pre_max_size, int nms_post_max_size, int with_velocity, float *bboxes,
                                float *scores, int64_t *labels, int32_t *counts, void *workspace,
                                size_t workspace_bytes, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * anchor_head_postprocess      the SSD head's post-processing of PointPillars / SECOND (the reference runs it as Python
 *                              over Paddle ops: pointpillars.py:105-129 + rotate_nms_pcdet), batch size 1.
 *   cls [A*C, H, W], box [A*7, H, W], dir [A*2, H, W]: fp32 NCHW planes on the device; anchor i = (y * W + x) * A + a
 *   reads cls[a*C + c], box[a*7 + k], dir[a*2 + d].  anchors [H*W*A, 7] (x, y, z, w, l, h, r) fp32 on the device.
 *   Anchor mask (skipped when anchor_cells is NULL or anchor_area_threshold < 0): anchor_cells [H*W*A] int4 (x0, y0, x1,
 *   y1) are the static clipped cell bounds of fused_get_anchors_area; the pillar occupancy of coors [num_voxels, 4]
 *   (b, z, y, x) int32 on a grid_ny x grid_nx grid gives each anchor an area, and it is kept iff area > threshold.
 *   Candidates: max sigmoid score >= score_threshold.  The first nms_pre_max_size in descending score order (ties: ascending
 *   anchor index) are decoded (second_box_decode), suppressed by rotated NMS (rotate_nms_pcdet's box layout), cut to
 *   nms_post_max_size, direction-fixed and filtered by post_center_range_host (6 floats, inclusive; NULL: no filter).
 *   Outputs (device), sized for nms_post_max_size rows: boxes [., 7], scores, labels int64, anchor_index_out int32 (may be
 *   NULL), counts [2] int32 = (candidates, rows).  No row is emitted when nothing passes.
 * ------------------------------------------------------------------------------------------- */
size_t p3d_anchor_head_postprocess_workspace_bytes(int num_anchors, int grid_ny, int grid_nx, int nms_pre_max_size);
int p3d_anchor_head_postprocess(const float *cls, const float *box, const float *dir, int H, int W, int A, int C,
                                const float *anchors, const int32_t *anchor_cells, const int32_t *coors,
                                const int32_t *num_voxels_dev, int grid_ny, int grid_nx, float anchor_area_threshold,
                                float score_threshold, float iou_threshold, int nms_pre_max_size, int nms_post_max_size,
                                const float *post_center_range_host, float *boxes_out, float *scores_out,
                                int64_t *labels_out, int32_t *anchor_index_out, int32_t *counts_out, void *workspace,
                                size_t workspace_bytes, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Sparse 3-D convolution      replaces the paddle.sparse.nn layer calls made by SparseResNet3D /
 *   SparseNet3D (paddle3d/models/middle_encoders/sparse_resnet.py:31-60,84-111,125-206;
 *   sparsenet.py:38-52,75-155): SubmConv3D / Conv3D (+ BatchNorm(eval) + residual add + ReLU fused).
 *
 * Rulebook ("neighbour map") build.  coords are [n, 4] int32 (batch, z, y, x); spatial = (D, H, W).
 *   p3d_sparse_rulebook_subm : nbr [n_cap, K] int32, nbr[i][k] = input row at coord(i) - pad + k or -1
 *                              (K = kD*kH*kW, pad = k/2; shared by every SubM layer of a stage).
 *   p3d_sparse_rulebook_conv : strided Conv3D: writes the output coordinate list out_coords
 *                              [out_cap, 4] (site order is unspecified), the device counters
 *                              n_out_dev (int32[4]) and nbr [out_cap, K] with
 *                              nbr[o][k] = input row at o*stride - pad + k or -1.
 *   n_in_dev / n_out_dev are device scalars so the whole backbone runs without a host sync.
 *   n_out_dev[0] = number of output sites (clamped to out_cap), n_out_dev[1] = 1 if sites were
 *   dropped because out_cap was too small, n_out_dev[2] = unclamped count (a lower bound once the
 *   dedup table itself is full), n_out_dev[3] = internal table-full flag.
 * ------------------------------------------------------------------------------------------- */
size_t p3d_sparse_rulebook_workspace_bytes(int64_t n_in_cap, int64_t n_out_cap);
int p3d_sparse_rulebook_subm(const int32_t *coords, const int32_t *n_in_dev, int64_t n_in_cap, int batch,
                             const int *spatial_host, const int *ksize_host, int32_t *nbr, void *workspace,
                             size_t workspace_bytes, p3d_stream_t stream);
int p3d_sparse_rulebook_conv(const int32_t *coords, const int32_t *n_in_dev, int64_t n_in_cap, int batch,
                             const int *spatial_host, const int *ksize_host, const int *stride_host,
                             const int *pad_host, int32_t *out_coords, int32_t *n_out_dev, int64_t out_cap,
                             int32_t *nbr, void *workspace, size_t workspace_bytes, p3d_stream_t stream);

/* Caller-owned coordinate tables (one per index set / resolution level): the same rulebooks with every level's
 * table built exactly once per frame.  p3d_sparse_table_build hashes an index set's coordinates;
 * p3d_sparse_rulebook_subm_t only looks neighbours up in it; p3d_sparse_rulebook_conv_t looks the inputs up in
 * table_in and leaves in table_out the table of the OUTPUT index set (a by-product of enumerating its sites), ready
 * for the next stage.  Tables are p3d_sparse_table_bytes(rows_cap) bytes, 16-byte aligned. */
size_t p3d_sparse_table_bytes(int64_t rows_cap);
int p3d_sparse_table_build(const int32_t *coords, const int32_t *n_dev, int64_t n_cap, int batch,
                           const int *spatial_host, void *table, size_t table_bytes, p3d_stream_t stream);
int p3d_sparse_rulebook_subm_t(const int32_t *coords, const int32_t *n_dev, int64_t n_cap, int batch,
                               const int *spatial_host, const int *ksize_host, const void *table, size_t table_bytes,
                               int32_t *nbr, p3d_stream_t stream);
int p3d_sparse_rulebook_conv_t(const int32_t *coords, const int32_t *n_in_dev, int64_t n_in_cap, int batch,
                               const int *spatial_host, const int *ksize_host, const int *stride_host,
                               const int *pad_host, const void *table_in, size_t table_in_bytes, int32_t *out_coords,
                               int32_t *n_out_dev, int64_t out_cap, void *table_out, size_t table_out_bytes,
                               int32_t *nbr, p3d_stream_t stream);

/* One resolution level in two launches: p3d_sparse_rulebook_conv_t plus, when nbr_subm is given, the SubM neighbour map
 * [out_cap, prod(subm_ksize)] of the NEW level (odd kernel, "same" padding) looked up in table_out - what a following
 * p3d_sparse_rulebook_subm_t on the output index set would return. */
int p3d_sparse_rulebook_level_t(const int32_t *coords, const int32_t *n_in_dev, int64_t n_in_cap, int batch,
                                const int *spatial_host, const int *ksize_host, const int *stride_host,
                                const int *pad_host, const void *table_in, size_t table_in_bytes, int32_t *out_coords,
                                int32_t *n_out_dev, int64_t out_cap, void *table_out, size_t table_out_bytes,
                                int32_t *nbr, const int *subm_ksize_host, int32_t *nbr_subm, p3d_stream_t stream);

/* Unfused elementwise epilogue (BatchNorm(eval) / sparse.add / ReLU on a materialised tensor):
 *   out[r, c] = act(x[r, c] * scale[c] + shift[c] (+ residual[r, c])); out may alias x. */
int p3d_sparse_affine_act(const float *x, const int32_t *n_dev, int64_t n_cap, int C, const float *scale,
                          const float *shift, const float *residual, int relu, float *out, p3d_stream_t stream);

/* Gather-GEMM-scatter in output-stationary form:
 *   out[o, :] = act( (sum_k in[nbr[o][k], :] @ W[k]) * scale + shift (+ residual[o, :]) )
 *   in [n_in, Cin] fp32; W [K, Cin, Cout] fp32 (Paddle's [kD,kH,kW,Cin,Cout]); scale/shift [Cout]
 *   (BatchNorm(eval) and conv bias folded by the caller; NULL = identity); residual [n_out, Cout] or
 *   NULL; relu != 0 applies max(.,0).  n_out_dev: device row count (NULL = n_out_cap rows).
 *   precision: P3D_CONV_FP32 = fp32 FMA on CUDA cores; P3D_CONV_TF32X3 = tcgen05 tensor cores with
 *   3xTF32 split accumulation in TMEM (fp32-level accuracy). */
enum p3d_conv_precision { P3D_CONV_FP32 = 0, P3D_CONV_TF32X3 = 1 };
/* Weight pre-pack for P3D_CONV_TF32X3 (once per layer): splits W [K, Cin, Cout] into tf32 hi / lo and lays it out
 * as the shared-memory image the tensor-core kernel streams with cp.async.bulk.  Needs Cin, Cout multiples of
 * 16 (Cin multiple of 32 above 32); returns P3D_ERR_UNSUPPORTED otherwise (use P3D_CONV_FP32 for such layers).
 * With precision == P3D_CONV_TF32X3 the `weight` argument of p3d_sparse_conv_gather_gemm is this packed buffer. */
size_t p3d_sparse_conv_packed_weight_bytes(int K, int Cin, int Cout);
int p3d_sparse_conv_pack_weights(const float *weight, int K, int Cin, int Cout, float *packed, p3d_stream_t stream);
int p3d_sparse_conv_gather_gemm(const float *in, const int32_t *nbr, const int32_t *n_out_dev, int64_t n_out_cap,
                                int K, int Cin, int Cout, const float *weight, const float *scale,
                                const float *shift, const float *residual, int relu, int precision, float *out,
                                p3d_stream_t stream);

/* Tensor-core gather-GEMM with split-K over the kernel taps for the wide layers (Cout >= 64): layers with few
 * 128-row tiles are spread over 2 - 3 CTAs per tile; partial sums go to the caller's scratch slabs and are added in a
 * fixed order by a finalize pass that also applies the epilogue (deterministic).  Same contract as
 * p3d_sparse_conv_gather_gemm(precision = P3D_CONV_TF32X3); with workspace == NULL it runs unsplit. */
size_t p3d_sparse_conv_splitk_workspace_bytes(int64_t n_out_cap, int Cin, int Cout);
int p3d_sparse_conv_gather_gemm_tf32x3_ws(const float *in, const int32_t *nbr, const int32_t *n_out_dev,
                                          int64_t n_out_cap, int K, int Cin, int Cout, const float *packed_weight,
                                          const float *scale, const float *shift, const float *residual, int relu,
                                          float *out, void *workspace, size_t workspace_bytes, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Split-row activations for the tensor-core path.  A "split" row tensor stores every row as its tf32 hi half
 * followed by its tf32 lo half: [n][2][C] fp32 words (x ~= hi + lo, error <= 2^-22 |x|).  Keeping activations in
 * this form between sparse-conv layers moves the 3xTF32 split out of the gather loop (paid once per produced
 * element instead of once per gathering neighbour) and lets the kernel gather with cp.async.
 *   p3d_rows_convert_layout: src_layout 0 = fp32 rows [n, C] -> split; 1 = split -> fp32 rows (hi + lo).
 *   p3d_sparse_conv_gather_gemm_split: same contract as p3d_sparse_conv_gather_gemm(precision = TF32X3) with
 *     in_split [n_in][2][Cin], residual_split [n_out][2][Cout] or NULL, packed weights
 *     (p3d_sparse_conv_pack_weights), and out_f32 [n_out, Cout] and / or out_split [n_out][2][Cout] (either may be
 *     NULL, not both).  Persistent grid sized to the device row count.
 *   p3d_sparse_conv_gather_gemm_split_ws: the same with a scratch buffer of
 *     p3d_sparse_conv_splitk_workspace_bytes(n_out_cap, Cin, Cout) bytes; when present the wide layers run split-K over
 *     taps (partial sums in the scratch slabs, added in slab order by a finalize kernel: deterministic).
 * ------------------------------------------------------------------------------------------- */
int p3d_rows_convert_layout(const float *src, int src_layout, const int32_t *n_dev, int64_t n_cap, int C, float *dst,
                            p3d_stream_t stream);
int p3d_sparse_conv_gather_gemm_split(const float *in_split, const int32_t *nbr, const int32_t *n_out_dev,
                                      int64_t n_out_cap, int K, int Cin, int Cout, const float *packed_weight,
                                      const float *scale, const float *shift, const float *residual_split, int relu,
                                      float *out_f32, float *out_split, p3d_stream_t stream);
int p3d_sparse_conv_gather_gemm_split_ws(const float *in_split, const int32_t *nbr, const int32_t *n_out_dev,
                                         int64_t n_out_cap, int K, int Cin, int Cout, const float *packed_weight,
                                         const float *scale, const float *shift, const float *residual_split, int relu,
                                         float *out_f32, float *out_split, void *workspace, size_t workspace_bytes,
                                         p3d_stream_t stream);
/* EXPERIMENTAL (round-2 groundwork, not on the default path): the same layer with the row gather done by the TMA
 * engine (cp.async.bulk.tensor tile::gather4 through a tensor map over in_split [n_in_rows][2*Cin]) instead of
 * cp.async from 8 producer warps.  Cin >= 32 only (P3D_ERR_UNSUPPORTED otherwise). */
int p3d_sparse_conv_gather_gemm_split_tma(const float *in_split, int64_t n_in_rows, const int32_t *nbr,
                                          const int32_t *n_out_dev, int64_t n_out_cap, int K, int Cin, int Cout,
                                          const float *packed_weight, const float *scale, const float *shift,
                                          const float *residual_split, int relu, float *out_f32, float *out_split,
                                          void *workspace, size_t workspace_bytes, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * fp16-pair ("H16") activations: the default tensor-core path of the sparse layers (csrc/sparse_conv_f16.cu).
 * x = hi + lo' * 2^-11 with hi = fp16(x), lo' = fp16((x - hi) * 2^11): the same 22 significant bits as the tf32 pair
 * in half the bytes (a row of C channels is 4*C bytes: groups of KC = min(C, 32) channels, each [hi KC | lo' KC] halfs).
 * Valid for |x| < 65504; values outside are saturated and bit 0 of *status_dev is set (use the tf32 split path for
 * such data).  Same layer contract as p3d_sparse_conv_gather_gemm_split (paddle.sparse.nn.SubmConv3D / Conv3D +
 * BatchNorm(eval) + add + ReLU, sparse_resnet.py:31-60,84-111):
 *   p3d_sparse_conv_f16_pack_weights   W[K][Cin][Cout] fp32 -> k-blocks of the (hi | lo') weight image
 *   p3d_rows_convert_h16               to_h16 != 0: fp32 rows [n, C] -> H16 rows; 0: H16 rows -> fp32 rows
 *   p3d_sparse_conv_f16                persistent kernel, split-K over taps chosen on the device (up to max_splits,
 *                                      bounded by the workspace); workspace = p3d_sparse_conv_f16_workspace_bytes(...)
 *                                      bytes whose first align_up(tiles * 4) bytes (tickets) must be ZERO on first use
 *                                      (the kernel leaves them zero); workspace NULL or max_splits <= 1: no split.
 * ------------------------------------------------------------------------------------------- */
/* fp16-pair plumbing around the tensor-core layers: the 5-channel input layer emitting pair rows directly, and the last
 * level's rows scattered straight into the pixel H16 image [batch, ny, nx][D * C] the dense RPN reads (the fp16-pair form
 * of to_dense + transpose + reshape, sparse_resnet.py:202-206; duplicates impossible: sites are unique). */
int p3d_sparse_conv_small_cin_h16(const float *in, const int32_t *nbr, const int32_t *n_out_dev, int64_t n_out_cap, int K,
                                  int Cin, int Cout, const float *weight, const float *scale, const float *shift, int relu,
                                  float *out_f32, void *out_h16, int32_t *status_dev, p3d_stream_t stream);
int p3d_sparse_rows_to_pixel_h16(const void *rows_h16, const int32_t *coords, const int32_t *n_dev, int n_cap, int C,
                                 int batch, int D, int ny, int nx, void *out_pixel_h16, p3d_stream_t stream);
size_t p3d_sparse_conv_f16_packed_weight_bytes(int K, int Cin, int Cout);
int p3d_sparse_conv_f16_pack_weights(const float *weight, int K, int Cin, int Cout, void *packed, int32_t *status_dev,
                                     p3d_stream_t stream);
int p3d_rows_convert_h16(const void *src, int to_h16, const int32_t *n_dev, int64_t n_cap, int C, void *dst,
                         int32_t *status_dev, p3d_stream_t stream);
size_t p3d_sparse_conv_f16_workspace_bytes(int64_t n_out_cap, int Cout, int max_splits);
int p3d_sparse_conv_f16(const void *in_h16, const int32_t *nbr, const int32_t *n_out_dev, int64_t n_out_cap, int K,
                        int Cin, int Cout, const void *packed_weight, const float *scale, const float *shift,
                        const void *residual_h16, int relu, float *out_f32, void *out_h16, void *workspace,
                        size_t workspace_bytes, int max_splits, int32_t *status_dev, p3d_stream_t stream);

/* Narrow layers (Cin, Cout) in {(16,16), (16,32), (32,32)}: register gather + warp MMA (csrc/sparse_conv_wm.cu), same
 * H16 rows in and out, same fused epilogue and the same three-product arithmetic as p3d_sparse_conv_f16; only the weight
 * image differs (mma.sync fragment order, k permuted so that a lane's fragment is 4 contiguous channels of a row).
 * Missing neighbours cost nothing here (predicated-off loads), which is what bounds the tcgen05 kernel at these widths.
 * Work is cut stream-K style into equal (tile, tap) ranges per warp; a tile cut by a range boundary is summed by the last
 * warp to finish it, pieces in warp order (deterministic).  workspace = p3d_sparse_conv_wm_workspace_bytes(...) bytes whose
 * first align_up(ceil(n_out_cap / 16) * 4) bytes (tickets) must be ZERO on first use (the kernel leaves them zero).
 * p3d_sparse_conv_wm_packed_weight_bytes returns 0 for unsupported shapes. */
size_t p3d_sparse_conv_wm_packed_weight_bytes(int K, int Cin, int Cout);
int p3d_sparse_conv_wm_pack_weights(const float *weight, int K, int Cin, int Cout, void *packed, int32_t *status_dev,
                                    p3d_stream_t stream);
size_t p3d_sparse_conv_wm_workspace_bytes(int64_t n_out_cap, int Cout);
int p3d_sparse_conv_wm(const void *in_h16, const int32_t *nbr, const int32_t *n_out_dev, int64_t n_out_cap, int K, int Cin,
                       int Cout, const void *packed_weight, const float *scale, const float *shift,
                       const void *residual_h16, int relu, float *out_f32, void *out_h16, void *workspace,
                       size_t workspace_bytes, int32_t *status_dev, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * SURVEY.md 8f-1 (parity-green, performance not measured yet): dense 2-D convolution on tcgen05 for the RPN / neck /
 * CenterHead (reference: backbones/second_backbone.py:72-120, necks/second_fpn.py:99-160,
 * detection/centerpoint/center_head.py:43-220).  Images are "pixel split rows" [B*H*W][2][C] (the split-row format
 * of the sparse layers with row = pixel).
 *   p3d_nchw_to_pixel_split: fp32 [B, C, H, W] -> pixel split rows.
 *   p3d_dense_conv2d_packed_weight_bytes / p3d_dense_conv2d_split: weights = per N tile (n_tile = 16 | 64 | 128 output
 *     channels, zero-padded) the image p3d_sparse_conv_pack_weights makes of W[tap][Cin][n_tile], tiles concatenated.
 *     up == 1: Conv2D(kh x kw, stride 1 | 2, zero padding pad); up > 1: Conv2DTranspose with kernel = stride = up
 *     (pass kh = kw = stride = up, pad = 0).  Epilogue v * scale[c] + shift[c] (either may be NULL), optional ReLU.
 *     Output: split rows of out_C channels written at column out_c0 (channel concat), and / or fp32 NCHW planes
 *     [B, Cout, out_H, out_W].  Cin % 32 == 0; Cout % 16 == 0 for split-row output.
 * ------------------------------------------------------------------------------------------- */
int p3d_nchw_to_pixel_split(const float *in, int B, int C, int H, int W, float *out_split, p3d_stream_t stream);
size_t p3d_dense_conv2d_packed_weight_bytes(int taps, int Cin, int Cout, int n_tile);
int p3d_dense_conv2d_split(const float *in_split, int B, int H, int W, int Cin, const float *packed_weight, int Cout,
                           int n_tile, int kh, int kw, int stride, int pad, int up, const float *scale,
                           const float *shift, int relu, float *out_split, int out_C, int out_c0, float *out_nchw,
                           p3d_stream_t stream);

/* EXPERIMENTAL (never run on a GPU yet): the grouped 3x3 output convs of CenterHead's SeparateHeads
 * (center_head.py:80-117) as one CUDA-core launch.  in_split: pixel split rows [B*H*W][2][in_C]; group g convolves
 * channels [g*Cin, (g+1)*Cin) with weight [groups][9][Cin][4] (outputs zero-padded to 4) + bias [groups][4] and
 * writes cnt[g] fp32 planes from plane0[g] of out_nchw [B, planes, H, W] (plane0 / cnt are HOST arrays). */
int p3d_head_final_conv(const float *in_split, int B, int H, int W, int in_C, int Cin, int groups, const float *weight,
                        const float *bias, const int32_t *plane0_host, const int32_t *cnt_host, int planes,
                        float *out_nchw, p3d_stream_t stream);
int p3d_head_final_conv_h16(const void *in_h16, int B, int H, int W, int in_C, int Cin, int groups, const float *weight,
                            const float *bias, const int32_t *plane0_host, const int32_t *cnt_host, int planes,
                            float *out_nchw, p3d_stream_t stream);

/* fp16-pair dense convolution (csrc/dense_conv_f16.cu): same layer contract as p3d_dense_conv2d_split on pixel H16
 * rows [B*H*W][C / 32 groups][hi 32 | lo' 32] halfs.  3x3 / stride 1 / pad 1 layers load the haloed tile once per
 * 32-channel group and read the 9 taps through shifted UMMA descriptors; everything else loads one box per tap.
 * mode 0 = auto, 1 = force per-tap loads; m_tiles 0 = auto, 1 or 2 M tiles (8 x 16 pixels each) per work item. */
int p3d_nchw_to_pixel_h16(const float *in, int B, int C, int H, int W, void *out_h16, int32_t *status_dev,
                          p3d_stream_t stream);
int p3d_pixel_h16_to_nchw(const void *in_h16, int B, int C, int H, int W, float *out, p3d_stream_t stream);
size_t p3d_dense_conv2d_f16_packed_weight_bytes(int taps, int Cin, int Cout, int n_tile);
int p3d_dense_conv2d_f16_pack_weights(const float *weight_tci, int taps, int Cin, int n_tile, void *packed,
                                      int32_t *status_dev, p3d_stream_t stream);
/* ---------------------------------------------------------------------------------------------
 * bev_pool rank preparation      replaces LSSViewTransformer.voxel_pooling_prepare_v2
 *   (paddle3d/models/transformers/bevdet_transformer.py:230-274): frustum points coor [B, N, D, H, W, 3] fp32 ->
 *   ranks_bev / ranks_depth / ranks_feat sorted by ranks_bev (ties: ascending point index = stable argsort),
 *   interval_starts / interval_lengths; all outputs int32 [B*N*D*H*W] (capacity), counts_dev = {n_kept, n_intervals}.
 *   Entries beyond the counts are zero.  grid_size_host = (X, Y, Z) cells, lower bound / interval per axis (x, y, z).
 * ------------------------------------------------------------------------------------------- */
size_t p3d_bev_pool_prepare_workspace_bytes(int64_t num_points);
int p3d_bev_pool_prepare(const float *coor, int B, int N, int D, int H, int W, const float *grid_lower_bound_host,
                         const float *grid_interval_host, const int32_t *grid_size_host, int32_t *ranks_bev,
                         int32_t *ranks_depth, int32_t *ranks_feat, int32_t *interval_starts, int32_t *interval_lengths,
                         int32_t *counts_dev, void *workspace, size_t workspace_bytes, p3d_stream_t stream);

/* Grouped 3x3 output convs of the CenterHead (center_head.py:80-117) as one tensor-core launch: group g reads input
 * channels [g * Cin, (g + 1) * Cin) of the in_C-channel H16 image, uses weight tile g (pack with n_tile = 16, columns
 * >= cnt[g] zero), bias [groups][16], and writes cnt[g] fp32 planes from plane0[g] (device int32 arrays). */
int p3d_grouped_head_conv_f16(const void *in_h16, int B, int H, int W, int in_C, int Cin, int groups,
                              const void *packed_weight, const float *bias, const int32_t *plane0_dev,
                              const int32_t *cnt_dev, int planes, float *out_nchw, int32_t *status_dev, p3d_stream_t stream);
/* The same output convs with the 9 taps in the GEMM's N dimension (default for Cin = 32 / 64 / 128 and <= 3 output
 * channels per group; a wider conv is split into several groups over the same input slice): one [256 haloed pixels x Cin]
 * x [Cin x 27] GEMM per 14 x 14 output tile, then every pixel adds its 9 shifted partial sums.  Group g reads input
 * channels [cin0[g], cin0[g] + Cin) (cin0_dev null: g * Cin); packed_weight: per group
 * p3d_dense_conv2d_f16_pack_weights(taps 1, Cin, n_tile 32) of W2[c][tap * 3 + co]; bias [groups][4]. */
int p3d_head_out_conv_f16(const void *in_h16, int B, int H, int W, int in_C, int Cin, int groups, const void *packed_weight,
                          const float *bias, const int32_t *cin0_dev, const int32_t *plane0_dev, const int32_t *cnt_dev,
                          int planes, float *out_nchw, p3d_stream_t stream);
int p3d_dense_conv2d_f16(const void *in_h16, int B, int H, int W, int Cin, const void *packed_weight, int Cout, int n_tile,
                         int kh, int kw, int stride, int pad, int up, const float *scale, const float *shift, int relu,
                         void *out_h16, int out_C, int out_c0, float *out_nchw, int mode, int m_tiles,
                         int32_t *status_dev, p3d_stream_t stream);

/* EXPERIMENTAL (never run on a GPU yet), SURVEY.md 8f-2: PillarFeatureNet with one PFNLayer
 * (models/voxel_encoders/pillar_encoder.py:156-210, :81-106) fused into one launch: voxels [n, M, F] + counts + coors
 * [n, 4] (b, z, y, x) -> pillar features [n, C].  weight [F + 5, C] (paddle.nn.Linear layout, no bias); BatchNorm1D
 * folded by the caller: y = x * bn_scale[c] + bn_shift[c].  Rows >= *num_voxels_dev (if given) are left untouched. */
int p3d_pillar_feature_net(const float *voxels, const int32_t *num_points_per_voxel, const int32_t *coors,
                           const int32_t *num_voxels_dev, int64_t n_cap, int max_points, int num_point_dim,
                           int out_channels, const float *weight, const float *bn_scale, const float *bn_shift,
                           const float *voxel_size_host, const float *point_cloud_range_host, float *out,
                           p3d_stream_t stream);
/* The same layer with PointPillarsScatter and the pixel fp16-pair conversion folded into its epilogue: zeroes the pixel
 * H16 image out_pixel_h16 [batch * ny * nx][C / 32][hi 32 | lo' 32] halfs, then writes each pillar's C channels into the
 * pixel (b * ny + y) * nx + x of its coors (b, z, y, x); z is ignored, rows outside the grid or with b >= batch are
 * skipped.  Cells are unique by construction (hard_voxelize emits one row per cell), so there is no duplicate handling.
 * Same fp32 arithmetic as p3d_pillar_feature_net: the image equals p3d_nchw_to_pixel_h16 of the scattered canvas bit for
 * bit.  |x| > 65504 is saturated and sets bit 0 of *status_dev (may be NULL).  Null pointers or misaligned coors / image
 * (16 bytes) return P3D_ERR_INVALID_ARG; max_points > 64, num_point_dim > 8 or C % 32 != 0 P3D_ERR_UNSUPPORTED. */
int p3d_pillar_feature_net_pixel_h16(const float *voxels, const int32_t *num_points_per_voxel, const int32_t *coors,
                                     const int32_t *num_voxels_dev, int64_t n_cap, int max_points, int num_point_dim,
                                     int out_channels, const float *weight, const float *bn_scale, const float *bn_shift,
                                     const float *voxel_size_host, const float *point_cloud_range_host, int batch, int ny,
                                     int nx, void *out_pixel_h16, int32_t *status_dev, p3d_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* P3D_B200_H_ */
