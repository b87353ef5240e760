"""ctypes binding of libp3d_b200.so (the C ABI in include/p3d_b200.h).

There is NO CPU fallback: if the CUDA library is missing or a tensor is not on a CUDA device the
call raises.  torch is used only as the device-memory / stream provider (the role Paddle's
allocator plays under the real custom-op glue, see INTEGRATION.md).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libp3d_b200.so")
_lib = None

c_f32p = C.c_void_p
_i64 = C.c_int64
_int = C.c_int
_f = C.c_float
_sz = C.c_size_t
_vp = C.c_void_p

# name -> (restype, argtypes); must list every symbol declared in include/p3d_b200.h
SIGNATURES = {
    "p3d_status_string": (C.c_char_p, [_int]),
    "p3d_last_cuda_error": (_int, []),
    "p3d_abi_version": (_int, []),
    "p3d_hard_voxelize_workspace_bytes": (_sz, [_i64, _int, _int]),
    "p3d_hard_voxelize": (_int, [_vp, _i64, _int, _vp, _vp, _int, _int, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "p3d_voxelize_mean": (_int, [_vp, _i64, _int, _vp, _vp, _int, _int, _int, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "p3d_voxel_mean": (_int, [_vp, _vp, _vp, _int, _int, _int, _vp, _vp]),
    "p3d_scatter_dense_workspace_bytes": (_sz, [_int, _int, _int, _int]),
    "p3d_scatter_dense": (_int, [_vp, _vp, _vp, _int, _int, _int, _int, _int, _int, _int, _vp, _vp, _sz, _vp]),
    "p3d_bev_pool_v2": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _vp, _i64, _vp]),
    "p3d_bev_pool_v2_bkwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _vp, _i64, _vp, _i64, _vp]),
    "p3d_boxes_overlap_bev": (_int, [_vp, _int, _vp, _int, _vp, _vp]),
    "p3d_boxes_iou_bev": (_int, [_vp, _int, _vp, _int, _vp, _vp]),
    "p3d_nms_workspace_bytes": (_sz, [_int]),
    "p3d_nms": (_int, [_vp, _int, _f, _int, _vp, _vp, _vp, _sz, _vp]),
    "p3d_centerpoint_postprocess_workspace_bytes": (_sz, [_int, _int, _int, _int, _int]),
    "p3d_centerpoint_postprocess": (_int, [_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _vp, _vp, _vp, _vp,
                                           _int, _f, _f, _int, _int, _int, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "p3d_anchor_head_postprocess_workspace_bytes": (_sz, [_int, _int, _int, _int]),
    "p3d_anchor_head_postprocess": (_int, [_vp, _vp, _vp, _int, _int, _int, _int, _vp, _vp, _vp, _vp, _int, _int, _f, _f,
                                           _f, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "p3d_sparse_rulebook_workspace_bytes": (_sz, [_i64, _i64]),
    "p3d_sparse_rulebook_subm": (_int, [_vp, _vp, _i64, _int, _vp, _vp, _vp, _vp, _sz, _vp]),
    "p3d_sparse_rulebook_conv": (_int, [_vp, _vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _sz,
                                        _vp]),
    "p3d_sparse_table_bytes": (_sz, [_i64]),
    "p3d_sparse_table_build": (_int, [_vp, _vp, _i64, _int, _vp, _vp, _sz, _vp]),
    "p3d_sparse_rulebook_subm_t": (_int, [_vp, _vp, _i64, _int, _vp, _vp, _vp, _sz, _vp, _vp]),
    "p3d_sparse_rulebook_conv_t": (_int, [_vp, _vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp, _i64, _vp, _sz,
                                          _vp, _vp]),
    "p3d_sparse_rulebook_level_t": (_int, [_vp, _vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp, _i64, _vp, _sz,
                                           _vp, _vp, _vp, _vp]),
    "p3d_sparse_affine_act": (_int, [_vp, _vp, _i64, _int, _vp, _vp, _vp, _int, _vp, _vp]),
    "p3d_sparse_conv_packed_weight_bytes": (_sz, [_int, _int, _int]),
    "p3d_sparse_conv_pack_weights": (_int, [_vp, _int, _int, _int, _vp, _vp]),
    "p3d_rows_convert_layout": (_int, [_vp, _int, _vp, _i64, _int, _vp, _vp]),
    "p3d_sparse_conv_gather_gemm_split": (_int, [_vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _int, _vp,
                                                 _vp, _vp]),
    "p3d_sparse_conv_gather_gemm_split_ws": (_int, [_vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _int, _vp,
                                                    _vp, _vp, _sz, _vp]),
    "p3d_sparse_conv_gather_gemm_split_tma": (_int, [_vp, _i64, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _int,
                                                     _vp, _vp, _vp, _sz, _vp]),
    "p3d_sparse_conv_splitk_workspace_bytes": (_sz, [_i64, _int, _int]),
    "p3d_sparse_conv_small_cin_h16": (_int, [_vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp, _int, _vp, _vp, _vp, _vp]),
    "p3d_sparse_rows_to_pixel_h16": (_int, [_vp, _vp, _vp, _int, _int, _int, _int, _int, _int, _vp, _vp]),
    "p3d_sparse_conv_f16_packed_weight_bytes": (_sz, [_int, _int, _int]),
    "p3d_sparse_conv_f16_pack_weights": (_int, [_vp, _int, _int, _int, _vp, _vp, _vp]),
    "p3d_rows_convert_h16": (_int, [_vp, _int, _vp, _i64, _int, _vp, _vp, _vp]),
    "p3d_sparse_conv_f16_workspace_bytes": (_sz, [_i64, _int, _int]),
    "p3d_sparse_conv_f16": (_int, [_vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _int, _vp, _vp, _vp, _sz,
                                   _int, _vp, _vp]),
    "p3d_sparse_conv_wm_packed_weight_bytes": (_sz, [_int, _int, _int]),
    "p3d_sparse_conv_wm_pack_weights": (_int, [_vp, _int, _int, _int, _vp, _vp, _vp]),
    "p3d_sparse_conv_wm_workspace_bytes": (_sz, [_i64, _int]),
    "p3d_sparse_conv_wm": (_int, [_vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _int, _vp, _vp, _vp, _sz,
                                  _vp, _vp]),
    "p3d_nchw_to_pixel_split": (_int, [_vp, _int, _int, _int, _int, _vp, _vp]),
    "p3d_dense_conv2d_packed_weight_bytes": (_sz, [_int, _int, _int, _int]),
    "p3d_pillar_feature_net": (_int, [_vp, _vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "p3d_pillar_feature_net_pixel_h16": (_int, [_vp, _vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _vp, _int,
                                                _int, _int, _vp, _vp, _vp]),
    "p3d_head_final_conv": (_int, [_vp, _int, _int, _int, _int, _int, _int, _vp, _vp, _vp, _vp, _int, _vp, _vp]),
    "p3d_head_final_conv_h16": (_int, [_vp, _int, _int, _int, _int, _int, _int, _vp, _vp, _vp, _vp, _int, _vp, _vp]),
    "p3d_nchw_to_pixel_h16": (_int, [_vp, _int, _int, _int, _int, _vp, _vp, _vp]),
    "p3d_pixel_h16_to_nchw": (_int, [_vp, _int, _int, _int, _int, _vp, _vp]),
    "p3d_dense_conv2d_f16_packed_weight_bytes": (_sz, [_int, _int, _int, _int]),
    "p3d_dense_conv2d_f16_pack_weights": (_int, [_vp, _int, _int, _int, _vp, _vp, _vp]),
    "p3d_bev_pool_prepare_workspace_bytes": (_sz, [_i64]),
    "p3d_bev_pool_prepare": (_int, [_vp, _int, _int, _int, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                    _vp]),
    "p3d_head_out_conv_f16": (_int, [_vp, _int, _int, _int, _int, _int, _int, _vp, _vp, _vp, _vp, _vp, _int, _vp, _vp]),
    "p3d_grouped_head_conv_f16": (_int, [_vp, _int, _int, _int, _int, _int, _int, _vp, _vp, _vp, _vp, _int, _vp, _vp, _vp]),
    "p3d_dense_conv2d_f16": (_int, [_vp, _int, _int, _int, _int, _vp, _int, _int, _int, _int, _int, _int, _int, _vp, _vp,
                                    _int, _vp, _int, _int, _vp, _int, _int, _vp, _vp]),
    "p3d_dense_conv2d_split": (_int, [_vp, _int, _int, _int, _int, _vp, _int, _int, _int, _int, _int, _int, _int, _vp, _vp,
                                      _int, _vp, _int, _int, _vp, _vp]),
    "p3d_sparse_conv_gather_gemm_tf32x3_ws": (_int, [_vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _int, _vp,
                                                     _vp, _sz, _vp]),
    "p3d_sparse_conv_gather_gemm": (_int, [_vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _int, _int,
                                           _vp, _vp]),
}


class P3DError(RuntimeError):
    pass


def lib():
    """Load the CUDA library; fail loudly when it has not been built (no fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise P3DError("libp3d_b200.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(paddle3d_b200 has no CPU or library fallback)")
        _lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(_lib, name)
            fn.restype = res
            fn.argtypes = args
    return _lib


_DEBUG_SYNC = bool(os.environ.get("P3D_DEBUG_SYNC"))


def check(rc, what):
    if _DEBUG_SYNC and rc == 0:  # debugging aid: surface asynchronous kernel faults at the call that caused them
        import torch
        try:
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            raise P3DError("%s: kernel fault (%s)" % (what, e))
    if rc != 0:
        l = lib()
        msg = l.p3d_status_string(rc).decode()
        extra = " (cudaError %d)" % l.p3d_last_cuda_error() if rc == -3 else ""
        raise P3DError("%s failed: %s%s" % (what, msg, extra))


def fptr(arr):
    """Host float/int array (ctypes array) -> void*"""
    return C.cast(arr, C.c_void_p)


def host_floats(vals):
    return (C.c_float * len(vals))(*[float(v) for v in vals])


def host_ints(vals):
    return (C.c_int * len(vals))(*[int(v) for v in vals])
