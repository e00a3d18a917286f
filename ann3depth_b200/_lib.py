"""ctypes binding of liba3d.so (the C-ABI declared in include/a3d.h).

The library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is NO fallback:
if the shared object is missing, or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("A3D_LIB") or os.path.join(_HERE, "liba3d.so")     # A3D_LIB: alternate build (experiments)

A3D_F32, A3D_BF16 = 0, 1
A3D_E4M3 = 3                          # E4M3 codes: the FP8 inference mode
A3D_ENOTSUP = -5
IMPL_AUTO, IMPL_SIMT, IMPL_TC = 0, 1, 2
EPI_RELU, EPI_SIGMOID = 1, 2
OP_FWD, OP_DGRAD, OP_WGRAD = 0, 1, 2
DM_SCALE_NONE, DM_SCALE_MEDIAN = 0, 1
# a3d_depth_metrics slots (A3D_DM_*), in order
DM_SLOTS = ("n", "abs_rel", "sq_rel", "sq", "log", "log_sq", "log10", "delta1", "delta2", "delta3", "nonfinite")


class A3DError(RuntimeError):
    pass


ABI_VERSION = 201          # include/a3d.h A3D_VERSION


class ConvDesc(C.Structure):
    """Mirror of `a3d_conv_desc` (include/a3d.h)."""
    _fields_ = [(n, C.c_int) for n in
                ("N", "H", "W", "C", "K", "R", "S", "stride_h", "stride_w", "pad_t", "pad_l", "P", "Q", "ldy", "impl",
                 "dil_w", "pix_pitch")]


class AugmentDesc(C.Structure):
    """Mirror of `a3d_augment_desc` (include/a3d.h)."""
    _fields_ = [(n, C.c_float) for n in
                ("scale_lo", "scale_hi", "max_rotation_deg", "crop_fraction", "flip_prob", "color_lo", "color_hi",
                 "aspect")]


A3D_U8 = 2
AUG_PARAMS = 16                       # A3D_AUG_PARAMS: floats per image in the packed parameter rows
AUG_VALUE_COLOR, AUG_VALUE_DEPTH = 0, 1

_vp, _i, _f, _sz, _u = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_uint

# name -> (restype, argtypes); every symbol include/a3d.h declares
SIGNATURES = {
    "a3d_version": (_i, []),
    "a3d_last_error": (C.c_char_p, []),
    "a3d_create": (_i, [_i, C.POINTER(_vp)]),
    "a3d_destroy": (_i, [_vp]),
    "a3d_sm_count": (_i, [_vp]),
    "a3d_launch_count": (C.c_uint64, [_vp]),
    "a3d_resize_bilinear_tf1": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp]),
    "a3d_resize_bilinear_tf1_s2d": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp]),
    "a3d_resize_bilinear_tf1_s2d_u8": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp]),
    "a3d_conv2d_pool4_fwd": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _u, _vp, _sz, _vp]),
    "a3d_pool4_bwd": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp, _sz, _vp]),
    "a3d_gather_sum_f32": (_i, [_vp, _vp, _vp, _i, _sz, _vp, _vp]),
    "a3d_scatter_cast_bf16": (_i, [_vp, _vp, _vp, _i, _sz, _vp, _vp]),
    "a3d_conv2d_ws_bytes": (_sz, [_vp, C.POINTER(ConvDesc), _i]),
    "a3d_conv2d_fwd": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _i, _u, _vp, _sz, _vp]),
    "a3d_conv2d_dgrad": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "a3d_conv2d_dgrad_prepare": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp]),
    "a3d_conv2d_dgrad_prepared": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "a3d_conv2d_wgrad": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "a3d_dense_fwd": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _i, _vp, _i, _i, _i, _u, _i, _vp]),
    "a3d_dense_dgrad": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "a3d_stamp": (_i, [_vp, _vp, _vp]),
    "a3d_pairwise_dense_act": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _u, _vp]),
    "a3d_pairwise_dense_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _sz, _u, _vp]),
    "a3d_dcnf_workspace_bytes": (_sz, [_vp, _i, _i, _i, _i, _i, _i]),
    "a3d_dcnf_create": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp, C.POINTER(_vp)]),
    "a3d_dcnf_destroy": (_i, [_vp]),
    "a3d_dcnf_configure": (_i, [_vp, _i]),
    "a3d_dcnf_segment": (_i, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(_sz), C.POINTER(_sz), C.POINTER(_i * 4)]),
    "a3d_dcnf_arena": (_i, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_sz)]),
    "a3d_dcnf_sync_weights": (_i, [_vp, _vp]),
    "a3d_dcnf_global_step": (C.c_longlong, [_vp]),
    "a3d_dcnf_step": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "a3d_dcnf_infer": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "a3d_dcnf_state": (_i, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "a3d_msdn_workspace_bytes": (_sz, [_vp, _i, _i, _i, _i, _i, _i]),
    "a3d_msdn_create": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp, C.POINTER(_vp)]),
    "a3d_msdn_destroy": (_i, [_vp]),
    "a3d_msdn_configure": (_i, [_vp, _f, C.c_uint64]),
    "a3d_msdn_segment": (_i, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(_sz), C.POINTER(_sz), C.POINTER(_i * 4)]),
    "a3d_msdn_arena": (_i, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp),
                            C.POINTER(_sz)]),
    "a3d_msdn_sync_weights": (_i, [_vp, _vp]),
    "a3d_msdn_set_step": (_i, [_vp, C.c_longlong, C.POINTER(_i * 4), _vp]),
    "a3d_msdn_global_step": (C.c_longlong, [_vp]),
    "a3d_msdn_step_begin": (_i, [_vp, _vp]),
    "a3d_msdn_step_enqueue": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "a3d_msdn_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "a3d_msdn_infer": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "a3d_msdn_losses": (_vp, [_vp]),
    "a3d_conv2d_ws_bytes_tf32": (_sz, [_vp, C.POINTER(ConvDesc), _i]),
    "a3d_conv2d_fwd_tf32": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _u, _vp, _sz, _vp]),
    "a3d_conv2d_dgrad_tf32": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "a3d_conv2d_wgrad_tf32": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp]),
    "a3d_dense_fwd_tf32": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _vp, _i, _i, _i, _u, _vp]),
    "a3d_dense_dgrad_tf32": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _f, _u, _vp]),
    "a3d_dense_wgrad_tf32": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp, _i, _i, _i, _vp]),
    "a3d_resize_bilinear_tf1_s2d_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp]),
    "a3d_maxpool2x2_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _vp, _vp]),
    "a3d_maxpool2x2_idx_bwd_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "a3d_act_bwd_f32": (_i, [_vp, _vp, _i, _vp, _vp, _f, _vp, _sz, _i, _u, _vp]),
    "a3d_scatter_channel_f32": (_i, [_vp, _vp, _vp, _sz, _i, _i, _vp]),
    "a3d_pool4_reduce_f32": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _sz, _u, _vp]),
    "a3d_pool4_bwd_f32": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp, _sz, _vp]),
    "a3d_bias_grad_f32": (_i, [_vp, _vp, _sz, _i, _i, _vp, _vp]),
    "a3d_scatter_f32": (_i, [_vp, _vp, _vp, _i, _sz, _vp, _vp]),
    "a3d_split_tf32": (_i, [_vp, _vp, _sz, _i, C.c_longlong, _vp, _vp, _vp]),
    "a3d_conv2d_ws_bytes_tf32x3": (_sz, [_vp, C.POINTER(ConvDesc)]),
    "a3d_conv2d_fwd_tf32x3": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _u, _vp, _sz, _vp]),
    "a3d_dense_ws_bytes_tf32x3": (_sz, [_i, _i, _i]),
    "a3d_dense_fwd_tf32x3": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _vp, _sz, _i, _i, _i, _u, _vp]),
    "a3d_conv_k1_fwd_f32": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _u, _vp]),
    "a3d_conv_k1_dgrad_f32": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp]),
    "a3d_conv_k1_wgrad_f32": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp]),
    "a3d_allgather_multi": (_i, [_vp, _vp, _vp, _i, _i, _vp]),
    "a3d_dense_dgrad_act": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _f, _u, _vp]),
    "a3d_dense_wgrad": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp, _i, _i, _i, _i, _vp]),
    "a3d_dense_wgrad_adam": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _f, _f, _f, _f, _vp, _vp]),
    "a3d_bias_grad_bf16": (_i, [_vp, _vp, _sz, _i, _i, _vp, _i, _sz, _vp]),
    "a3d_dense_epilogue_bwd": (_i, [_vp, _vp, _vp, _vp, _f, _vp, _sz, _u, _vp]),
    "a3d_maxpool2x2_fwd": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _vp]),
    "a3d_maxpool2x2_relu_bwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "a3d_maxpool2x2_fwd_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _vp, _vp]),
    "a3d_maxpool2x2_idx_bwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "a3d_relu_bwd": (_i, [_vp, _vp, _vp, _i, _vp, _sz, _i, _vp]),
    "a3d_silog_loss": (_i, [_vp, _vp, _vp, _i, _i, _f, _vp, _vp, _vp, _vp, _i, _vp]),
    "a3d_adam_tf": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _sz, _f, _f, _f, _f, _f, _vp, _vp]),
    "a3d_adam_tf_bf16g": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _sz, _f, _f, _f, _f, _f, _vp, _vp]),
    "a3d_sgd": (_i, [_vp, _vp, _vp, _vp, _sz, _f, _f, _vp]),
    "a3d_bernoulli_mask": (_i, [_vp, _vp, _sz, _f, C.c_uint64, _vp, _vp]),
    "a3d_increment_i64": (_i, [_vp, _vp, _vp]),
    "a3d_cast_f32_bf16": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "a3d_scatter_channel_bf16": (_i, [_vp, _vp, _vp, _sz, _i, _i, _vp]),
    "a3d_space_to_depth2": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "a3d_fill_zero": (_i, [_vp, _vp, _sz, _vp]),
    "a3d_apply_mask_f32": (_i, [_vp, _vp, _vp, _sz, _vp]),
    "a3d_crf_fwd_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "a3d_pairwise_dense": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "a3d_mean_f32": (_i, [_vp, _vp, _i, _vp, _vp]),
    "a3d_scale_cast_bf16": (_i, [_vp, _vp, _vp, _sz, _f, _vp]),
    "a3d_pairwise_features": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _f, _vp, _vp, _vp]),
    "a3d_pairwise_ws_bytes": (_sz, [_i, _i, _i]),
    "a3d_tile_means": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "a3d_extract_patches": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _vp]),
    "a3d_extract_patches_s2d": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _vp]),
    "a3d_image_cells_s2d": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "a3d_window_gather": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "a3d_window_scatter_sum": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "a3d_depth_metrics": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _i, _f, _f, _i, _vp, _vp, _vp]),
    "a3d_augment_draw": (_i, [_vp, C.POINTER(AugmentDesc), _i, C.c_uint64, _vp, _vp, _vp]),
    "a3d_resize_affine_tf1_s2d": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "a3d_resize_affine_tf1": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _vp, _i, _vp]),
    "a3d_quantize_rows_e4m3": (_i, [_vp, _vp, _i, _i, C.c_longlong, _vp, _vp, _vp]),
    "a3d_quantize_ws_bytes_e4m3": (_sz, [_i, _sz]),
    "a3d_quantize_e4m3": (_i, [_vp, _vp, _i, _sz, _vp, _vp, _vp, _sz, _vp]),
    "a3d_maxpool2x2_quantize_e4m3": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _sz, _vp]),
    "a3d_resize_bilinear_tf1_s2d_e4m3": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp]),
    "a3d_conv2d_fwd_fp8": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _vp, _i, _u, _vp, _sz, _vp]),
    "a3d_conv2d_pool4_fwd_fp8": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _vp, _u, _vp]),
    "a3d_dense_fwd_fp8": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _u, _vp]),
    "a3d_comm_unique_id": (_i, [C.c_char_p, _vp]),
    "a3d_comm_init": (_i, [_vp, C.c_char_p, _vp, _i, _i]),
    "a3d_comm_destroy": (_i, [_vp]),
    "a3d_allreduce_sum": (_i, [_vp, _vp, _sz, _i, _vp]),
    "a3d_reduce_scatter_sum": (_i, [_vp, _vp, _sz, _i, _vp]),
    "a3d_allgather": (_i, [_vp, _vp, _sz, _i, _vp]),
    # engine unit-test hook (not part of the drop-in surface)
    "a3d_debug_tc_gemm": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "a3d_debug_tc_gemm_v": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "a3d_debug_tc_gemm_tf32": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "a3d_debug_tc_gemm_fp8": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp]),
}

_lib = None


def signature_names():
    return list(SIGNATURES)


def load():
    """dlopen liba3d.so and bind every declared symbol.  Raises A3DError if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise A3DError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU or PyTorch fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name, None)
        if fn is None:
            raise A3DError(f"{LIB_PATH} does not export {name}: stale build, run `make -C ann3depth_b200/csrc`")
        fn.restype = res
        fn.argtypes = args
    if lib.a3d_version() != ABI_VERSION:           # e.g. a3d_conv_desc grew two fields in 200: a stale .so misreads it
        raise A3DError(f"{LIB_PATH} is ABI version {lib.a3d_version()}, this host code expects {ABI_VERSION}: rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().a3d_last_error().decode(errors="replace")
        raise A3DError(f"liba3d {what} failed (rc={rc}): {msg}")
