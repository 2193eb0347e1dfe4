"""ctypes binding of libmonoflex_b200.so (include/monoflex_b200.h). There is NO fallback: if the shared library is
missing or a call fails, a RuntimeError is raised (the reference's AT_ASSERTM/AT_ERROR also surface as RuntimeError,
/root/reference/model/backbone/DCNv2/src/dcn_v2.h:25-45)."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmonoflex_b200.so")
_lib = None

_P, _I, _F, _LL, _SZ = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_longlong, ctypes.c_size_t

# name -> argtypes (restype int unless stated). Mirrors include/monoflex_b200.h one to one.
SIGNATURES = {
    "mf_version": [],
    "mf_set_conv_impl": [_I],
    "mf_conv_block_n": [_I],
    "mf_pack_conv_weight": [_P, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "mf_pack_conv_weight_dgrad": [_P, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "mf_pack_conv_weights_batched": [_P, _I, _P],
    "mf_conv2d_nhwc_f16": [_P, _I, _I, _I, _I, _I, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _I, _I, _I, _P, _I, _P],
    "mf_pack_conv_weight_split": [_P, _I, _I, _I, _I, _I, _I, _P, _P],
    "mf_conv2d_nhwc_f16x2": [_P, _I, _I, _I, _I, _I, _I, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _I, _I, _I, _I, _P, _I, _I,
                             _I, _I, _P],
    "mf_head_conv_f16x2": [_P, _I, _I, _I, _I, _I, _I, _P, _I, _I, _I, _P, _P, _I, _P, _P, _I, _P, _P, _P, _P, _I, _I, _P, _P],
    "mf_head2_reduce": [_P, _P, _P, _P, _I, _I, _I, _I, _P],
    "mf_dcn_nhwc_f16x2": [_P, _I, _I, _I, _I, _I, _I, _P, _I, _P, _I, _I, _I, _P, _P, _I, _P, _I, _I, _P],
    "mf_conv2d_rows_f16x2": [_P, _I, _I, _I, _I, _I, _I, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _I, _I, _I, _P, _I, _I, _P],
    "mf_pack_image_pair8": [_P, _P, _I, _I, _I, _I, _P],
    "mf_pack_image_split": [_P, _P, _I, _I, _I, _I, _P],
    "mf_maxpool2_split": [_P, _I, _P, _I, _I, _I, _I, _I, _I, _I, _P],
    "mf_upsample_add_split": [_P, _I, _P, _P, _I, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "mf_edge_gather_split": [_P, _I, _I, _I, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "mf_edge_head_add_split": [_P, _I, _I, _P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "mf_split_to_nchw_f32": [_P, _I, _I, _P, _I, _I, _I, _P],
    "mf_conv2d_rows_f16": [_P, _I, _I, _I, _I, _I, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _I, _I, _I, _P, _I, _P],
    "mf_head_fused": [_P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _I, _P, _P],
    "mf_edge_mask": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
    "mf_dcn_nhwc_f16": [_P, _I, _I, _I, _I, _I, _P, _I, _P, _I, _I, _I, _P, _P, _I, _I, _P, _I, _P],
    "mf_pack_image": [_P, _P, _I, _I, _I, _I, _P],
    "mf_nchw_f32_to_nhwc_f16": [_P, _P, _I, _I, _I, _I, _P],
    "mf_nhwc_f16_to_nchw_f32": [_P, _P, _I, _I, _I, _I, _P],
    "mf_pack_offmask": [_P, _P, _P, _I, _I, _P],
    "mf_maxpool2_nhwc_f16": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
    "mf_upsample_add_nhwc_f16": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "mf_edge_gather": [_P, _I, _I, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "mf_edge_head_add": [_P, _P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "mf_sigmoid_clamp": [_P, _LL, _P],
    "mf_focal_loss_forward": [_P, _P, _LL, _P, _P],
    "mf_focal_loss_backward": [_P, _P, _LL, _P, _P, _P],
    "mf_conv2d_wgrad_nhwc_f16": [_P, _I, _I, _I, _I, _I, _P, _I, _I, _I, _I, _I, _P, _P],
    "mf_conv2d_wgrad_rect_nhwc_f16": [_P, _I, _I, _I, _I, _I, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "mf_maxpool2_bwd_nhwc_f16": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P],
    "mf_upsample_bwd_workspace": [_I, _I, _I, _I, _I],
    "mf_upsample_bwd_nhwc_f16": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "mf_sigmoid_clamp_bwd": [_P, _P, _P, _LL, _P],
    "mf_column_sum_workspace": [_LL, _I],
    "mf_column_sum_nhwc_f16": [_P, _I, _LL, _I, _P, _P, _P],
    "mf_edge_gather_bwd": [_P, _P, _I, _I, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P],
    "mf_edge_head_add_bwd": [_P, _P, _I, _P, _P, _P, _I, _I, _P, _P, _P, _I, _I, _I, _I, _P],
    "mf_add_rows_f16": [_P, _I, _P, _I, _LL, _I, _P],
    "mf_interleave2x2_nhwc_f16": [_P, _P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _P],
    "mf_dcn_sample_cols_nhwc_f16": [_P, _I, _P, _I, _P, _I, _I, _I, _I, _P],
    "mf_dcn_col2im_nhwc_f16": [_P, _I, _P, _I, _P, _P, _I, _P, _I, _I, _I, _I, _P],
    "mf_bn_train_workspace": [_LL, _I],
    "mf_bn_train_forward": [_P, _I, _LL, _I, _P, _P, _F, _F, _I, _P, _P, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P, _P],
    "mf_bn_train_backward": [_P, _I, _P, _I, _P, _I, _LL, _I, _P, _P, _P, _I, _P, _I, _P, _I, _P, _P, _P, _P],
    "mf_bn_sync_forward_stats": [_P, _I, _LL, _I, _P, _P, _P],
    "mf_bn_sync_forward_apply": [_P, _I, _LL, _I, _P, ctypes.c_double, _P, _P, _F, _F, _I, _P, _P, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P],
    "mf_bn_sync_backward_stats": [_P, _I, _P, _I, _P, _I, _LL, _I, _P, _P, _I, _P, _P, _P, _P, _P],
    "mf_bn_sync_backward_apply": [_P, _I, _P, _I, _P, _I, _LL, _I, _P, _P, _P, _P, ctypes.c_double, _I, _P, _I, _P, _I, _P, _P],
    "mf_selftest_mn_major": [_P, _P, _P, _P],
    "mf_loss_obj_cols": [],
    "mf_loss_forward": [_P] * 7 + [_I] * 6 + [_P, _P, _P],
    "mf_loss_backward": [_P] * 7 + [_I] * 6 + [_P, _P, _P, _P, _P],
    "mf_adamw_chunk": [],
    "mf_adamw_step_p2p": [_P, _P, _I, _I, ctypes.c_ulonglong, ctypes.c_ulonglong, _P, _P, _P, _LL, _F, _F, _F, _F, _LL, _F, _P],
    "mf_adamw_step_dyn": [_P, _P, _P, _P, _P, _LL, _F, _F, _F, _F, _F, _F, _P, _P, _I, _P],
    "mf_adamw_step": [_P, _P, _P, _P, _P, _LL, _F, _F, _F, _F, _LL, _F, _F, _P],
    "mf_preprocess_images_u8": [_P, _P, _P, _I, _I, _I, _P, _P, _I, _P, _P],
    "mf_draw_heatmaps": [_P, _I, _I, _I, _I, _I, _P, _P],
    "mf_nms_hm": [_P, _P, _I, _I, _I, _P],
    "mf_decode_detections": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                             _P, _P],
    "mf_dcn_v2_forward": [_P, _P, _P, _P, _P, _P] + [_I] * 14 + [_P, _SZ, _P],
    "mf_dcn_v2_backward": [_P] * 11 + [_I] * 14 + [_P, _SZ, _P],
    "mf_dcn_v2_backward_workspace": [_I] * 14,
    "mf_dcn_v2_psroi_pooling_forward": [],
    "mf_dcn_v2_psroi_pooling_backward": [],
}


def load():
    """dlopen the in-tree library (built by __graft_entry__.build()); raises if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("monoflex_b200: %s not built - run `python __graft_entry__.py` (nvcc, sm_100a). "
                               "There is no CPU or PyTorch fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        lib.mf_last_error.restype = ctypes.c_char_p
        lib.mf_last_error.argtypes = []
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = _SZ if name.endswith("_workspace") else _I
        _lib = lib
        if os.environ.get("MF_CONV_IMPL"):            # diagnostics only: 1 = CUDA-core cross-check kernels
            lib.mf_set_conv_impl(int(os.environ["MF_CONV_IMPL"]))
    return _lib


def call(name, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (name, rc, lib.mf_last_error().decode()))
    return rc


def ptr(t):
    """device pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def stream():
    import torch
    return torch.cuda.current_stream().cuda_stream
