"""ctypes binding of ``liblfb200.so`` (C ABI declared in ``include/lfb200.h``).

There is deliberately no fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'liblfb200.so')

c_f32p = ctypes.c_void_p     # device pointers are passed as raw addresses
c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_float = ctypes.c_float
c_vp = ctypes.c_void_p

CAM_STRIDE = 40
CAMGRAD_STRIDE = 20


class ConvDesc(ctypes.Structure):
    """lf_conv_desc (include/lfb200.h)."""
    _fields_ = [('ndim', c_int), ('n', c_int), ('d', c_int), ('h', c_int), ('w', c_int),
                ('cin', c_int), ('cout', c_int), ('k', c_int), ('scale', c_float), ('act', c_int),
                ('slope', c_float), ('norm', c_int), ('precision', c_int)]


class LossDesc(ctypes.Structure):
    """lf_loss_desc (include/lfb200.h)."""
    _fields_ = [('n', c_int), ('p', c_int), ('width', c_int), ('height', c_int),
                ('z_span', c_float), ('eps', c_float),
                ('pix_stride', c_int), ('hyp_stride', c_int), ('tz_stride', c_int)]


_SIGNATURES = {
    'lf_version': (ctypes.c_char_p, []),
    'lf_last_error': (ctypes.c_char_p, []),
    'lf_sm_count': (c_int, []),
    'lf_resample_o2c_fwd': (c_int, [c_f32p, c_f32p, c_f32p, c_int, c_int, c_int, c_int, c_vp]),
    'lf_resample_o2c_fwd_split_supported': (c_int, [c_int, c_int]),
    'lf_resample_o2c_fwd_split': (c_int, [c_f32p, c_f32p, c_vp, c_int, c_int, c_int, c_int, c_vp]),
    'lf_resample_o2c_bwd_cam_ws': (c_i64, [c_int, c_int]),
    'lf_resample_o2c_bwd_cam': (c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_int, c_int, c_int, c_int, c_vp]),
    'lf_resample_o2c_bwd_cam_block': (c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_int, c_int, c_int, c_int, c_vp]),
    'lf_resample_o2c_bwd_vol': (c_int, [c_f32p, c_f32p, c_f32p, c_int, c_int, c_int, c_int, c_vp]),
    'lf_resample_c2o_fwd': (c_int, [c_f32p, c_f32p, c_f32p, c_int, c_int, c_int, c_vp]),
    'lf_resample_c2o_bwd_vol': (c_int, [c_f32p, c_f32p, c_f32p, c_int, c_int, c_int, c_vp]),
    'lf_conv_fwd': (c_int, [ctypes.POINTER(ConvDesc), c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_vp]),
    'lf_conv3d_dz_supported': (c_int, [ctypes.POINTER(ConvDesc)]),
    'lf_split_bytes': (c_i64, [c_int] * 5),
    'lf_split_pack': (c_int, [c_f32p, c_vp] + [c_int] * 5 + [c_vp]),
    'lf_conv3d_dz_weight_bytes': (c_i64, [c_int, c_int]),
    'lf_conv3d_dz_pack_weights': (c_int, [c_f32p, c_vp, c_int, c_int, c_vp]),
    'lf_conv3d_dz': (c_int, [ctypes.POINTER(ConvDesc), c_vp, c_vp, c_f32p, c_f32p, c_vp, c_f32p, c_vp]),
    'lf_conv3d_dz_bwd_epi': (c_int, [ctypes.POINTER(ConvDesc), c_vp, c_vp, c_vp, c_f32p, c_int, c_float, c_int, c_f32p, c_vp, c_vp]),
    'lf_actnorm_bwd_split': (c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_vp] + [c_int] * 6 + [c_float, c_int, c_vp]),
    'lf_ibr_blend_bwd': (c_int, [c_f32p, c_f32p, c_f32p, c_int, c_int, c_int, c_int, c_vp]),
    'lf_ibr_warp_blend_bwd': (c_int, [c_f32p, c_f32p, c_float, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_int, c_int, c_int, c_int, c_int, c_vp]),
    'lf_gru_gates1_bwd': (c_int, [c_f32p] * 8 + [c_i64, c_vp]),
    'lf_gru_gates2_bwd': (c_int, [c_f32p] * 7 + [c_i64, c_vp]),
    'lf_lstm_gates_fwd': (c_int, [c_f32p] * 4 + [c_i64, c_int, c_vp]),
    'lf_lstm_gates_bwd': (c_int, [c_f32p] * 6 + [c_i64, c_int, c_vp]),
    'lf_softmax_blend_fwd': (c_int, [c_f32p] * 4 + [c_int, c_int, c_i64, c_int, c_vp]),
    'lf_softmax_blend_bwd': (c_int, [c_f32p] * 6 + [c_int, c_int, c_i64, c_int, c_vp]),
    'lf_depth_sum_fwd': (c_int, [c_f32p, c_f32p, c_int, c_int, c_i64, c_int, c_vp]),
    'lf_conv3d_ws_supported': (c_int, [ctypes.POINTER(ConvDesc)]),
    'lf_conv3d_ws_weight_bytes': (c_i64, [c_int, c_int, c_int]),
    'lf_conv3d_ws_pack_weights': (c_int, [c_f32p, c_vp, c_int, c_int, c_int, c_vp]),
    'lf_conv3d_ws_scratch': (c_i64, [ctypes.POINTER(ConvDesc)]),
    'lf_conv3d_ws': (c_int, [ctypes.POINTER(ConvDesc), c_vp, c_vp, c_f32p, c_f32p, c_f32p, c_f32p, c_vp]),
    'lf_expand_tc_supported': (c_int, [ctypes.POINTER(ConvDesc)]),
    'lf_expand_tc_weight_bytes': (c_i64, [c_int, c_int, c_int]),
    'lf_expand_tc_pack_weights': (c_int, [c_f32p, c_vp, c_int, c_int, c_int, c_vp]),
    'lf_expand_tc_bwd_epi': (c_int, [ctypes.POINTER(ConvDesc), c_vp, c_vp, c_vp, c_f32p, c_int, c_float, c_int, c_vp, c_f32p, c_vp]),
    'lf_collapse_tc_supported': (c_int, [ctypes.POINTER(ConvDesc)]),
    'lf_collapse_tc_weight_bytes': (c_i64, [c_int, c_int, c_int]),
    'lf_collapse_tc_pack_weights': (c_int, [c_f32p, c_vp, c_int, c_int, c_int, c_vp]),
    'lf_collapse_tc': (c_int, [ctypes.POINTER(ConvDesc), c_vp, c_vp, c_f32p, c_f32p, c_f32p, c_vp]),
    'lf_set_option': (c_int, [ctypes.c_char_p, c_int]),
    'lf_conv3d_dw_supported': (c_int, [ctypes.POINTER(ConvDesc)]),
    'lf_conv3d_dw_ws': (c_i64, [ctypes.POINTER(ConvDesc)]),
    'lf_conv3d_dw': (c_int, [ctypes.POINTER(ConvDesc), c_vp, c_vp, c_f32p, c_f32p, c_f32p, c_vp]),
    'lf_conv3d_dz_timeline': (c_int, [ctypes.POINTER(ConvDesc), c_vp, c_vp, c_f32p, c_f32p, c_vp, c_f32p, c_vp, c_vp]),
    'lf_conv_tc_weight_bytes': (c_i64, [c_int, c_int, c_int]),
    'lf_conv_tc_pack_weights': (c_int, [c_f32p, c_vp, c_int, c_int, c_int, c_vp]),
    'lf_conv_tc_supported': (c_int, [ctypes.POINTER(ConvDesc)]),
    'lf_conv_tc_passes': (c_int, [ctypes.POINTER(ConvDesc)]),
    'lf_conv_bwd_data_fused': (c_int, [ctypes.POINTER(ConvDesc), c_f32p, c_f32p, c_f32p, c_int, c_float, c_int, c_f32p, c_f32p, c_vp]),
    'lf_actnorm_bwd': (c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_i64, c_int, c_i64, c_int, c_int, c_float, c_int, c_vp]),
    'lf_conv_bwd_weight': (c_int, [ctypes.POINTER(ConvDesc), c_f32p, c_f32p, c_f32p, c_f32p, c_vp]),
    'lf_interp_fwd': (c_int, [c_f32p, c_f32p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_vp]),
    'lf_interp_bwd': (c_int, [c_f32p, c_f32p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_vp]),
    'lf_fuse_pool_fwd': (c_int, [c_f32p, c_f32p, c_int, c_int, c_i64, c_int, c_int, c_vp]),
    'lf_fuse_pool_bwd': (c_int, [c_f32p, c_f32p, c_f32p, c_int, c_int, c_i64, c_int, c_int, c_vp]),
    'lf_gru_gates1': (c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_i64, c_vp]),
    'lf_gru_gates2': (c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_i64, c_vp]),
    'lf_camera_o2c_fwd': (c_int, [c_f32p] * 5 + [c_int, c_float, c_float, c_vp]),
    'lf_camera_o2c_bwd': (c_int, [c_f32p] * 6 + [c_int, c_vp]),
    'lf_adam_step': (c_int, [c_f32p] * 4 + [c_int, c_int, c_f32p, c_f32p, c_float, c_float, c_float, c_vp]),
    'lf_refine_record': (c_int, [c_f32p, c_int, c_int] + [c_f32p] * 11 + [c_vp, c_int, c_f32p, c_vp]),
    'lf_plateau_step': (c_int, [c_f32p] * 4 + [c_int, c_float, c_float, c_float, c_vp]),
    'lf_pose_loss_fwd': (c_int, [ctypes.POINTER(LossDesc)] + [c_f32p] * 8 + [c_vp, c_vp]),
    'lf_pose_loss_search_fwd': (c_int, [ctypes.POINTER(LossDesc)] + [c_f32p] * 8 + [c_vp, c_vp]),
    'lf_pose_loss_bwd': (c_int, [ctypes.POINTER(LossDesc)] + [c_f32p] * 12 + [c_vp, c_vp]),
    'lf_pose_loss_fwd_ws': (c_i64, [ctypes.POINTER(LossDesc)]),
    'lf_pose_loss_bwd_ws': (c_i64, [ctypes.POINTER(LossDesc)]),
    'lf_conv_bwd_data_epi_supported': (c_int, [ctypes.POINTER(ConvDesc)]),
    'lf_conv_bwd_data_epi': (c_int, [ctypes.POINTER(ConvDesc), c_f32p, c_f32p, c_f32p, c_f32p, c_int, ctypes.c_float, c_int, c_f32p, c_vp]),
    'lf_heads_fwd': (c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_i64, c_int, c_int, ctypes.c_float, c_vp]),
    'lf_heads_bwd': (c_int, [c_f32p, c_f32p, c_f32p, c_i64, c_int, c_int, ctypes.c_float, c_vp]),
    'lf_ibr_reproject_fwd': (c_int, [c_f32p] * 7 + [c_int] * 5 + [c_vp]),
    'lf_ibr_blend_fwd': (c_int, [c_f32p] * 3 + [c_int] * 5 + [c_vp]),
    'lf_ibr_warp_blend_fwd': (c_int, [c_f32p, c_f32p, ctypes.c_float] + [c_f32p] * 4 + [c_int] * 5 + [c_vp]),
}

_lib = None


def symbols():
    """Names of every entry point the binding expects (== what include/lfb200.h declares)."""
    return sorted(_SIGNATURES)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"latentfusion_b200: native library {LIB_PATH} is missing. Build it with "
                f"`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc, sm_100a). "
                f"There is no CPU/PyTorch fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)      # AttributeError if the .so does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status, what):
    if status == 0:
        return
    msg = lib().lf_last_error().decode('utf-8', 'replace')
    if status < 0:
        raise ValueError(f"{what}: {msg}")
    raise RuntimeError(f"{what}: CUDA error {status}: {msg}")
