"""ctypes binding of libnfe_b200.so (C ABI declared in include/nfe_b200.h).

The library is loaded on first use.  There is no fallback of any kind: if the shared object has not
been built (python -m nerffaceediting_b200.build) the first kernel call raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libnfe_b200.so")

DEC_OSG, DEC_DISENTANGLED, DEC_SEGMENTATION = 0, 1, 2
PREC_FP32, PREC_BF16X3, PREC_BF16 = 0, 1, 2

c_f32p = ctypes.c_void_p   # device pointers travel as integers
c_i64 = ctypes.c_int64
c_u64 = ctypes.c_uint64
c_int = ctypes.c_int
c_float = ctypes.c_float
c_double = ctypes.c_double
c_vp = ctypes.c_void_p


class NfeMlp(ctypes.Structure):
    _fields_ = [("w1", c_vp), ("b1", c_vp), ("w2", c_vp), ("b2", c_vp),
                ("in_dim", c_int), ("hidden", c_int), ("out_dim", c_int),
                ("wgain1", c_float), ("bgain1", c_float), ("wgain2", c_float), ("bgain2", c_float)]


class NfeRenderCfg(ctypes.Structure):
    _fields_ = [("kind", c_int), ("channels", c_int), ("height", c_int), ("width", c_int),
                ("s_c", c_int), ("s_f", c_int), ("color_dim", c_int), ("seg_dim", c_int),
                ("white_back", c_int), ("box_warp", c_float), ("density_noise", c_float),
                ("stochastic", c_int), ("seed", c_u64), ("offset", c_u64), ("precision", c_int),
                ("affine_scale", c_vp), ("affine_shift", c_vp), ("affine_items", c_int), ("sigma_only", c_int), ("image_layout", c_int),
                ("geometry_only", c_int)]


class NfeModconvArgs(ctypes.Structure):
    _fields_ = [("x", c_vp), ("weight", c_vp), ("styles", c_vp), ("noise", c_vp), ("noise_batch_stride", c_i64), ("bias", c_vp), ("y", c_vp),
                ("filter", c_vp), ("fh", c_int), ("fw", c_int), ("batch", c_int), ("in_ch", c_int), ("out_ch", c_int), ("in_h", c_int),
                ("in_w", c_int), ("ksize", c_int), ("up", c_int), ("demodulate", c_int), ("flip_weight", c_int), ("act", c_int),
                ("alpha", c_float), ("gain", c_float), ("clamp", c_float), ("dtype", c_int), ("weight_batch_stride", c_i64)]


_MLP_P = ctypes.POINTER(NfeMlp)
_CFG_P = ctypes.POINTER(NfeRenderCfg)

# name -> (restype, argtypes); must list every symbol include/nfe_b200.h declares
SIGNATURES = {
    "nfe_version": (c_int, []),
    "nfe_last_error": (ctypes.c_char_p, []),
    "nfe_launch_count": (c_u64, []),
    "nfe_timing_enable": (c_int, [c_int]),
    "nfe_timing_read": (c_int, [ctypes.POINTER(c_double), ctypes.POINTER(c_i64), c_int, c_int]),
    "nfe_bench_l2_gather": (c_int, [c_vp, c_i64, c_int, c_int, c_int, ctypes.POINTER(c_i64), c_vp, c_vp]),
    "nfe_plane_stats": (c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "nfe_plane_normalize": (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp]),
    "nfe_plane_denormalize": (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp]),
    "nfe_plane_normalize_staged": (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "nfe_planes_to_channel_last": (c_int, [c_vp, c_i64, c_int, c_i64, c_vp, c_vp]),
    "nfe_generate_rays": (c_int, [c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp]),
    "nfe_ray_limits_box": (c_int, [c_vp, c_vp, c_i64, c_float, c_vp, c_vp, c_vp]),
    "nfe_sample_stratified": (c_int, [c_i64, c_int, c_int, c_vp, c_double, c_double, c_vp, c_vp, c_vp, c_int, c_u64, c_u64, c_vp, c_vp]),
    "nfe_sample_planes_fwd": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_i64, c_float, c_vp, c_vp]),
    "nfe_decoder_fwd": (c_int, [c_int, c_int, _MLP_P, _MLP_P, c_vp, c_vp, c_int, c_i64, c_int, c_vp, c_vp, c_vp, c_vp]),
    "nfe_composite_fwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "nfe_importance_resample": (c_int, [c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_int, c_u64, c_u64, c_vp, c_vp, c_vp, c_vp]),
    "nfe_sample_pdf": (c_int, [c_vp, c_vp, c_i64, c_int, c_int, c_int, c_vp, c_int, c_u64, c_u64, c_float, c_vp, c_vp]),
    "nfe_unify_samples":(c_int, [c_vp] * 8 + [c_i64, c_int, c_int, c_int, c_int] + [c_vp] * 4 + [c_vp]),
    "nfe_render_workspace_bytes": (c_i64, [_CFG_P, c_int, c_i64]),
    "nfe_render_fwd": (c_int, [_CFG_P, _MLP_P, _MLP_P, c_vp, c_vp, c_int, c_vp, c_vp, c_int, c_i64, c_vp, c_vp,
                               c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "nfe_render_workspace_layout": (c_int, [_CFG_P, c_int, c_i64, ctypes.POINTER(c_i64)]),
    "nfe_composite_bwd": (c_int, [c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "nfe_feature_mean_fwd": (c_int, [c_vp, c_int, c_int, c_int, c_float, c_vp, c_vp, c_vp, c_int, c_i64, c_int, c_vp, c_vp]),
    "nfe_feature_mean_bwd": (c_int, [c_vp, c_int, c_int, c_int, c_float, c_vp, c_vp, c_vp, c_int, c_i64, c_int, c_vp, c_vp]),
    "nfe_planes_from_channel_last": (c_int, [c_vp, c_i64, c_int, c_i64, c_vp, c_vp]),
    "nfe_field_bwd": (c_int, [c_int, c_vp, c_vp, c_int, c_int, c_int, c_float, c_vp, c_vp, c_vp, c_int, c_i64, c_int, _MLP_P, _MLP_P, c_vp, c_vp,
                              c_vp, c_vp] + [c_vp] * 8 + [c_vp, c_vp, c_int, c_vp, c_vp] + [c_vp]),
    "nfe_run_model_bwd": (c_int, [c_int, c_vp, c_vp, c_int, c_int, c_int, c_float, c_vp, c_int, c_i64, _MLP_P, _MLP_P, c_vp, c_vp,
                                  c_vp, c_vp] + [c_vp] * 8 + [c_vp, c_vp, c_int, c_vp, c_vp] + [c_vp]),
    "nfe_remap_seg": (c_int, [c_vp, c_i64, c_vp, c_vp]),
    "nfe_seg_cross_entropy_fwd": (c_int, [c_vp, c_vp, c_int, c_int, c_i64, c_vp, c_vp, c_vp]),
    "nfe_seg_cross_entropy_bwd": (c_int, [c_vp, c_vp, c_int, c_int, c_i64, c_vp, c_vp, c_vp]),
    "nfe_hist_dist_fwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_i64, c_float, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "nfe_hist_dist_bwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_i64, c_float, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "nfe_plane_normalize_bwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "nfe_resize_bilinear": (c_int, [c_vp, c_i64, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "nfe_finish_depth": (c_int, [c_vp, c_i64, c_vp, c_vp]),
    "nfe_run_model_fwd": (c_int, [_CFG_P, _MLP_P, _MLP_P, c_vp, c_vp, c_int, c_vp, c_int, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "nfe_bias_act": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_i64, c_int, c_int, c_int, c_float, c_float, c_float, c_vp]),
    "nfe_layout_convert": (c_int, [c_vp, c_vp, c_i64, c_int, c_i64, c_int, c_int, c_vp]),
    "nfe_image_accumulate": (c_int, [c_vp, c_vp, c_i64, c_int, c_i64, c_int, c_vp]),
    "nfe_modconv_workspace_bytes": (c_i64, [ctypes.POINTER(NfeModconvArgs)]),
    "nfe_modulated_conv2d": (c_int, [ctypes.POINTER(NfeModconvArgs), c_vp, c_i64, c_vp]),
    "nfe_upfirdn2d": (c_int, [c_vp, c_vp, c_vp] + [c_int] * 8 + [ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)] + [c_int] * 9 + [c_float, c_int, c_vp]),
}

_lib = None


def load():
    """Load (once) and return the ctypes library with every prototype set."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"nerffaceediting_b200: CUDA library not built ({LIB_PATH} missing). "
                "Run `python -m nerffaceediting_b200.build`; there is no CPU or PyTorch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)   # AttributeError if the .so is stale
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc, what):
    """Mirror TORCH_CHECK: a non-zero return becomes a RuntimeError carrying nfe_last_error()."""
    if rc != 0:
        msg = load().nfe_last_error()
        raise RuntimeError(f"{what}: {msg.decode() if msg else 'error %d' % rc}")


def launch_count():
    return int(load().nfe_launch_count())


STAGES = ("field_coarse", "resample", "field_fine", "march_final", "run_model")


def timing_enable(on=True):
    check(load().nfe_timing_enable(int(bool(on))), "nfe_timing_enable")


def timing_read(reset=True):
    """{stage: (total_ms, launches)} of the stages recorded since the last reset (waits for them)."""
    ms = (c_double * len(STAGES))()
    cnt = (c_i64 * len(STAGES))()
    check(load().nfe_timing_read(ms, cnt, len(STAGES), int(bool(reset))), "nfe_timing_read")
    return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(STAGES)}
