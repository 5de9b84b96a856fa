"""ctypes binding of libipr_b200.so (the C ABI declared in include/ipr_b200.h).

The library is the product: there is no PyTorch/CPU fallback.  Loading it without the built
``.so`` raises, and every op in ``ops.py`` refuses non-CUDA tensors.
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IPR_B200_LIB") or os.path.join(_PKG, "libipr_b200.so")   # override: A/B runs of two builds

c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_f32 = ctypes.c_float
c_ptr = ctypes.c_void_p
c_size = ctypes.c_size_t

SIGN_MAX_LAYERS = 64


class SnLayer(ctypes.Structure):
    """ipr_sn_layer_t"""
    _fields_ = [("w", c_ptr), ("u", c_ptr), ("v", c_ptr), ("sigma", c_ptr), ("grad", c_ptr), ("grad_out", c_ptr),
                ("rows", ctypes.c_int32), ("cols", ctypes.c_int32), ("scratch_off", ctypes.c_int64),
                ("u_snap", c_ptr), ("v_snap", c_ptr)]


class SignLayer(ctypes.Structure):
    """ipr_sign_layer_t"""
    _fields_ = [("gamma", c_ptr), ("sign", c_ptr), ("grad", c_ptr), ("n", ctypes.c_int32),
                ("reserved", ctypes.c_int32)]


# name -> (restype, argtypes); mirrors include/ipr_b200.h one to one (tests/test_abi.py checks it).
SIGNATURES = {
    "ipr_version": (c_int, []),
    "ipr_strerror": (ctypes.c_char_p, [c_int]),
    "ipr_launch_count": (ctypes.c_uint64, []),
    "ipr_paste_patch_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "ipr_trigger_pair_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_int, c_int, c_int,
                                     c_ptr, c_ptr, c_i64, c_ptr]),
    "ipr_crop_patch_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "ipr_crop_postproc_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "ipr_crop_clamp01_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "ipr_bitmask_scatter_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_f32, c_ptr]),
    "ipr_transform_dist_f32": (c_int, [c_ptr, c_ptr, c_i64, c_ptr]),
    "ipr_transform_var_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_ptr]),
    "ipr_ssim_workspace_bytes": (c_size, [c_i64, c_int, c_int, c_int]),
    "ipr_ssim_fwd_bwd_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_size, c_i64, c_int, c_int, c_int,
                                     c_int, c_f32, c_f32, c_ptr]),
    "ipr_ssim_per_sample_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_size, c_i64, c_int, c_int, c_int, c_ptr]),
    "ipr_sign_loss_fwd_bwd_f32": (c_int, [ctypes.POINTER(SignLayer), c_int, c_f32, c_f32, c_int, c_f32, c_ptr, c_ptr]),
    "ipr_sign_ber_i32": (c_int, [ctypes.POINTER(SignLayer), c_int, c_ptr, c_ptr]),
    "ipr_bicubic_resize_f32": (c_int, [c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_int, c_ptr]),
    "ipr_pdq_dct_matrix_host": (None, [c_ptr]),
    "ipr_pdq_hash_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_ptr]),
    "ipr_hash_pvalue": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_ptr]),
    "ipr_tapgemm_m_tiles": (c_int, [c_ptr]),
    "ipr_tapgemm_stats_rows": (c_int, [c_ptr]),
    "ipr_tapgemm_bf16": (c_int, [c_ptr, c_ptr]),
    "ipr_wgrad_workspace_bytes": (c_size, [c_ptr]),
    "ipr_wgrad_total_kblocks": (c_int, [c_ptr]),
    "ipr_wgrad_bf16": (c_int, [c_ptr, c_ptr]),
    "ipr_im2col3_bf16": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_ptr]),
    "ipr_col2im3_f32": (c_int, [c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_int, c_ptr]),
    "ipr_tapfold3_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_ptr]),
    "ipr_tapfold3_band_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_ptr]),
    "ipr_bn_finalize_f32": (c_int, [c_ptr, c_int, c_int, ctypes.c_double, c_f32, c_f32, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "ipr_bn_apply_relu_bf16": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_int, c_ptr]),
    "ipr_bn_bwd_workspace_bytes": (c_size, [c_int]),
    "ipr_bn_relu_bwd_bf16": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_ptr, c_f32, c_f32, c_ptr, c_size, c_i64, c_int, c_ptr]),
    "ipr_dfc_fwd_bf16": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_ptr]),
    "ipr_dfc_bwd_bf16": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_f32, c_int, c_int, c_ptr, c_ptr, c_ptr]),
    "ipr_colsum_workspace_bytes": (c_size, [c_int]),
    "ipr_colsum_partials_f32": (c_int, [c_ptr, c_int, c_int, c_int, c_ptr, c_int, c_f32, c_ptr, c_size, c_ptr]),
    "ipr_colsum_bf16": (c_int, [c_ptr, c_i64, c_int, c_ptr, c_int, c_f32, c_ptr, c_ptr, c_size, c_ptr]),
    "ipr_sn_scratch_floats": (c_size, [c_int, c_int]),
    "ipr_sn_power_iter_f32": (c_int, [c_ptr, c_int, c_int, c_f32, c_ptr, c_ptr]),
    "ipr_sn_weight_grad_f32": (c_int, [c_ptr, c_int, c_ptr, c_ptr]),
    "ipr_adam_flat_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_f32, c_f32, c_f32, c_f32, c_f32, c_f32, c_int,
                                  c_ptr, c_ptr, c_ptr]),
    "ipr_gather_pack_bf16": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_i64, c_ptr]),
    "ipr_hinge_d_loss_f32": (c_int, [c_ptr, c_ptr, c_int, c_f32, c_ptr, c_ptr, c_ptr, c_ptr]),
    "ipr_gen_adv_loss_f32": (c_int, [c_ptr, c_int, c_f32, c_ptr, c_ptr, c_ptr]),
    "ipr_im2col_nhwc_bf16": (c_int, [c_ptr, c_ptr] + [c_int] * 12 + [c_ptr]),
    "ipr_col2im_nhwc_bf16": (c_int, [c_ptr, c_ptr, c_ptr] + [c_int] * 12 + [c_ptr]),
    "ipr_nchw_to_nhwc_bf16": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_int, c_ptr]),
    "ipr_finish_nchw_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "ipr_pixel_shuffle2_nhwc_bf16": (c_int, [c_ptr, c_ptr, c_i64, c_int, c_int, c_int, c_int, c_ptr]),
    "ipr_add_bf16": (c_int, [c_ptr, c_ptr, c_ptr, c_i64, c_ptr]),
    "ipr_norm_workspace_bytes": (c_size, [c_int, c_int]),
    "ipr_norm_fwd_bf16": (c_int, [c_ptr, c_ptr, c_ptr, c_int, c_i64, c_int, c_int, c_f32, c_f32, c_ptr, c_ptr, c_ptr, c_ptr,
                                  c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_f32, c_ptr, c_ptr, c_size, c_ptr]),
    "ipr_norm_bwd_bf16": (c_int, [c_ptr, c_ptr, c_ptr, c_int, c_i64, c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                  c_ptr, c_int, c_ptr, c_f32, c_f32, c_int, c_f32, c_ptr, c_ptr, c_ptr, c_size, c_ptr]),
    "ipr_pointwise_loss_workspace_bytes": (c_size, []),
    "ipr_pointwise_loss_f32": (c_int, [c_ptr, c_ptr, c_f32, c_i64, c_int, c_f32, c_ptr, c_ptr, c_ptr, c_size, c_ptr]),
    "ipr_randn_f32": (c_int, [c_ptr, c_i64, ctypes.c_uint64, c_ptr, c_ptr, c_ptr]),
    "ipr_wgrad_tiles": (c_int, [c_ptr]),
    "ipr_wgrad_reduce_f32": (c_int, [c_ptr, c_int, c_int, c_int, c_int, c_ptr, c_ptr, c_i64, c_ptr, c_int, c_f32, c_ptr]),
    "ipr_wgrad_reduce_taps_f32": (c_int, [c_ptr, c_int, c_int, c_int, c_int, c_int, c_ptr, c_int, c_i64, c_i64, c_ptr, c_int,
                                          ctypes.c_float, c_ptr]),
    "ipr_prune_workspace_bytes": (c_size, [c_i64]),
    "ipr_prune_magnitude_f32": (c_int, [c_ptr, c_ptr, c_int, c_i64, c_i64, c_ptr, c_size, c_ptr]),
    "ipr_negate_indexed_f32": (c_int, [c_ptr, c_ptr, c_i64, c_ptr]),
}

_lib = None


def lib():
    """Load (once) and return the C-ABI library.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libipr_b200.so is not built (%s). Run `python -m ipr_gan_b200.build` -- "
                "there is no CPU fallback for the IPR-GAN hot path." % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)          # AttributeError here = header/library drift
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


class IprError(RuntimeError):
    pass


def check(code, what):
    if code != 0:
        msg = lib().ipr_strerror(code)
        raise IprError("%s failed: %s (code %d)" % (what, msg.decode() if msg else "?", code))


def launch_count():
    return int(lib().ipr_launch_count())
