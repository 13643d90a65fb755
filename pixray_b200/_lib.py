"""ctypes binding of the C-ABI library (include/pixray_b200.h).

The CUDA extension is the product: if the shared library is missing this module raises -- there is no CPU or
PyTorch fallback anywhere in the package.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libpixray_b200.so")


class ClipCfg(C.Structure):
    _fields_ = [("width", C.c_int), ("layers", C.c_int), ("heads", C.c_int), ("patch", C.c_int),
                ("image_res", C.c_int), ("out_dim", C.c_int)]


class Config(C.Structure):
    _fields_ = [
        ("device", C.c_int), ("rank", C.c_int), ("world", C.c_int), ("drawer", C.c_int),
        ("image_h", C.c_int), ("image_w", C.c_int),
        ("z_channels", C.c_int), ("n_embed", C.c_int), ("ch", C.c_int), ("num_res_blocks", C.c_int),
        ("attn_resolution", C.c_int), ("n_levels", C.c_int), ("resolution", C.c_int),
        ("ch_mult", C.c_int * 8),
        ("grid_rows", C.c_int), ("grid_cols", C.c_int),
        ("cutn", C.c_int), ("cut_size", C.c_int),
        ("n_clip", C.c_int), ("clip", ClipCfg * 2),
        ("noise_fac", C.c_float), ("seed", C.c_uint64),
        ("op_dtype", C.c_int), ("grad_scale", C.c_float),
        ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float),
        ("fft_decay", C.c_float), ("fft_colors", C.c_float), ("fft_contrast", C.c_float),
        ("cut_aspect", C.c_float), ("cut_src_h", C.c_int), ("cut_src_w", C.c_int), ("reserved", C.c_int * 2),
    ]


class CutParams(C.Structure):
    _fields_ = [("transforms", C.c_void_p), ("zoom_padding", C.c_int), ("fill", C.c_float),
                ("noise_facs", C.c_void_p), ("noise", C.c_void_p), ("color_jitter", C.c_void_p)]


class Status(C.Structure):
    _fields_ = [("iter", C.c_int), ("loss_sum", C.c_float), ("best_loss", C.c_float), ("best_iter", C.c_int),
                ("num_loss_drop", C.c_int), ("stopped", C.c_int), ("rebuilt", C.c_int), ("lr", C.c_float),
                ("n_losses", C.c_int), ("losses", C.c_float * 64)]


class TestGemmDesc(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("a_mode", C.c_int),
        ("lda", C.c_longlong), ("a_mn_extent", C.c_longlong), ("a_k_extent", C.c_longlong),
        ("a_bs0", C.c_longlong), ("a_bs1", C.c_longlong),
        ("b", C.c_void_p), ("b_mode", C.c_int), ("b_batched", C.c_int),
        ("ldb", C.c_longlong), ("b_mn_extent", C.c_longlong), ("b_k_extent", C.c_longlong),
        ("b_bs0", C.c_longlong), ("b_bs1", C.c_longlong),
        ("nb0", C.c_int), ("nb1", C.c_int),
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int), ("block_n", C.c_int), ("fmt", C.c_int),
        ("alpha", C.c_float), ("bias", C.c_void_p), ("bias_per_row", C.c_int), ("act", C.c_int),
        ("aux_in", C.c_void_p), ("aux_out", C.c_void_p), ("res_f32", C.c_void_p), ("res_f16", C.c_void_p),
        ("out_f32", C.c_void_p), ("out_f16", C.c_void_p),
        ("ldc", C.c_longlong), ("c_bs0", C.c_longlong), ("c_bs1", C.c_longlong),
        ("stream", C.c_void_p), ("repeat", C.c_int), ("n_store", C.c_int), ("cta_group", C.c_int), ("tma_epi", C.c_int),
    ]


# every symbol include/pixray_b200.h declares (tests check the library exports all of them)
EXPORTS = [
    "pxr_last_error", "pxr_version", "pxr_create", "pxr_destroy", "pxr_load_weight", "pxr_finalize",
    "pxr_set_prompts", "pxr_set_comm", "pxr_get_unique_id", "pxr_synth", "pxr_vqgan_encode", "pxr_make_cutouts", "pxr_encode_image",
    "pxr_prompt_loss", "pxr_backward", "pxr_step", "pxr_iterate", "pxr_reset_optimizer", "pxr_set_optimizer", "pxr_sync",
    "pxr_num_kernel_launches", "pxr_get_stream", "pxr_z_numel", "pxr_z_bounds", "pxr_test_gemm", "pxr_test_conv", "pxr_debug_read", "pxr_profile_iteration", "pxr_profile_iteration2",
    "pxr_test_attention", "pxr_test_color_jitter_host", "pxr_test_color_jitter_device", "pxr_set_color_jitter", "pxr_set_image_prompts", "pxr_set_image_prompts_sized", "pxr_add_aux_loss", "pxr_add_filter", "pxr_clear_filters", "pxr_set_filter_shifts", "pxr_clear_aux_losses", "pxr_add_anchor", "pxr_clear_anchors", "pxr_num_losses", "pxr_read_losses",
    "pxr_test_pool_bounds", "pxr_test_groupnorm", "pxr_set_spot_prompts", "pxr_set_spot_mask", "pxr_state_size", "pxr_save_state", "pxr_load_state", "pxr_set_schedule", "pxr_poll_status", "pxr_set_batches", "pxr_set_z_grad", "pxr_vdiff_set_schedule", "pxr_vdiff_set_clip_embed", "pxr_vdiff_set_iteration", "pxr_vdiff_renoise",
]

_lib = None


def load():
    """Load libpixray_b200.so (built in-tree by `make` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension is the product and there is no fallback. "
            "Run `make` (or __graft_entry__.build()) first.")
    lib = C.CDLL(LIB_PATH)
    for name in EXPORTS:
        try:
            fn = getattr(lib, name)
        except AttributeError:
            continue  # tests/test_abi.py reports missing exports; individual callers fail loudly
        if name in ("pxr_last_error", "pxr_version"):
            fn.restype = C.c_char_p
        elif name == "pxr_destroy":
            fn.restype = None
        else:
            fn.restype = C.c_int
    if hasattr(lib, "pxr_last_error"):
        lib.pxr_last_error.argtypes = [C.c_void_p]
    if hasattr(lib, "pxr_set_optimizer"):
        lib.pxr_set_optimizer.argtypes = [C.c_void_p, C.c_int]
    _lib = lib
    return lib
