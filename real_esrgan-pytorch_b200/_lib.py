"""ctypes binding of libresr.so (C ABI declared in include/resr.h). torch is used only for device memory and streams."""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RESR_LIB_PATH") or os.path.join(_HERE, "lib", "libresr.so")  # override: A/B builds in development


class ResrError(RuntimeError):
    pass


class ConvDesc(Structure):
    """struct resr_conv_desc (include/resr.h)."""
    _fields_ = [
        ("in16", c_void_p),
        ("n", c_int), ("h", c_int), ("w", c_int), ("c_total", c_int), ("cin", c_int), ("cout", c_int),
        ("fmt_in", c_int), ("mode", c_int),
        ("weight", c_void_p), ("bias", c_void_p),
        ("ep_mode", c_int), ("lrelu", c_int), ("clamp01", c_int),
        ("out16", c_void_p),
        ("out16_fmt", c_int), ("out16_cstride", c_int), ("out16_choff", c_int), ("out16_up2", c_int),
        ("outf", c_void_p),
        ("outf_cstride", c_int), ("outf_choff", c_int),
        ("res1", c_void_p), ("res2", c_void_p),
        ("res_cstride", c_int), ("res_choff", c_int),
        ("res16", c_int), ("res16_fmt", c_int),
        ("out_nchw", c_void_p),
        ("out_nchw_c", c_int),
        ("reverse", c_int),
        ("vmask", c_void_p), ("vmask_words", c_int), ("vmask_shift", c_int),
        ("out_u8", c_void_p),
        ("out_nchw_raw", c_void_p),
        ("mask16", c_void_p), ("mask16_cstride", c_int), ("mask16_choff", c_int),
        ("out16_scale", c_float),
        ("res2_scale", c_float),
        ("res2_cstride", c_int),
        ("slice_nores_mask", ctypes.c_uint), ("slice_noutf_mask", ctypes.c_uint), ("slice_no16_mask", ctypes.c_uint),
        ("out16_slice_fixed", c_int),
    ]


class ConvPlan(Structure):
    """struct resr_conv_plan (include/resr.h)."""
    _fields_ = [("pair", c_int), ("nout", c_int), ("nslices", c_int), ("bw", c_int), ("bn", c_int), ("mode", c_int),
                ("nxs", c_int), ("ncg", c_int), ("tail_ksteps", c_int), ("nepi", c_int), ("epi_bufs", c_int),
                ("nstages", c_int), ("masked", c_int), ("units", ctypes.c_longlong), ("clusters", ctypes.c_longlong)]


class ResizeSpec(Structure):
    """struct resr_resize_spec (include/resr.h)."""
    _fields_ = [("mode", c_int), ("out_h", c_int), ("out_w", c_int), ("scale", c_double)]


class NoiseSpec(Structure):
    """struct resr_noise_spec (include/resr.h)."""
    _fields_ = [("type", c_int), ("param", c_void_p), ("gray", c_void_p), ("gray_any", c_int), ("draws_color", c_void_p),
                ("draws_gray", c_void_p), ("seed", ctypes.c_ulonglong)]


class DegradePlan(Structure):
    """struct resr_degrade_plan (include/resr.h)."""
    _fields_ = [("batch", c_int), ("hr_h", c_int), ("hr_w", c_int),
                ("usm_radius", c_int), ("usm_sigma", c_int), ("usm_weight", c_float), ("usm_threshold", c_float),
                ("blur1", c_int), ("blur2", c_int), ("final_order", c_int), ("kernel_size", c_int), ("sinc_batched", c_int),
                ("resize1", ResizeSpec), ("resize2", ResizeSpec), ("resize3", ResizeSpec),
                ("noise1", NoiseSpec), ("noise2", NoiseSpec),
                ("jpeg1_quality", c_void_p), ("jpeg2_quality", c_void_p),
                ("crop_top", c_int), ("crop_left", c_int), ("image_size", c_int), ("upscale", c_int),
                ("rng_state", c_void_p)]


class KernelParams(Structure):
    """struct resr_kernel_params (include/resr.h)."""
    _fields_ = [("type", c_int), ("kernel_size", c_int), ("isotropic", c_int), ("reserved", c_int),
                ("sigma_x", c_double), ("sigma_y", c_double), ("theta", c_double), ("beta", c_double),
                ("cutoff", c_double)]


class KernelDrawConfig(Structure):
    """struct resr_kernel_draw_config (include/resr.h)."""
    _fields_ = [("n_sizes", c_int), ("sizes", c_int * 16), ("sinc_size_split", c_int), ("final_size", c_int),
                ("sinc_prob1", c_double), ("sinc_prob2", c_double), ("sinc_prob3", c_double),
                ("prob1", c_double * 6), ("prob2", c_double * 6),
                ("sigma_range1", c_double * 2), ("sigma_range2", c_double * 2),
                ("gen_beta_range1", c_double * 2), ("gen_beta_range2", c_double * 2),
                ("plateau_beta_range1", c_double * 2), ("plateau_beta_range2", c_double * 2)]


# name -> (restype, argtypes); every symbol include/resr.h declares must be listed here (tests check both ways).
SIGNATURES = {
    "resr_version": (c_int, []),
    "resr_last_error": (c_char_p, []),
    "resr_generator_create": (c_int, [POINTER(c_void_p), c_int, c_int, c_int]),
    "resr_generator_destroy": (None, [c_void_p]),
    "resr_generator_num_params": (c_size_t, []),
    "resr_generator_num_tensors": (c_int, []),
    "resr_generator_tensor_span": (c_int, [c_int, POINTER(c_size_t), POINTER(c_size_t)]),
    "resr_generator_load_params": (c_int, [c_void_p, c_void_p, c_void_p]),
    "resr_generator_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "resr_generator_workspace_bytes_for": (c_size_t, [c_void_p, c_int, c_int, c_int]),
    "resr_generator_set_precision": (c_int, [c_void_p, c_int]),
    "resr_generator_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "resr_generator_forward_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "resr_generator_forward_u8_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "resr_tensor_to_image_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "resr_generator_forward_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "resr_generator_forward_host_async": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "resr_generator_host_sync": (c_int, [c_void_p]),
    "resr_canvas_pack": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "resr_generator_forward_many_workspace_bytes": (c_size_t, [c_void_p, c_void_p, c_void_p, c_int]),
    "resr_generator_forward_many": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "resr_generator_forward_many_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t,
                                               c_void_p]),
    "resr_generator_launches_per_forward": (c_int, []),
    "resr_set_conv_pair_policy": (c_int, [c_int]),
    "resr_conv3x3": (c_int, [POINTER(ConvDesc), c_void_p]),
    "resr_conv3x3_plan": (c_int, [POINTER(ConvDesc), c_int, POINTER(ConvPlan)]),
    "resr_nchw_to_nhwc16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "resr_filter2d": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "resr_usm_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "resr_niqe_num_blocks": (c_int, [c_int, c_int, c_int, c_int]),
    "resr_niqe_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "resr_niqe_features": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "resr_niqe_many_workspace_bytes": (c_size_t, [c_void_p, c_void_p, c_int, c_int, c_int]),
    "resr_niqe_features_many": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                                        c_void_p]),
    "resr_augment_batch_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "resr_usm_backward_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "resr_usm_sharp_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_float,
                                        c_void_p, c_size_t, c_void_p]),
    "resr_usm_sharp": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_void_p,
                               c_size_t, c_void_p]),
    "resr_resize": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_double, c_double, c_void_p]),
    "resr_gaussian_noise_apply": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                          c_int, c_int, c_int, c_void_p]),
    "resr_poisson_workspace_bytes": (c_size_t, [c_int]),
    "resr_unique_count_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "resr_poisson_rates": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "resr_poisson_noise_apply": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                         c_int, c_int, c_int, c_void_p, c_size_t, c_int, c_void_p]),
    "resr_gaussian_noise_sampled": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                            ctypes.c_ulonglong, c_void_p, c_void_p]),
    "resr_poisson_noise_sampled": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                           ctypes.c_ulonglong, c_void_p, c_void_p, c_size_t, c_void_p]),
    "resr_jpeg": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                          c_void_p]),
    "resr_degrade_workspace_bytes": (c_size_t, [POINTER(DegradePlan)]),
    "resr_degrade_batch": (c_int, [POINTER(DegradePlan), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_size_t, c_void_p]),
    "resr_adam_ema_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_float,
                                   c_float, ctypes.c_longlong, c_float, c_float, c_void_p]),
    "resr_synthesize_kernels": (c_int, [POINTER(KernelParams), c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "resr_synthesize_kernels_device": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "resr_draw_degradation_kernel_params": (c_int, [POINTER(KernelDrawConfig), c_int, ctypes.c_ulonglong, c_void_p, c_void_p, c_void_p]),
    "resr_generator_train_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "resr_generator_forward_train": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "resr_generator_backward_l1": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t,
                                           c_void_p]),
    "resr_generator_train_step_l1": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                             c_void_p, c_size_t, c_void_p]),
    "resr_generator_step_is_graph": (c_int, [c_void_p]),
    "resr_generator_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "resr_conv3x3_wgrad_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "resr_generator_grad_buckets": (c_int, [c_void_p, c_int]),
    "resr_generator_wait_grad_bucket": (c_int, [c_void_p, c_int, c_void_p]),
    "resr_conv3x3_wgrad_nhwc_workspace_bytes": (c_size_t, []),
    "resr_conv3x3_wgrad_nhwc": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                        c_void_p, c_size_t, c_void_p]),
    "resr_conv3x3_wgrad": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                   c_void_p, c_size_t, c_void_p]),
    "resr_crop": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
}

_lib = None


def lib():
    """Loads libresr.so on first use. Fails loudly: there is no other implementation to fall back to."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ResrError(
                f"{LIB_PATH} is missing: build it with `make` (or `python -c 'import __graft_entry__ as g; g.build()'`). "
                "resr_b200 has no CPU / PyTorch fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().resr_last_error()
        raise ResrError(f"libresr error {rc}: {msg.decode() if msg else '?'}")


def stream_ptr(device=None):
    """Current CUDA stream of `device` (default: the current device) as the `void* stream` of the C ABI."""
    import torch
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def canvas_pack(sizes, max_width=0):
    """resr_canvas_pack: `sizes` is a sequence of (h, w) LR sizes. Returns ([(x0, y0)] in input order, (canvas_h, canvas_w))."""
    n = len(sizes)
    hs = (c_int * n)(*[int(h) for h, _ in sizes])
    ws = (c_int * n)(*[int(w) for _, w in sizes])
    x0, y0, ch, cw = (c_int * n)(), (c_int * n)(), c_int(), c_int()
    check(lib().resr_canvas_pack(hs, ws, n, int(max_width), x0, y0, ctypes.byref(ch), ctypes.byref(cw)))
    return list(zip(x0, y0)), (ch.value, cw.value)


def ptr(t):
    """Device (or host) pointer of a torch tensor as c_void_p; None -> NULL."""
    if t is None:
        return c_void_p(0)
    return c_void_p(t.data_ptr())
