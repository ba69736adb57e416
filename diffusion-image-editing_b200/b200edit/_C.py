"""ctypes binding of include/b200edit.h (the C ABI of libb200edit.so)."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libb200edit.so")


class B2EError(RuntimeError):
    pass


class StepCoeffs(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("sqrt_a_t", "sqrt_b_t", "sqrt_a_prev", "dir_coef", "sigma",
                                         "a_t_sq", "variance", "a_t", "a_prev")]


class GuidedStepParams(C.Structure):
    _fields_ = [("c", StepCoeffs), ("clip", C.c_int32), ("clip_range", C.c_float),
                ("has_noise", C.c_int32), ("noise_batched", C.c_int32), ("guide", C.c_int32),
                ("has_target", C.c_int32 * 4), ("target", C.c_float * 4), ("coef", C.c_float * 4),
                ("mask_grad", C.c_int32), ("mask_batched", C.c_int32), ("no_step", C.c_int32)]


class L2RegParams(C.Structure):
    _fields_ = [("base", GuidedStepParams), ("lambda_", C.c_float), ("loss_scale", C.c_float)]


class ColorGradParams(C.Structure):
    _fields_ = [("has_target", C.c_int32 * 4), ("target", C.c_float * 4), ("k", C.c_float * 4), ("lam_scale", C.c_float),
                ("use_mask_pred", C.c_int32), ("mask_batched", C.c_int32)]


class UNetConfig(C.Structure):
    _fields_ = [("sample_size", C.c_int32), ("in_channels", C.c_int32), ("out_channels", C.c_int32),
                ("n_blocks", C.c_int32), ("block_out_channels", C.c_int32 * 8),
                ("down_attn", C.c_int32 * 8), ("up_attn", C.c_int32 * 8),
                ("layers_per_block", C.c_int32), ("norm_num_groups", C.c_int32),
                ("norm_eps", C.c_float), ("attention_head_dim", C.c_int32),
                ("flip_sin_to_cos", C.c_int32), ("freq_shift", C.c_float), ("downsample_padding", C.c_int32),
                ("cross_attention_dim", C.c_int32), ("num_attention_heads", C.c_int32), ("precision", C.c_int32)]


class VQDecConfig(C.Structure):
    _fields_ = [("sample_size", C.c_int32), ("latent_channels", C.c_int32), ("out_channels", C.c_int32),
                ("n_blocks", C.c_int32), ("block_out_channels", C.c_int32 * 8), ("layers_per_block", C.c_int32),
                ("norm_num_groups", C.c_int32), ("norm_eps", C.c_float), ("num_vq_embeddings", C.c_int32),
                ("precision", C.c_int32)]


class VQEncConfig(C.Structure):
    _fields_ = [("sample_size", C.c_int32), ("in_channels", C.c_int32), ("latent_channels", C.c_int32),
                ("n_blocks", C.c_int32), ("block_out_channels", C.c_int32 * 8), ("layers_per_block", C.c_int32),
                ("norm_num_groups", C.c_int32), ("norm_eps", C.c_float), ("double_z", C.c_int32), ("precision", C.c_int32)]


class ClipConfig(C.Structure):
    _fields_ = [("vocab_size", C.c_int32), ("hidden_size", C.c_int32), ("intermediate_size", C.c_int32),
                ("num_layers", C.c_int32), ("num_heads", C.c_int32), ("max_positions", C.c_int32), ("precision", C.c_int32)]


class ResNetConfig(C.Structure):
    _fields_ = [("input_size", C.c_int32), ("in_channels", C.c_int32), ("bottleneck", C.c_int32),
                ("layers", C.c_int32 * 4), ("width", C.c_int32), ("num_classes", C.c_int32), ("head", C.c_int32),
                ("precision", C.c_int32), ("grad_precision", C.c_int32)]


class LpipsConfig(C.Structure):
    _fields_ = [("input_size", C.c_int32), ("precision", C.c_int32), ("grad_precision", C.c_int32)]


_P, _I64, _I, _F, _SZ = C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_size_t

# name -> (restype, argtypes); every symbol include/b200edit.h declares
PROTOTYPES = {
    "b2e_version": (_I, []),
    "b2e_last_error": (C.c_char_p, []),
    "b2e_device_check": (_I, []),
    "b2e_launch_count": (_I64, []),
    "b2e_step_coeffs_compute": (_I, [_P, _I, _F, _I, _I, _F, _I, C.POINTER(StepCoeffs)]),
    "b2e_guided_step_f32": (_I, [_P, _P, _P, _P, _P, _P, _I64, _I64, _I64, C.POINTER(GuidedStepParams), _P]),
    "b2e_l2reg_workspace_bytes": (_SZ, [_I64, _I64, _I64]),
    "b2e_guided_step_l2reg_f32": (_I, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64,
                                       C.POINTER(L2RegParams), _P, _SZ, _P]),
    "b2e_apply_guidance_grad_f32": (_I, [_P, _P, _P, _I64, _I64, _I, _F, _P]),
    "b2e_color_loss_grad_workspace_bytes": (_SZ, []),
    "b2e_color_loss_grad_f32": (_I, [_P, _P, _P, _P, _I64, _I64, _I64, C.POINTER(ColorGradParams), _P, _SZ, _P]),
    "b2e_lpips_guidance_grad_f32": (_I, [_P, _P, _P, _P, _I64, _I64, _I64, C.POINTER(ColorGradParams), _P]),
    "b2e_apply_latent_guidance_f32": (_I, [_P, _P, _P, _I64, _I64, _I, _F, _F, _F, _P]),
    "b2e_pred_x0_f32": (_I, [_P, _P, _P, _I64, _F, _F, _P]),
    "b2e_renoise_f32": (_I, [_P, _P, _P, _I64, _F, _F, _F, _F, _P]),
    "b2e_cfg_combine_f32": (_I, [_P, _P, _P, _I64, _F, _P]),
    "b2e_apply_mask_f32": (_I, [_P, _P, _P, _P, _I64, _I64, _P]),
    "b2e_to_uint8_f32": (_I, [_P, _P, _I64, _I64, _I64, _P]),
    "b2e_axpby_f32": (_I, [_P, _P, _P, _I64, _F, _F, _P]),
    "b2e_loss_workspace_bytes": (_SZ, []),
    "b2e_l2_distance_f32": (_I, [_P, _P, _I64, _P, _P, _SZ, _P]),
    "b2e_channel_l1_f32": (_I, [_P, _I64, _I64, _I64, _P, _P, _P, _SZ, _P]),
    "b2e_seg_area_head_workspace_bytes": (_SZ, []),
    "b2e_seg_area_head_f32": (_I, [_P, _I64, _I64, C.POINTER(C.c_int32), _I, _F, _P, _P, _P, _SZ, _P]),
    "b2e_classifier_head_f32": (_I, [_P, _I64, _I, _I, _I, _I, _F, _P, _P, _P]),
    "b2e_seg_area_head_batched_workspace_bytes": (_SZ, [_I64]),
    "b2e_seg_area_head_batched_f32": (_I, [_P, _I64, _I64, _I64, C.POINTER(C.c_int32), _I, _F, _F, _P, _P, _P, _SZ, _P]),
    "b2e_classifier_head_batched_f32": (_I, [_P, _I64, _I, _I, _I, _I, _F, _F, _P, _P, _P]),
    "b2e_sample_xts_f32": (_I, [_P, _P, _P, _P, _P, _I64, _I64, _P]),
    "b2e_extract_noise_f32": (_I, [_P, _P, _P, _P, _I64, C.POINTER(StepCoeffs), _P]),
    "b2e_mask_workspace_bytes": (_SZ, [_I64, _I64, _I64, _I64]),
    "b2e_mask_from_seg": (_I, [_P, _I64, _I64, C.POINTER(C.c_int32), _I, _I, _I, _I64, _I64, _I, _I,
                               _P, _P, _SZ, _P]),
    "b2e_mask_batched_workspace_bytes": (_SZ, [_I64, _I64, _I64, _I64, _I64]),
    "b2e_mask_from_seg_batched": (_I, [_P, _I64, _I64, _I64, C.POINTER(C.c_int32), _I, _I, _I, _I64, _I64, _I, _I,
                                       _P, _P, _SZ, _P]),
    "b2e_resize_bilinear_aa_f32": (_I, [_P, _I64, _I64, _P, _I64, _I64, _P, _SZ, _P]),
    "b2e_morphology2d_f32": (_I, [_P, _P, _P, _I64, _I64, _I64, _I64, _I64, _I, _I, _I, _F, _P]),
    "b2e_unet_create": (_I, [C.POINTER(UNetConfig), _I64, C.POINTER(_P)]),
    "b2e_vqdec_create": (_I, [C.POINTER(VQDecConfig), _I64, C.POINTER(_P)]),
    "b2e_vqenc_create": (_I, [C.POINTER(VQEncConfig), _I64, C.POINTER(_P)]),
    "b2e_clip_create": (_I, [C.POINTER(ClipConfig), _I64, C.POINTER(_P)]),
    "b2e_clip_forward": (_I, [_P, _P, _I64, _P, _I64, _P]),
    "b2e_resnet_create": (_I, [C.POINTER(ResNetConfig), _I64, C.POINTER(_P)]),
    "b2e_resnet_backward": (_I, [_P, _P, _P, _I64, _P]),
    "b2e_resnet_forward_labels": (_I, [_P, _P, _P, _I64, _P]),
    "b2e_lpips_create": (_I, [C.POINTER(LpipsConfig), _I64, C.POINTER(_P)]),
    "b2e_lpips_set_reference": (_I, [_P, _P, _I64, _P]),
    "b2e_lpips_forward": (_I, [_P, _P, _P, _I64, _P, _I64, _P]),
    "b2e_lpips_backward": (_I, [_P, _P, _P, _I64, _P]),
    "b2e_unet_enable_grad": (_I, [_P, _I]),
    "b2e_vqdec_backward": (_I, [_P, _P, _P, _I64, _P]),
    "b2e_unet_destroy": (None, [_P]),
    "b2e_unet_num_params": (_I, [_P]),
    "b2e_unet_param_info": (_I, [_P, _I, C.POINTER(C.c_char_p), C.POINTER(_I64), C.POINTER(_I64)]),
    "b2e_unet_set_param": (_I, [_P, C.c_char_p, _P, _I64, _P]),
    "b2e_unet_workspace_bytes": (_SZ, [_P]),
    "b2e_unet_bind_workspace": (_I, [_P, _P, _SZ]),
    "b2e_unet_forward": (_I, [_P, _P, _P, _P, _I64, _P]),
    "b2e_unet_forward_cond": (_I, [_P, _P, _P, _P, _I64, _P, _I64, _P]),
    "b2e_unet_flops": (C.c_double, [_P, _I64]),
    "b2e_unet_launches_per_forward": (_I, [_P]),
    "b2e_unet_op_desc": (C.c_char_p, [_P, _I]),
    "b2e_unet_profile": (_I, [_P, _P, _P, _P, _I64, _P, _I, C.POINTER(_I), C.POINTER(C.c_float),
                              C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(_I)]),
    "b2e_act_dtype": (_I, []),
    "b2e_conv2d_nhwc_f16": (_I, [_P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, _I64, _I, _I, _P]),
    "b2e_conv2d_bench_f16": (_I, [_I64, _I64, _I64, _I64, _I64, _I, _I, _I, _I, _P, _P]),
    "b2e_bilinear_ac_argmax_f16": (_I, [_P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _I, _P]),
    "b2e_upsample_conv3x3_nhwc_f16": (_I, [_P, _P, _P, _P, _I64, _I64, _I64, _I64, _I64, _P]),
    "b2e_attention_f16": (_I, [_P, _I64, _I64, _P, _I64, _I64, _I64, _P, _I64, _I64, _I64, _I64, _I64, _I64, _I64, _I64,
                               _I, _I, _I, _P]),
    "b2e_attention_bwd_fp32": (_I, [_P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, _P]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise B2EError(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build` "
            "(there is no CPU / PyTorch fallback for this path)")
    lib_ = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib_, name)  # AttributeError if the library does not export the symbol
        fn.restype = res
        fn.argtypes = args
    return lib_


lib = _load()


def check(rc: int, what: str = ""):
    if rc != 0:
        raise B2EError(f"{what or 'libb200edit'} failed ({rc}): {lib.b2e_last_error().decode()}")


def launch_count() -> int:
    return int(lib.b2e_launch_count())


_device_ok = False


def require_device():
    """Fail loudly unless the current CUDA device is a B200 (sm_100)."""
    global _device_ok
    if not _device_ok:
        import torch
        if not torch.cuda.is_available():
            raise B2EError("no CUDA device: the b200edit operators have no CPU fallback")
        check(lib.b2e_device_check(), "b2e_device_check")
        _device_ok = True


def fast_precision() -> str:
    """Name of the engine's 16-bit operand type: "fp16" (default build) or "bf16" (-DB2E_ACT_BF16 build)."""
    return "bf16" if lib.b2e_act_dtype() == 1 else "fp16"


def resolve_precision(precision, who: str):
    """-> (name, b2e config value).  None / "fp16" (the build's 16-bit type: fp16 operands, fp32 accumulation) or
    "fp32" (fp32-accurate mode: split hi + lo 16-bit operands, three products per GEMM).  Asking for the 16-bit type the
    library was NOT built for raises instead of silently computing in another precision."""
    fast = fast_precision()
    if precision is None:
        precision = fast
    if precision == "fp32":
        return "fp32", 1
    if precision in ("fp16", "bf16"):
        if precision != fast:
            raise ValueError(f"{who}: libb200edit.so is built for {fast} operands; precision={precision!r} is not available "
                             f"(use precision=None / {fast!r} / 'fp32')")
        return fast, 0
    raise ValueError(f"{who}: precision must be '{fast}' or 'fp32' (got {precision!r})")


def resolve_grad_precision(grad_precision, precision, who: str) -> int:
    """-> b2e config value of a loss network's ``grad_precision``.  None: 0, the 16-bit backward; "fp32": 1, the
    fp32-accurate backward (split hi + lo gradients and dgrad weights), which needs the fp32-accurate forward
    (``precision`` "fp32", as resolve_precision names it).  Anything else raises ValueError."""
    if grad_precision is None:
        return 0
    if grad_precision != "fp32":
        raise ValueError(f"{who}: grad_precision must be None or 'fp32' (got {grad_precision!r})")
    if precision != "fp32":
        raise ValueError(f"{who}: grad_precision='fp32' needs precision='fp32' (got precision={precision!r})")
    return 1
