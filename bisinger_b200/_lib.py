"""ctypes binding of libbisinger_b200.so (the C-ABI in include/bisinger_b200.h).

The CUDA library is the product; this module only loads it and translates error codes into
``RuntimeError``.  There is deliberately no fallback: if the shared library has not been built
(``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C bisinger_b200/csrc``) the import
of any compute entry point fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BSG_LIB_PATH") or os.path.join(_HERE, "libbisinger_b200.so")   # BSG_LIB_PATH: A/B builds in experiments

BSG_PRECISION_BF16 = 0
BSG_PRECISION_BF16X3 = 1
BSG_PRECISION_FP16X2 = 2
PRECISIONS = {"bf16": BSG_PRECISION_BF16, "bf16x3": BSG_PRECISION_BF16X3, "fp16x2": BSG_PRECISION_FP16X2}
DEFAULT_PRECISION = "fp16x2"   # meets the 1e-2 mel tolerance over 100 steps with 2 MMAs per product (DESIGN.md §5)


class DiffnetConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("in_dims", "hidden_size", "residual_channels", "residual_layers",
                                       "dilation_cycle", "timesteps", "k_step", "precision")]


class Schedule(C.Structure):
    _fields_ = [(n, C.POINTER(C.c_float)) for n in (
        "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod", "sqrt_recip_alphas_cumprod",
        "sqrt_recipm1_alphas_cumprod", "posterior_mean_coef1", "posterior_mean_coef2",
        "posterior_log_variance_clipped")]


class HifiganConfig(C.Structure):
    _fields_ = [
        ("num_mels", C.c_int), ("upsample_initial_channel", C.c_int), ("num_upsamples", C.c_int),
        ("upsample_rates", C.c_int * 8), ("upsample_kernel_sizes", C.c_int * 8),
        ("num_kernels", C.c_int), ("resblock_kernel_sizes", C.c_int * 4),
        ("num_dilations", C.c_int), ("resblock_dilation_sizes", (C.c_int * 4) * 4),
        ("use_pitch_embed", C.c_int), ("audio_sample_rate", C.c_int), ("harmonic_num", C.c_int),
        ("precision", C.c_int),
    ]


class PeConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("n_mel_bins", "hidden_size", "prenet_layers", "conv_layers", "predictor_layers", "kernel_size",
                                       "predictor_kernel", "predictor_hidden", "gn_group_size", "left_padding", "pitch_norm",
                                       "use_uv")] + [("f0_mean", C.c_float), ("f0_std", C.c_float)]


class FftConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("hidden_size", "num_layers", "num_heads", "ffn_kernel", "ffn_act", "use_pos_embed", "out_dims")]


# every symbol include/bisinger_b200.h declares (tests check that the library exports all of them)
EXPORTS = (
    "bsg_abi_version", "bsg_last_error", "bsg_kernel_launch_count",
    "bsg_diffusion_plan_create", "bsg_diffusion_plan_destroy", "bsg_diffusion_sample", "bsg_diffusion_sample_plms", "bsg_diffnet_forward",
    "bsg_diffusion_time_kernel",
    "bsg_diffusion_q_sample", "bsg_diffusion_p_sample", "bsg_diffnet_forward_steps", "bsg_diffusion_plms_update",
    "bsg_hifigan_plan_create", "bsg_hifigan_plan_destroy", "bsg_hifigan_forward", "bsg_hifigan_source",
    "bsg_pe_plan_create", "bsg_pe_plan_destroy", "bsg_pe_forward",
    "bsg_fft_plan_create", "bsg_fft_plan_destroy", "bsg_fft_forward", "bsg_fft_forward_masked",
    "bsg_selftest_conv",
)

_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built. bisinger_b200 has no CPU or "
            "PyTorch fallback -- build it with `make -C bisinger_b200/csrc` (or __graft_entry__.build()).")
    L = C.CDLL(LIB_PATH)
    vp, fp, ip = C.c_void_p, C.c_void_p, C.c_int
    L.bsg_abi_version.restype = C.c_int
    L.bsg_last_error.restype = C.c_char_p
    L.bsg_kernel_launch_count.restype = C.c_ulonglong
    L.bsg_diffusion_plan_create.argtypes = [C.POINTER(DiffnetConfig), C.POINTER(C.c_float), C.c_size_t, C.POINTER(Schedule),
                                            C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.POINTER(vp)]
    L.bsg_diffusion_plan_destroy.argtypes = [vp]
    L.bsg_diffusion_plan_destroy.restype = None
    L.bsg_diffusion_sample.argtypes = [vp, fp, fp, fp, fp, C.c_ulonglong, fp, ip, ip, fp, fp, vp]
    L.bsg_diffusion_sample_plms.argtypes = [vp, fp, fp, fp, C.c_ulonglong, fp, C.POINTER(C.c_float), ip, ip, ip, fp, fp, vp]
    L.bsg_diffnet_forward.argtypes = [vp, fp, ip, fp, ip, ip, fp, vp]
    L.bsg_diffusion_time_kernel.argtypes = [vp, ip, ip, ip, ip, C.POINTER(C.c_float), vp]
    tp, ull = C.POINTER(C.c_int), C.c_ulonglong
    L.bsg_diffusion_q_sample.argtypes = [vp, fp, tp, fp, ull, ip, ip, fp, vp]
    L.bsg_diffusion_p_sample.argtypes = [vp, fp, tp, fp, ull, fp, ull, ip, ip, ip, fp, vp]
    L.bsg_diffnet_forward_steps.argtypes = [vp, fp, tp, fp, ull, ip, ip, fp, vp]
    L.bsg_diffusion_plms_update.argtypes = [vp, fp, tp, C.POINTER(C.c_float), ip, ip, fp, fp, fp, fp, ip, ip, fp, vp]
    L.bsg_hifigan_plan_create.argtypes = [C.POINTER(HifiganConfig), C.POINTER(C.c_float), C.c_size_t, C.c_int, C.POINTER(vp)]
    L.bsg_hifigan_plan_destroy.argtypes = [vp]
    L.bsg_hifigan_plan_destroy.restype = None
    L.bsg_hifigan_forward.argtypes = [vp, fp, fp, fp, fp, C.c_ulonglong, ip, ip, fp, vp]
    L.bsg_hifigan_source.argtypes = [vp, fp, fp, fp, C.c_ulonglong, ip, ip, fp, vp]
    L.bsg_pe_plan_create.argtypes = [C.POINTER(PeConfig), C.POINTER(C.c_float), C.c_size_t, C.c_int, C.POINTER(vp)]
    L.bsg_pe_plan_destroy.argtypes = [vp]
    L.bsg_pe_plan_destroy.restype = None
    L.bsg_pe_forward.argtypes = [vp, fp, ip, ip, fp, fp, vp]
    L.bsg_fft_plan_create.argtypes = [C.POINTER(FftConfig), C.POINTER(C.c_float), C.c_size_t, C.c_int, C.POINTER(vp)]
    L.bsg_fft_plan_destroy.argtypes = [vp]
    L.bsg_fft_plan_destroy.restype = None
    L.bsg_fft_forward.argtypes = [vp, fp, fp, ip, ip, fp, fp, vp]
    L.bsg_fft_forward_masked.argtypes = [vp, fp, vp, fp, ip, ip, fp, fp, vp]
    L.bsg_selftest_conv.argtypes = [fp, C.POINTER(C.c_float), C.POINTER(C.c_float), ip, ip, ip, ip, ip, C.POINTER(C.c_int),
                                    ip, ip, fp, vp]
    if L.bsg_abi_version() != 1:
        raise RuntimeError("libbisinger_b200.so ABI version mismatch")
    _lib = L
    return L


def check(status: int) -> None:
    if status != 0:
        raise RuntimeError("bisinger_b200: " + lib().bsg_last_error().decode("utf-8", "replace"))


def resolve_seed(seed) -> int:
    """``seed=None`` (the default of every entry point): a fresh 62-bit Philox key drawn from torch's global CPU generator, so that
    repeated calls get fresh noise as in the reference (which draws from the global RNG: shallow_diffusion_tts.py:163, source.py:54,133)
    while ``torch.manual_seed(s)`` still makes a run reproducible.  An explicit integer is used as is."""
    if seed is None:
        import torch
        return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())
    return int(seed) & (2 ** 64 - 1)


def launch_count() -> int:
    return int(lib().bsg_kernel_launch_count())


def fptr(t):
    """float* view of a contiguous float32 torch tensor living on the host (plan-creation inputs)."""
    assert t.dtype.is_floating_point and t.is_contiguous() and t.device.type == "cpu"
    return C.cast(t.data_ptr(), C.POINTER(C.c_float))


def dev_ptr(t, dtype=None):
    """Device pointer of a contiguous CUDA tensor (or None)."""
    if t is None:
        return None
    import torch
    if not t.is_cuda:
        raise RuntimeError("bisinger_b200: tensor must live on a CUDA device (no CPU path exists)")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"bisinger_b200: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise RuntimeError("bisinger_b200: tensor must be contiguous")
    return C.c_void_p(t.data_ptr())


def current_stream_ptr(device):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
