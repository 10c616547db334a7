"""ctypes binding of ``libflowdiff.so`` (the C ABI declared in ``include/flowdiff.h``).

There is no fallback: if the library is missing or the device is not sm_100 every op raises.
PyTorch is used for device memory and streams only; pointers are passed as plain integers.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_long, c_size_t, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libflowdiff.so")

_P, _I, _L, _F = c_void_p, c_int, c_long, c_float

# name -> (restype, argtypes); must list every symbol include/flowdiff.h declares
SIGNATURES = {
    "fd_version": (c_int, []),
    "fd_arch": (c_char_p, []),
    "fd_last_error": (c_char_p, []),
    "fd_device_check": (c_int, []),
    "fd_num_sms": (c_int, []),
    "fd_launch_count": (ctypes.c_ulonglong, []),
    "fd_backwarp_fwd": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "fd_backwarp_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "fd_photo_epe_workspace_floats": (c_size_t, [_I, _I, _I]),
    "fd_warp_div_selftest": (c_int, [_F, _P, _P]),
    "fd_warp_bwd_workspace_floats": (c_size_t, [_I, _I, _I, _I]),
    "fd_backwarp_photo_epe_fwd": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "fd_backwarp_photo_epe_bwd": (c_int, [_P, _P, _P, _P, _P, _F, _F, _P, _P, _P, _I, _I, _I, _I, _P]),
    "fd_splat_fwd": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "fd_splat_ingrad": (c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "fd_splat_flowgrad": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "fd_splat_prepare": (c_int, [_P, _P, _I, _I, _I, _P]),
    "fd_splat_finish": (c_int, [_P, _P, _I, _I, _I, _I, _P]),
    "fd_splat_fwd_workspace_floats": (c_size_t, [_I, _I, _I, _I, _I]),
    "fd_forward_warp_sum3": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "fd_nan_mse_workspace_floats": (c_size_t, [_I, _I, _I]),
    "fd_nan_mse_fwd": (c_int, [_P, _P, _P, _P, _I, _I, _I, _L, _L, _P]),
    "fd_nan_mse_bwd": (c_int, [_P, _P, _P, _F, _P, _I, _I, _I, _L, _L, _L, _P]),
    "fd_q_sample": (c_int, [_P, _P, _P, _P, _P, _P, _I, _L, _P]),
    "fd_ddim_step": (c_int, [_P, _P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _I, _P]),
    "fd_ddpm_step": (c_int, [_P, _P, _P, _P, _P, _L, _F, _F, _F, _P]),
    "fd_dpmpp_step": (c_int, [_P, _P, _P, _P, _P, _P, _L, _F, _F, _F, _F, _I, _P]),
    "fd_pack_input_pad": (c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "fd_pack_input_wide": (c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "fd_prep_weight": (c_int, [_P, _P, _I, _I, _I, _I, _I, _I, _F, _P]),
    "fd_gn_silu": (c_int, [_P, _P, _P, _P, _P, _L, _P, _P, _I, _I, _I, _F, _P]),
    "fd_gn_silu_fast": (c_int, [_P, _P, _P, _P, _P, _L, _P, _P, _I, _I, _I, _F, _P]),
    "fd_chan_layernorm": (c_int, [_P, _P, _P, _P, _L, _I, _F, _P]),
    "fd_upsample2x": (c_int, [_P, _P, _I, _I, _I, _I, _P]),
    "fd_time_embed": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "fd_time_proj": (c_int, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "fd_linattn_workspace_floats": (c_size_t, [_I, _I]),
    "fd_linattn_tc_workspace_floats": (c_size_t, [_I, _I, _I]),
    "fd_linattn_tc_prep": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _P]),
    "fd_linattn_tc": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _P]),
    "fd_linattn": (c_int, [_P, _P, _P, _I, _I, _P]),
    "fd_linattn_context": (c_int, [_P, _I, _P, _P, _I, _I, _P]),
    "fd_attention": (c_int, [_P, _P, _I, _I, _P]),
    "fd_final_conv_crop": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "fd_nchw_to_nhwc_bf16": (c_int, [_P, _P, _I, _I, _I, _P]),
    "fd_nhwc_bf16_to_nchw": (c_int, [_P, _P, _I, _I, _I, _P]),
    "fd_conv_igemm": (c_int, [_P, _I, _P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "fd_conv_igemm_ex": (c_int, [_P, _I, _P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "fd_prep_weight_upconv": (c_int, [_P, _P, _I, _I, _P]),
    "fd_conv_igemm_up": (c_int, [_P, _I, _P, _P, _P, _I, _I, _I, _I, _P]),
    "fd_conv_igemm_rt": (c_int, [_P, _I, _P, _I, _P, _P, _P, _P, _P, _P, _F, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "fd_conv_igemm_rt_head": (c_int, [_P, _I, _P, _I, _P, _P, _P, _P, _P, _P, _F, _P, _P, _I, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "fd_attention_lse": (c_int, [_P, _P, _P, _I, _I, _P]),
    "fd_attention_bwd_workspace_floats": (c_size_t, [_I, _I]),
    "fd_attention_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _P]),
    "fd_linattn_stats": (c_int, [_P, _I, _P, _P, _I, _I, _P]),
    "fd_linattn_bwd_workspace_floats": (c_size_t, [_I, _I]),
    "fd_linattn_bwd": (c_int, [_P, _P, _P, _P, _P, _I, _I, _P]),
    "fd_linattn_stats_floats": (c_size_t, []),
    "fd_linattn_save": (c_int, [_P, _P, _P, _P, _I, _I, _P]),
    "fd_gn_silu_bwd_workspace_floats": (c_size_t, [_I, _I]),
    "fd_gn_silu_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _L, _P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _P]),
    "fd_chan_layernorm_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _L, _I, _F, _P]),
    "fd_upsample2x_bwd": (c_int, [_P, _P, _I, _I, _I, _I, _P]),
    "fd_add_bf16": (c_int, [_P, _P, _P, _L, _P]),
    "fd_bias_grad": (c_int, [_P, _P, _L, _I, _P]),
    "fd_final_conv_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "fd_conv3x3_gnsilu_in": (c_int, [_P, _P, _P, _P, _P, _L, _F, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "fd_prep_weight_dgrad": (c_int, [_P, _P, _I, _I, _I, _P]),
    "fd_prep_weight_batch": (c_int, [_P, _P, _I, _I, _F, _P]),
    "fd_prep_weight_dgrad_batch": (c_int, [_P, _P, _I, _I, _P]),
    "fd_prep_weight_bwd_batch": (c_int, [_P, _P, _I, _I, _F, _P]),
    "fd_prep_weight_bwd": (c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _P]),
    "fd_linear_bwd_w": (c_int, [_P, _L, _P, _L, _P, _P, _I, _I, _I, _I, _P]),
    "fd_linear_bwd_x": (c_int, [_P, _L, _P, _P, _L, _P, _L, _I, _I, _I, _I, _P]),
    "fd_time_embed_save": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "fd_sumsq": (c_int, [_P, _L, _P, _P]),
    "fd_adam_step": (c_int, [_P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _I, _P, _F, _F, _P]),
    "fd_adam_ema_step": (c_int, [_P, _P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _I, _P, _F, _F, _F, _P]),
    "fd_aug_photometric": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _P]),
    "fd_aug_blur3": (c_int, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "fd_aug_geometric": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "fd_loss_workspace_floats": (c_size_t, [_L]),
    "fd_tensor_stats_workspace_floats": (c_size_t, [_L]),
    "fd_tensor_stats": (c_int, [_P, _I, _L, _P, _P, _P]),
    "fd_soft_charb_fwd": (c_int, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "fd_soft_charb_bwd": (c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "fd_edge_smooth_fwd": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "fd_edge_smooth_bwd": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "fd_splat_fwd_multi": (c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "fd_splat_ingrad_multi": (c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "fd_splat_flowgrad_multi": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "fd_soft_charb_multi_workspace_floats": (c_size_t, [_I, _I, _I]),
    "fd_soft_charb_multi_fwd": (c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "fd_soft_charb_multi_bwd": (c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "fd_conv_wgrad": (c_int, [_P, _I, _P, _I, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
}


class FlowDiffError(RuntimeError):
    pass


_lib = None


def load(check_device: bool = False):
    """Load the shared library (once).  Raises FlowDiffError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FlowDiffError(
                f"{LIB_PATH} is missing: build it with `python -m opticalflowdiffusion_b200.build` "
                "(there is no CPU or PyTorch fallback for the flow_diffuser kernels)")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)            # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = res, args
        _lib = lib
    if check_device:
        rc = _lib.fd_device_check()
        if rc != 0:
            raise FlowDiffError(_lib.fd_last_error().decode())
    return _lib


def check(rc: int):
    if rc != 0:
        raise FlowDiffError(f"libflowdiff error {rc}: {load().fd_last_error().decode()}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise FlowDiffError("libflowdiff operates on CUDA tensors only (no CPU fallback)")


class nvtx_range:
    """NVTX range around a region of kernel launches when FD_NVTX=1 (ncu / nsys can then filter by range:
    `ncu --nvtx --nvtx-include "unet.backward/"`); a no-op otherwise."""

    enabled = os.environ.get("FD_NVTX", "0") not in ("", "0")

    def __init__(self, name: str):
        self.name = name

    def __enter__(self):
        if self.enabled:
            torch.cuda.nvtx.range_push(self.name)
        return self

    def __exit__(self, *exc):
        if self.enabled:
            torch.cuda.nvtx.range_pop()
        return False
