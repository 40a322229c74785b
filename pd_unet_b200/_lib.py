"""ctypes binding of libpdu_b200.so (include/pdu.h).  There is no CPU or PyTorch fallback: if the
library is missing, or a call fails, the operators raise."""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpdu_b200.so")

PDU_GEOM_PARALLEL, PDU_GEOM_FAN = 0, 1
WRAP_MODES = {"flip": 0, "periodic": 1, "clamp": 2}
LAYOUT_NCHW, LAYOUT_NHWC = 0, 1
NUFFT_IMAGE_SPLIT, NUFFT_KDATA_SPLIT = 1, 2
PDU_EINVAL, PDU_EUNSUPPORTED = -1, -4


class PduError(RuntimeError):
    """A libpdu_b200 entry point returned a negative PDU_E* code."""


class RadonGeomC(C.Structure):
    """pdu_radon_geom_t"""
    _fields_ = [("geom", C.c_int32), ("n", C.c_int32), ("n_angles", C.c_int32), ("det_count", C.c_int32),
                ("det_spacing", C.c_float), ("s_dist", C.c_float), ("d_dist", C.c_float),
                ("clip_to_circle", C.c_int32)]


_p = C.c_void_p
_G = C.POINTER(RadonGeomC)

# name -> (restype, argtypes); every symbol include/pdu.h declares
SIGNATURES = {
    "pdu_last_error": (C.c_char_p, []),
    "pdu_version": (C.c_int, []),
    "pdu_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "pdu_set_option": (C.c_int, [C.c_char_p, C.c_int]),
    "pdu_get_option": (C.c_int, [C.c_char_p, C.POINTER(C.c_int)]),
    "pdu_launch_count": (C.c_long, [C.c_int]),
    "pdu_device_error": (C.c_int, [C.c_int]),
    "pdu_last_kernel": (C.c_char_p, [C.c_char_p]),
    "pdu_radon_trig_f32": (C.c_int, [_p, _p, C.c_int, _p]),
    "pdu_radon_workspace_bytes": (C.c_size_t, [_G, C.c_int]),
    "pdu_radon_fwd_f32": (C.c_int, [_p, _p, _p, C.c_int, _G, _p, C.c_size_t, _p]),
    "pdu_radon_adj_f32": (C.c_int, [_p, _p, _p, C.c_int, _G, _p, C.c_size_t, _p]),
    "pdu_radon_adj_weighted_f32": (C.c_int, [_p, _p, _p, C.c_int, _G, C.c_int, _p, C.c_size_t, _p]),
    "pdu_filter_workspace_bytes": (C.c_size_t, [C.c_int]),
    "pdu_filter_prepare_f32": (C.c_int, [_p, _p, C.c_size_t, C.c_int, _p]),
    "pdu_filter_sinogram_f32": (C.c_int, [_p, _p, _p, _p, C.c_size_t, C.c_long, C.c_int, _p]),
    "pdu_filter_sinogram_weighted_f32": (C.c_int, [_p, _p, _p, _p, _p, C.c_size_t, C.c_long, C.c_int, _p]),
    "pdu_nufft_plan_create": (C.c_int, [C.POINTER(_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_int, _p, _p, _p, _p]),
    "pdu_nufft_plan_destroy": (C.c_int, [_p]),
    "pdu_nufft_workspace_bytes": (C.c_size_t, [_p, C.c_int]),
    "pdu_nufft_fwd_c64": (C.c_int, [_p, _p, _p, _p, _p, C.c_int, C.c_int, C.c_int, C.c_long, C.c_float, _p,
                                    C.c_size_t, _p]),
    "pdu_nufft_adj_c64": (C.c_int, [_p, _p, _p, _p, _p, C.c_int, C.c_int, C.c_int, C.c_long, C.c_float, _p,
                                    C.c_size_t, _p]),
    "pdu_nufft_csr_bytes": (C.c_size_t, [_p, C.c_long]),
    "pdu_nufft_csr_bytes2": (C.c_size_t, [_p, C.c_long, C.POINTER(C.c_size_t)]),
    "pdu_nufft_has_fused_path": (C.c_int, [_p]),
    "pdu_nufft_bins_bytes": (C.c_size_t, [_p, C.c_long, C.POINTER(C.c_size_t)]),
    "pdu_nufft_bins_build": (C.c_int, [_p, _p, C.c_long, _p, C.c_size_t, _p]),
    "pdu_nufft_binned_workspace_bytes": (C.c_size_t, [_p, C.c_int, C.c_long]),
    "pdu_nufft_fwd_binned_c64": (C.c_int, [_p, _p, _p, _p, C.c_int, C.c_int, C.c_int, C.c_long, C.c_float, _p, C.c_int, _p,
                                           C.c_size_t, _p]),
    "pdu_nufft_adj_binned_c64": (C.c_int, [_p, _p, _p, _p, _p, C.c_int, C.c_int, C.c_int, C.c_long, C.c_float, _p, C.c_int, _p,
                                           C.c_size_t, _p]),
    "pdu_nufft_adj_smaps_grad_c64": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, C.c_int, C.c_int, C.c_int, C.c_long, C.c_float,
                                               C.c_int, C.c_int, _p, C.c_size_t, _p]),
    "pdu_toep_plan_create": (C.c_int, [C.POINTER(_p), C.c_int, C.c_int]),
    "pdu_toep_workspace_bytes": (C.c_size_t, [_p, C.c_int]),
    "pdu_toep_kernel_c64": (C.c_int, [_p, _p, _p, _p, C.c_int, C.c_float, _p, C.c_size_t, _p]),
    "pdu_toep_apply_c64": (C.c_int, [_p, _p, _p, _p, C.c_int, _p, C.c_int, C.c_int, C.c_int, C.c_int, _p, C.c_size_t, _p]),
    "pdu_toep_smaps_grad_c64": (C.c_int, [_p, _p, _p, _p, _p, C.c_int, _p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                          C.c_int, _p, C.c_size_t, _p]),
    "pdu_toep_cg_workspace_bytes": (C.c_size_t, [_p, C.c_int, C.c_int, C.c_int]),
    "pdu_toep_cg_c64": (C.c_int, [_p, _p, _p, _p, _p, C.c_int, _p, C.c_int, C.c_int, C.c_int, _p, C.c_int, C.c_int, C.c_float,
                                  C.c_int, _p, C.c_size_t, _p]),
    "pdu_complex_from_split_f32": (C.c_int, [_p, _p, _p, C.c_long, C.c_long, _p]),
    "pdu_split_from_complex_f32": (C.c_int, [_p, _p, C.c_long, C.c_long, _p]),
    "pdu_nufft_csr_build": (C.c_int, [_p, _p, C.c_long, _p, C.c_size_t, _p]),
    "pdu_nufft_interp_adj_csr_c64": (C.c_int, [_p, _p, _p, _p, C.c_int, C.c_long, _p]),
    "pdu_nufft_adj_csr_c64": (C.c_int, [_p, _p, _p, _p, _p, C.c_int, C.c_int, C.c_int, C.c_long, C.c_float, _p, _p,
                                        C.c_size_t, _p]),
    "pdu_nufft_interp_fwd_c64": (C.c_int, [_p, _p, _p, _p, C.c_int, C.c_long, _p]),
    "pdu_nufft_interp_adj_c64": (C.c_int, [_p, _p, _p, _p, C.c_int, C.c_long, _p]),
    "pdu_concat_f32": (C.c_int, [_p, _p, _p, _p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_long, C.c_float, C.c_int, _p]),
    "pdu_concat_mixed_f32": (C.c_int, [_p, _p, _p, _p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_long, C.c_float, C.c_int,
                                       C.c_int, _p]),
    "pdu_residual_slice_f32": (C.c_int, [_p, _p, _p, _p, C.c_int, C.c_int, C.c_long, C.c_int, C.c_int, C.c_int, _p]),
    "pdu_bias_prelu_f32": (C.c_int, [_p, _p, _p, C.c_int, C.c_int, C.c_int, C.c_long, C.c_int, _p]),
    "pdu_bias_prelu_fwd_f32": (C.c_int, [_p, _p, _p, _p, C.c_int, C.c_int, C.c_int, C.c_long, C.c_int, _p]),
    "pdu_channel_sum_f32": (C.c_int, [_p, _p, _p, C.c_size_t, C.c_int, C.c_int, C.c_long, C.c_int, _p]),
    "pdu_bias_prelu_bwd_workspace_bytes": (C.c_size_t, [C.c_int]),
    "pdu_bias_prelu_bwd_f32": (C.c_int, [_p, _p, _p, _p, C.c_int, _p, _p, _p, _p, C.c_size_t, C.c_int, C.c_int, C.c_long, C.c_int, _p]),
    "pdu_bias_prelu_place_f32": (C.c_int, [_p, _p, _p, C.c_int, _p, C.c_long, _p, C.c_int, C.c_int, C.c_int, C.c_int, _p]),
    "pdu_axpby_f32": (C.c_int, [_p, C.c_float, _p, C.c_float, _p, C.c_long, _p]),
    "pdu_angular_upsample_f32": (C.c_int, [_p, _p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _p]),
    "pdu_angular_upsample_scaled_f32": (C.c_int, [_p, _p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, _p]),
    "pdu_concat_upsample_f32": (C.c_int, [_p, _p, _p, _p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_float, C.c_float, C.c_int, _p]),
    "pdu_angular_upsample_adj_f32": (C.c_int, [_p, _p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _p]),
}

_lib = None
_lock = threading.Lock()


def lib() -> C.CDLL:
    """The loaded library.  Raises if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise PduError(f"{LIB_PATH} is missing: build it with `make -C {_HERE}/csrc` "
                                   "(there is no CPU fallback)")
                handle = C.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(handle, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = handle
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().pdu_last_error()
        raise PduError(f"{what or 'libpdu_b200'} failed with code {rc}: {msg.decode(errors='replace') if msg else ''}")


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def require_cuda(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    """Contiguous CUDA tensor of the given dtype or an error -- never a silent host path."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise PduError(f"{name} is on {t.device}: the pd_unet_b200 operators run on CUDA only (no CPU fallback)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


def set_option(key: str, value: int) -> None:
    check(lib().pdu_set_option(key.encode(), int(value)), "pdu_set_option")


def launch_count(reset: bool = False) -> int:
    return int(lib().pdu_launch_count(1 if reset else 0))


def last_kernel(op: str) -> str:
    """The kernel (name, template shape, grid) the dispatcher of `op` chose in this thread's most recent call."""
    v = lib().pdu_last_kernel(op.encode())
    return v.decode() if v else ""


def device_error(reset: bool = False) -> int:
    """Non-zero if a kernel reported a pipeline time-out since the last reset (include/pdu.h)."""
    return int(lib().pdu_device_error(1 if reset else 0))
