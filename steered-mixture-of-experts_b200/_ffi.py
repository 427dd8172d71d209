"""ctypes binding of libsmoe_b200.so (include/smoe_b200.h).

There is NO fallback: if the library is missing or a call fails, this raises.  PyTorch is used
only for device memory and streams; every pointer handed to the library is `tensor.data_ptr()`.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsmoe_b200.so")

TPIX = 512
ABI_VERSION = 6           # SMOE_ABI_VERSION of include/smoe_b200.h (6 adds smoe_point_jacobian, smoe_jacobian; v5 calls unchanged)
NSCAL = 16
STATS_STRIDE = 24         # floats per batch in the host-visible block: scalars | counts | regsums | pad (16-byte rows)

EXPORTS = [
    "smoe_abi_version", "smoe_last_error", "smoe_param_count", "smoe_packed_stride", "smoe_num_tiles", "smoe_pix_stride",
    "smoe_pack_workspace_bytes", "smoe_backward_workspace_bytes", "smoe_backward_plan_bytes", "smoe_pack", "smoe_pack_fed", "smoe_forward", "smoe_loss", "smoe_loss_partials", "smoe_cotangent", "smoe_ssim_loss_workspace_bytes", "smoe_ssim_loss",
    "smoe_backward", "smoe_suggest_splits", "smoe_reduce_splits", "smoe_grad_finalize", "smoe_update_kernel_list",
    "smoe_adam_step", "smoe_step_begin", "smoe_spatial_keys", "smoe_xchg_window_bytes", "smoe_peer_alloc", "smoe_peer_free",
    "smoe_peer_export", "smoe_peer_open", "smoe_peer_close", "smoe_xchg_publish", "smoe_grad_finalize_peers",
    "smoe_xchg_reduce_tail", "smoe_xchg_status", "smoe_feed", "smoe_halo_pull", "smoe_quant_ranges_bytes", "smoe_quant_ranges", "smoe_quant_route", "smoe_fake_quant_theta", "smoe_ssim_workspace_bytes", "smoe_ssim", "smoe_sqerr", "smoe_quantize", "smoe_rescale",
    "smoe_colminmax", "smoe_point_tiles", "smoe_point_stride", "smoe_point_plan_bytes", "smoe_point_splits",
    "smoe_point_forward", "smoe_point_cotangent", "smoe_point_backward", "smoe_point_xgrad", "smoe_point_jacobian",
    "smoe_jacobian", "smoe_tangent_stride", "smoe_pack_tangent", "smoe_jvp", "smoe_point_jvp",
    "smoe_gn_state_stride", "smoe_point_gn_state_stride", "smoe_gn_state", "smoe_point_gn_state", "smoe_gn_diag",
    "smoe_point_gn_diag", "smoe_gn_diag_scatter",
]


class Cfg(C.Structure):
    _fields_ = [("d", C.c_int32), ("C", C.c_int32), ("precision", C.c_int32), ("margin", C.c_float),
                ("use_determinant", C.c_int32), ("train_inverse_cov", C.c_int32), ("use_yuv", C.c_int32),
                ("train_gammas", C.c_int32), ("only_y_gamma", C.c_int32), ("quantize_pis", C.c_int32),
                ("pis_lb", C.c_float), ("pis_ub", C.c_float), ("pis_bits", C.c_int32),
                ("quantization_mode", C.c_int32), ("q_lb", C.c_float * 5), ("q_ub", C.c_float * 5),
                ("q_bits", C.c_int32 * 5), ("use_diff_center", C.c_int32), ("kernel_count_as_norm_l1", C.c_int32),
                ("radial_as", C.c_int32), ("dense_exec", C.c_int32), ("eps_bits", C.c_int32)]


PIXEL_ABSENT, PIXEL_HALO = -1.0, -2.0          # SMOE_PIXEL_ABSENT / SMOE_PIXEL_HALO


class Batch(C.Structure):
    _fields_ = [("dims", C.c_int32 * 3), ("origin", C.c_int32 * 3), ("extent", C.c_int32 * 3),
                ("tile", C.c_int32 * 3), ("inv_count", C.c_float), ("halo", C.c_int32)]


MAX_PEERS = 8


class Peers(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("win", C.c_void_p * MAX_PEERS)]


class HaloMap(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("d", C.c_int32), ("C", C.c_int32),
                ("blk_lo", (C.c_int32 * 3) * MAX_PEERS), ("blk_hi", (C.c_int32 * 3) * MAX_PEERS),
                ("buf_lo", (C.c_int32 * 3) * MAX_PEERS), ("buf_dims", (C.c_int32 * 3) * MAX_PEERS),
                ("res", C.c_void_p * MAX_PEERS)]


class SsimRegion(C.Structure):
    _fields_ = [("lo", C.c_int32 * 3), ("n", C.c_int32 * 3), ("inv_count", C.c_float)]


class Adam(C.Structure):
    _fields_ = [("alpha", C.c_float * 3), ("beta1", C.c_float * 3), ("beta2", C.c_float * 3),
                ("epsilon", C.c_float * 3), ("grad_clip", C.c_float), ("train_musx", C.c_int32),
                ("train_gammas", C.c_int32)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` (nvcc, sm_100a). "
                "smoe_b200 has no CPU or PyTorch fallback.")
        _lib = C.CDLL(LIB_PATH)
        _lib.smoe_last_error.restype = C.c_char_p
        for name in ("smoe_pack_workspace_bytes", "smoe_backward_workspace_bytes", "smoe_backward_plan_bytes", "smoe_ssim_workspace_bytes",
                     "smoe_ssim_loss_workspace_bytes", "smoe_quant_ranges_bytes", "smoe_xchg_window_bytes",
                     "smoe_point_plan_bytes"):
            getattr(_lib, name).restype = C.c_size_t
        if _lib.smoe_abi_version() != ABI_VERSION:
            raise RuntimeError("libsmoe_b200.so ABI version mismatch")
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().smoe_last_error().decode()
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


def ptr(t):
    """Device (or host) pointer of a torch tensor / None."""
    if t is None:
        return C.c_void_p(0)
    assert t.is_contiguous()
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("smoe_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")
