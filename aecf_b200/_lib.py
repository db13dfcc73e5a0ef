"""ctypes binding of the C-ABI library ``csrc/libaecf_b200.so`` (``include/aecf_b200.h``).

This is the whole Python<->native boundary: plain pointers, sizes and a stream handle.  There is no
CPU implementation behind it -- if the library is missing, or a call fails, the error is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Optional

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libaecf_b200.so")
ABI_VERSION = 5

# enums of include/aecf_b200.h
F32, BF16 = 0, 1
K_MAJOR, MN_MAJOR = 0, 1
GEMM_AUTO, GEMM_SIMT, GEMM_TCGEN05 = 0, 1, 2
OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_ALIGNMENT, ERR_WORKSPACE, ERR_CUDA = 0, -1, -2, -3, -4, -5
PARAM_CAST_MAX_SEGMENTS = 8

EXPORTS = (
    "aecf_pool_fwd", "aecf_pool_bwd", "aecf_pool_bwd_workspace_bytes",
    "aecf_pool_loss_workspace_bytes", "aecf_pool_fwd_has_loss",
    "aecf_fold_score_cols", "aecf_pool_fwd_folded", "aecf_pool_bwd_folded", "aecf_fold_prepare", "aecf_fold_prepare_query",
    "aecf_fold_finish",
    "aecf_gemm", "aecf_gemm_aux", "aecf_gemm_workspace_bytes",
    "aecf_colsum", "aecf_colsum_workspace_bytes",
    "aecf_entropy_loss_fwd", "aecf_entropy_loss_bwd", "aecf_curriculum_mask", "aecf_curriculum_mask_bwd", "aecf_entropy_bwd", "aecf_sdpa_fwd", "aecf_sdpa_bwd",
    "aecf_param_cast", "aecf_fusion_fwd", "aecf_fusion_bwd", "aecf_fusion_workspace_bytes", "aecf_fusion_grad_sums_bytes",
    "aecf_peer_flag_bytes", "aecf_peer_enable_access", "aecf_peer_allreduce", "aecf_peer_export", "aecf_peer_import",
    "aecf_timing_enable", "aecf_timing_collect", "aecf_timing_site_name", "aecf_timing_site_gemm_kernel",
    "aecf_abi_version", "aecf_strerror", "aecf_last_cuda_error", "aecf_launch_count", "aecf_build_info",
    "aecf_gemm_last_kernel", "aecf_pool_last_kernel",
)


class PoolDesc(C.Structure):
    _fields_ = [
        ("device", C.c_int32), ("dtype", C.c_int32), ("batch", C.c_int64),
        ("num_tokens", C.c_int32), ("embed_dim", C.c_int32), ("num_heads", C.c_int32),
        ("training", C.c_int32), ("masking", C.c_int32), ("min_active", C.c_int32),
        ("q_is_shared", C.c_int32),
        ("base_mask_prob", C.c_float), ("entropy_target", C.c_float), ("dropout_p", C.c_float),
        ("seed", C.c_uint64), ("offset", C.c_uint64), ("row0", C.c_uint64),
        ("bias_stride_b", C.c_int64), ("bias_stride_h", C.c_int64),
        ("kv_stride_b", C.c_int64), ("kv_stride_m", C.c_int64),
        ("fold_key", C.c_int32), ("tgt_len", C.c_int32),
        ("rng_state", C.c_void_p),
        ("q_stride_b", C.c_int64), ("q_stride_s", C.c_int64), ("bias_stride_s", C.c_int64),
        ("loss_out", C.c_void_p), ("loss_workspace", C.c_void_p), ("loss_target", C.c_float), ("param_grads_f32", C.c_int32),
        ("row_index", C.c_void_p), ("src_rows", C.c_int64),
    ]


class GemmDesc(C.Structure):
    _fields_ = [
        ("device", C.c_int32),
        ("dtype_a", C.c_int32), ("dtype_b", C.c_int32), ("dtype_c", C.c_int32), ("dtype_bias", C.c_int32),
        ("a_layout", C.c_int32), ("b_layout", C.c_int32),
        ("accumulate", C.c_int32), ("impl", C.c_int32),
        ("m", C.c_int64), ("n", C.c_int64), ("k", C.c_int64),
        ("lda", C.c_int64), ("ldb", C.c_int64), ("ldc", C.c_int64),
    ]


class PeerDesc(C.Structure):
    _fields_ = [("device", C.c_int32), ("dtype", C.c_int32), ("world", C.c_int32), ("rank", C.c_int32),
                ("count", C.c_int64), ("average", C.c_int32), ("grid_limit", C.c_int32)]


class FusionTensors(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "query", "key", "value", "in_proj_weight", "in_proj_bias", "out_proj_weight", "out_proj_bias", "score_bias",
        "q_proj", "kv", "ctx", "out", "pooled", "entropy", "mask_rate", "masked", "mask_bits", "scores", "folded_w")]


class DpDesc(C.Structure):
    """aecf_dp_desc: the cross-rank gradient sum inside the backward (host arrays of `world` device pointers)."""
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("average", C.c_int32), ("reserved0", C.c_int32),
                ("sums", C.POINTER(C.c_void_p)), ("reduced", C.POINTER(C.c_void_p)), ("flags", C.POINTER(C.c_void_p))]


class FusionGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "d_out", "d_pooled", "d_entropy", "d_ctx", "d_kv", "d_q_rows",
        "d_key", "d_value", "d_query", "d_in_proj_weight", "d_in_proj_bias", "d_out_proj_weight", "d_out_proj_bias",
        "side_stream", "fork_event", "fork_event2", "join_event")] + [("dp", C.POINTER(DpDesc))]


SITE_COUNT = 22


class AecfError(RuntimeError):
    """A C-ABI call returned a negative status."""

    def __init__(self, status: int, what: str, detail: str = ""):
        self.status = status
        super().__init__(f"{what}: {detail}" if detail else what)


class UnsupportedShapeError(AecfError):
    """Valid for the reference, outside what the sm_100a kernels cover.  There is no fallback."""


_lib = None
_lock = threading.Lock()


def _declare(lib):
    vp, f32p, u8p = C.c_void_p, C.c_void_p, C.c_void_p
    lib.aecf_pool_fwd.restype = C.c_int
    lib.aecf_pool_fwd.argtypes = [C.POINTER(PoolDesc), vp, vp, f32p, vp, f32p, f32p, f32p, f32p, u8p, vp]
    lib.aecf_pool_bwd.restype = C.c_int
    lib.aecf_pool_bwd.argtypes = [C.POINTER(PoolDesc), vp, vp, f32p, vp, f32p, f32p, vp, vp, f32p, vp, C.c_size_t, vp]
    lib.aecf_pool_bwd_workspace_bytes.restype = C.c_size_t
    lib.aecf_pool_bwd_workspace_bytes.argtypes = [C.POINTER(PoolDesc)]
    lib.aecf_fold_score_cols.restype = C.c_int
    lib.aecf_fold_score_cols.argtypes = [C.c_int32, C.c_int32]
    lib.aecf_pool_fwd_folded.restype = C.c_int
    lib.aecf_pool_fwd_folded.argtypes = [C.POINTER(PoolDesc), f32p, vp, f32p, vp, f32p, f32p, f32p, f32p, u8p, vp]
    lib.aecf_pool_bwd_folded.restype = C.c_int
    lib.aecf_pool_bwd_folded.argtypes = [C.POINTER(PoolDesc), vp, f32p, vp, f32p, vp, f32p, f32p, vp, f32p, vp, C.c_size_t, vp]
    lib.aecf_fold_prepare.restype = C.c_int
    lib.aecf_fold_prepare.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, f32p, vp, vp, vp]
    lib.aecf_fold_prepare_query.restype = C.c_int
    lib.aecf_fold_prepare_query.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, f32p, vp, vp]
    lib.aecf_pool_loss_workspace_bytes.restype = C.c_size_t
    lib.aecf_pool_loss_workspace_bytes.argtypes = []
    lib.aecf_pool_fwd_has_loss.restype = C.c_int
    lib.aecf_pool_fwd_has_loss.argtypes = [C.POINTER(PoolDesc), C.c_int32]
    lib.aecf_fusion_grad_sums_bytes.restype = C.c_size_t
    lib.aecf_fusion_grad_sums_bytes.argtypes = [C.POINTER(PoolDesc)]
    lib.aecf_fold_finish.restype = C.c_int
    lib.aecf_fold_finish.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, f32p, f32p, vp, vp, f32p, vp]
    lib.aecf_gemm_aux.restype = C.c_int
    lib.aecf_gemm_aux.argtypes = [C.POINTER(GemmDesc), vp, vp, vp, vp, f32p, C.c_int32, C.c_int64, vp, C.c_size_t, vp]
    lib.aecf_gemm.restype = C.c_int
    lib.aecf_gemm.argtypes = [C.POINTER(GemmDesc), vp, vp, vp, vp, vp, C.c_size_t, vp]
    lib.aecf_gemm_workspace_bytes.restype = C.c_size_t
    lib.aecf_gemm_workspace_bytes.argtypes = [C.POINTER(GemmDesc)]
    lib.aecf_colsum.restype = C.c_int
    lib.aecf_colsum.argtypes = [C.c_int32, C.c_int32, C.c_int32, vp, C.c_int64, C.c_int64, C.c_int64, vp, vp,
                                C.c_size_t, vp]
    lib.aecf_colsum_workspace_bytes.restype = C.c_size_t
    lib.aecf_colsum_workspace_bytes.argtypes = [C.c_int64, C.c_int64]
    lib.aecf_entropy_loss_fwd.restype = C.c_int
    lib.aecf_entropy_loss_fwd.argtypes = [C.c_int32, f32p, C.c_int64, C.c_float, f32p, vp]
    lib.aecf_entropy_loss_bwd.restype = C.c_int
    lib.aecf_entropy_loss_bwd.argtypes = [C.c_int32, f32p, C.c_int64, C.c_float, f32p, f32p, vp]
    lib.aecf_curriculum_mask.restype = C.c_int
    lib.aecf_curriculum_mask.argtypes = [C.c_int32, f32p, C.c_int64, C.c_int32, C.c_int32, C.c_float, C.c_int32,
                                         C.c_uint64, C.c_uint64, C.c_uint64, f32p, f32p, f32p, vp]
    lib.aecf_curriculum_mask_bwd.restype = C.c_int
    lib.aecf_curriculum_mask_bwd.argtypes = [C.c_int32, f32p, C.c_int64, C.c_int32, C.c_float, C.c_int32, C.c_uint64, C.c_uint64,
                                             C.c_uint64, f32p, f32p, vp]
    lib.aecf_entropy_bwd.restype = C.c_int
    lib.aecf_entropy_bwd.argtypes = [C.c_int32, f32p, C.c_int64, C.c_int32, f32p, f32p, vp]
    lib.aecf_sdpa_fwd.restype = C.c_int
    lib.aecf_sdpa_fwd.argtypes = [C.c_int32, C.c_int32, vp, vp, vp, vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, vp]
    lib.aecf_sdpa_bwd.restype = C.c_int
    lib.aecf_sdpa_bwd.argtypes = [C.c_int32, C.c_int32, vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, C.c_int64, C.c_int32, C.c_int32,
                                  C.c_int32, vp]
    lib.aecf_param_cast.restype = C.c_int
    lib.aecf_param_cast.argtypes = [C.c_int32, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), vp, vp]
    lib.aecf_fusion_fwd.restype = C.c_int
    lib.aecf_fusion_fwd.argtypes = [C.POINTER(PoolDesc), C.POINTER(FusionTensors), vp, C.c_size_t, vp]
    lib.aecf_fusion_bwd.restype = C.c_int
    lib.aecf_fusion_bwd.argtypes = [C.POINTER(PoolDesc), C.POINTER(FusionTensors), C.POINTER(FusionGrads), vp, C.c_size_t, vp]
    lib.aecf_fusion_workspace_bytes.restype = C.c_size_t
    lib.aecf_fusion_workspace_bytes.argtypes = [C.POINTER(PoolDesc)]
    lib.aecf_peer_flag_bytes.restype = C.c_size_t
    lib.aecf_peer_flag_bytes.argtypes = []
    lib.aecf_peer_enable_access.restype = C.c_int
    lib.aecf_peer_enable_access.argtypes = [C.c_int32, C.c_int32]
    lib.aecf_peer_allreduce.restype = C.c_int
    lib.aecf_peer_allreduce.argtypes = [C.POINTER(PeerDesc), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), vp]
    lib.aecf_peer_export.restype = C.c_int
    lib.aecf_peer_export.argtypes = [C.c_int32, vp, vp, C.POINTER(C.c_int64)]
    lib.aecf_peer_import.restype = C.c_int
    lib.aecf_peer_import.argtypes = [C.c_int32, vp, C.POINTER(C.c_void_p)]
    lib.aecf_timing_enable.restype = C.c_int
    lib.aecf_timing_enable.argtypes = [C.c_int32]
    lib.aecf_timing_collect.restype = C.c_int
    lib.aecf_timing_collect.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_int32)]
    lib.aecf_timing_site_name.restype = C.c_char_p
    lib.aecf_timing_site_name.argtypes = [C.c_int32]
    lib.aecf_timing_site_gemm_kernel.restype = C.c_char_p
    lib.aecf_timing_site_gemm_kernel.argtypes = [C.c_int32]
    lib.aecf_abi_version.restype = C.c_int
    lib.aecf_abi_version.argtypes = []
    lib.aecf_strerror.restype = C.c_char_p
    lib.aecf_strerror.argtypes = [C.c_int]
    lib.aecf_last_cuda_error.restype = C.c_char_p
    lib.aecf_last_cuda_error.argtypes = []
    lib.aecf_launch_count.restype = C.c_uint64
    lib.aecf_launch_count.argtypes = []
    lib.aecf_build_info.restype = C.c_char_p
    lib.aecf_build_info.argtypes = []
    lib.aecf_gemm_last_kernel.restype = C.c_char_p
    lib.aecf_gemm_last_kernel.argtypes = []
    lib.aecf_pool_last_kernel.restype = C.c_char_p
    lib.aecf_pool_last_kernel.argtypes = []


def load():
    """Load the library once.  Raises if it has not been built: there is no other compute path."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"aecf_b200: {LIB_PATH} is missing. Build it with `python -m aecf_b200.build` "
                    "(nvcc, sm_100a). There is no CPU or PyTorch fallback for the fusion path.")
            lib = C.CDLL(LIB_PATH)
            _declare(lib)
            got = lib.aecf_abi_version()
            if got != ABI_VERSION:
                raise RuntimeError(f"aecf_b200: ABI version {got} != expected {ABI_VERSION}; rebuild the library")
            _lib = lib
    return _lib


def check(status: int, what: str) -> None:
    """Map a status code to the exception the reference would have raised for the same mistake."""
    if status == OK:
        return
    lib = load()
    msg = lib.aecf_strerror(status).decode()
    if status == ERR_CUDA:
        raise AecfError(status, what, f"{msg}: {lib.aecf_last_cuda_error().decode()}")
    if status == ERR_UNSUPPORTED:
        raise UnsupportedShapeError(status, what, msg)
    if status == ERR_INVALID:
        raise ValueError(f"{what}: {msg}")
    raise AecfError(status, what, msg)


def launch_count() -> int:
    return int(load().aecf_launch_count())


def gemm_last_kernel() -> str:
    """Which kernel the last aecf_gemm / aecf_gemm_aux call of this thread launched (diagnostics, A/B runs)."""
    return load().aecf_gemm_last_kernel().decode()


def pool_last_kernel() -> str:
    """Which pool kernel and schedule the last pool launch of this thread took (the backward of an autograd call runs on
    autograd's device thread: read it there, e.g. from a gradient hook)."""
    return load().aecf_pool_last_kernel().decode()


def build_info() -> str:
    return load().aecf_build_info().decode()


def timing_enable(on: bool) -> None:
    check(load().aecf_timing_enable(1 if on else 0), "aecf_timing_enable")


def timing_collect() -> dict:
    """{site name: (total ms, launches)} of the kernels enqueued since timing was enabled; synchronises."""
    lib = load()
    ms = (C.c_float * SITE_COUNT)()
    n = (C.c_int32 * SITE_COUNT)()
    check(lib.aecf_timing_collect(ms, n), "aecf_timing_collect")
    return {lib.aecf_timing_site_name(i).decode(): (float(ms[i]), int(n[i])) for i in range(SITE_COUNT) if n[i]}


def site_gemm_kernels() -> dict:
    """{launch site: the GEMM kernel it launched last} for the sites that launched one (diagnostics, A/B runs)."""
    lib = load()
    out = {}
    for i in range(SITE_COUNT):
        k = lib.aecf_timing_site_gemm_kernel(i).decode()
        if k:
            out[lib.aecf_timing_site_name(i).decode()] = k
    return out


def ptr(t) -> Optional[int]:
    return None if t is None else t.data_ptr()
