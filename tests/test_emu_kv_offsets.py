"""K/V token strides past 2^31 bytes, through the raw C ABI on the host emulation (tests/cuda_emu), on CPU tensors.

A sequence-first batch gives the pool kernels a token stride of B * 2D elements (unfolded) or B rows of D (folded), so at
large B the tokens of one sample lie gigabytes apart.  Every case here runs the same data twice: packed with
kv_strides = (0, 0), and spread over a buffer with a token stride of at least 2^31 bytes.  Forward outputs, mask bits and
gradients must be identical bit for bit.  The wide buffer is an anonymous mapping without a swap reservation: only the
pages the kernels touch are ever backed, so a case costs a few megabytes.  The kernels' view of it starts 2^31 bytes into
the mapping, so an offset that wraps to a negative 32-bit value reads mapped zero pages and fails the comparison instead
of faulting.
"""
import ctypes as C
import mmap

import pytest
import torch

from aecf_b200 import _lib, ops
from tests.emu_support import cuda_emulation  # noqa: F401  (fixture)

pytestmark = pytest.mark.usefixtures("cuda_emulation")

GUARD = 1 << 31                 # bytes of the mapping in front of the kernels' view
MAP_NORESERVE = getattr(mmap, "MAP_NORESERVE", 0x4000)      # Linux value; the mmap module exports it from Python 3.13
B, M, D, H = 4, 3, 64, 4


class WideBuffer:
    """`tokens` blocks of `rows` x `cols` elements, block m starting m * stride elements after block 0."""

    def __init__(self, dtype, tokens, rows, cols, stride):
        self.dtype, self.rows, self.cols, self.stride = dtype, rows, cols, stride
        es = torch.empty((), dtype=dtype).element_size()
        nbytes = GUARD + ((tokens - 1) * stride + rows * cols) * es
        self._map = mmap.mmap(-1, nbytes, flags=mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS | MAP_NORESERVE)
        self.flat = torch.frombuffer(self._map, dtype=torch.uint8)[GUARD:].view(dtype)

    def block(self, m):
        return self.flat[m * self.stride: m * self.stride + self.rows * self.cols].view(self.rows, self.cols)

    def data_ptr(self):
        return self.flat.data_ptr()


def _desc(dtype, kv_strides, tgt_len=1, q_is_shared=True):
    return ops.make_pool_desc(torch.device("cpu"), dtype, batch=B, num_tokens=M, embed_dim=D, num_heads=H, training=True,
                              masking=1, min_active=1, q_is_shared=q_is_shared, base_mask_prob=0.5, entropy_target=0.7,
                              dropout_p=0.1, seed=11, offset=3, row0=0, kv_strides=kv_strides, tgt_len=tgt_len)


def _fwd_outputs(rows, dtype):
    return dict(ctx=torch.zeros(rows, D, dtype=dtype), pooled=torch.zeros(rows, M), entropy=torch.zeros(rows),
                mask_rate=torch.zeros(rows), masked=torch.zeros(rows, M), bits=torch.zeros(rows, dtype=torch.uint8))


def _fwd(fn, desc, first, kv_ptr, rows, dtype):
    o = _fwd_outputs(rows, dtype)
    rc = fn(C.byref(desc), first, kv_ptr, None, o["ctx"].data_ptr(), o["pooled"].data_ptr(), o["entropy"].data_ptr(),
            o["mask_rate"].data_ptr(), o["masked"].data_ptr(), o["bits"].data_ptr(), None)
    _lib.check(rc, "pool forward")
    return o


def _assert_identical(got, want):
    differ = {k: float((got[k].double() - want[k].double()).abs().max()) for k in want if not torch.equal(got[k], want[k])}
    assert not differ, f"max |diff| per output: {differ}"


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_unfolded_token_stride_past_2gb(dtype, cuda_emulation):
    lib = cuda_emulation
    torch.manual_seed(1)
    es = torch.empty((), dtype=dtype).element_size()
    stride = (1 << 31) // es                       # token stride in elements: 2^31 bytes
    kv = torch.randn(B, M, 2 * D).to(dtype)
    q = torch.randn(D)
    d_ctx = torch.randn(B, D).to(dtype)
    d_pooled = torch.randn(B, M)
    wide = WideBuffer(dtype, M, B, 2 * D, stride)
    for m in range(M):
        wide.block(m).copy_(kv[:, m])
    packed, strided = _desc(dtype, (0, 0)), _desc(dtype, (2 * D, stride))
    got = _fwd(lib.aecf_pool_fwd, strided, q.data_ptr(), wide.data_ptr(), B, dtype)
    assert _lib.pool_last_kernel().startswith("stream M=3 J=1 PAD=0 fold=0 "), _lib.pool_last_kernel()
    want = _fwd(lib.aecf_pool_fwd, packed, q.data_ptr(), kv.data_ptr(), B, dtype)

    def bwd(desc, kv_ptr, d_kv_ptr):
        d_q, d_bias = torch.zeros(D), torch.zeros(2 * D)
        ws = torch.zeros(lib.aecf_pool_bwd_workspace_bytes(C.byref(desc)), dtype=torch.uint8)
        rc = lib.aecf_pool_bwd(C.byref(desc), q.data_ptr(), kv_ptr, None, d_ctx.data_ptr(), d_pooled.data_ptr(), None,
                               d_kv_ptr, d_q.data_ptr(), d_bias.data_ptr(), ws.data_ptr(), ws.numel(), None)
        _lib.check(rc, "aecf_pool_bwd")
        assert _lib.pool_last_kernel().startswith("bwd grid-stride M=3 J=1 PAD=0 fold=0 "), _lib.pool_last_kernel()
        return dict(d_q=d_q, d_bias_kv=d_bias)

    d_kv = torch.zeros(B, M, 2 * D, dtype=dtype)
    want.update(bwd(packed, kv.data_ptr(), d_kv.data_ptr()))
    d_wide = WideBuffer(dtype, M, B, 2 * D, stride)
    got.update(bwd(strided, wide.data_ptr(), d_wide.data_ptr()))
    got["d_kv"] = torch.stack([d_wide.block(m) for m in range(M)], 1)
    want["d_kv"] = d_kv
    _assert_identical(got, want)


def test_folded_token_stride_past_2gb(cuda_emulation):
    """Folded layout: the descriptor's strides count rows of v [., D], scores [., HS] and d_vs [., D + HSP]."""
    lib = cuda_emulation
    dtype = torch.bfloat16
    torch.manual_seed(2)
    hs, hsp = ops.fold_score_cols(dtype, H)
    rs_m = (1 << 31) // (D * 2)                    # rows between tokens: 2^31 bytes of v
    v = torch.randn(B, M, D).to(dtype)
    scores = torch.randn(B, M, hs)
    q_proj = torch.randn(D)
    d_ctx = torch.randn(B, D).to(dtype)
    d_pooled = torch.randn(B, M)
    v_wide = WideBuffer(dtype, M, B, D, rs_m * D)
    s_wide = WideBuffer(torch.float32, M, B, hs, rs_m * hs)
    for m in range(M):
        v_wide.block(m).copy_(v[:, m])
        s_wide.block(m).copy_(scores[:, m])
    packed, strided = _desc(dtype, (0, 0)), _desc(dtype, (1, rs_m))
    got = _fwd(lib.aecf_pool_fwd_folded, strided, s_wide.data_ptr(), v_wide.data_ptr(), B, dtype)
    assert _lib.pool_last_kernel().startswith("stream M=3 J=1 PAD=0 fold=1 "), _lib.pool_last_kernel()
    want = _fwd(lib.aecf_pool_fwd_folded, packed, scores.data_ptr(), v.data_ptr(), B, dtype)

    def bwd(desc, s_ptr, v_ptr, d_vs_ptr):
        d_bias = torch.zeros(2 * D)
        ws = torch.zeros(lib.aecf_pool_bwd_workspace_bytes(C.byref(desc)), dtype=torch.uint8)
        rc = lib.aecf_pool_bwd_folded(C.byref(desc), q_proj.data_ptr(), s_ptr, v_ptr, None, d_ctx.data_ptr(),
                                      d_pooled.data_ptr(), None, d_vs_ptr, d_bias.data_ptr(), ws.data_ptr(), ws.numel(), None)
        _lib.check(rc, "aecf_pool_bwd_folded")
        assert _lib.pool_last_kernel().startswith("bwd grid-stride M=3 J=1 PAD=0 fold=1 "), _lib.pool_last_kernel()
        return dict(d_bias_kv=d_bias)

    d_vs = torch.zeros(B, M, D + hsp, dtype=dtype)
    want.update(bwd(packed, scores.data_ptr(), v.data_ptr(), d_vs.data_ptr()))
    d_wide = WideBuffer(dtype, M, B, D + hsp, rs_m * (D + hsp))
    got.update(bwd(strided, s_wide.data_ptr(), v_wide.data_ptr(), d_wide.data_ptr()))
    got["d_vs"] = torch.stack([d_wide.block(m) for m in range(M)], 1)
    want["d_vs"] = d_vs
    _assert_identical(got, want)


def test_multi_query_token_stride_past_2gb(cuda_emulation):
    """Two queries per sample (tgt_len = 2, per-row queries): the multi-query forward and backward kernels."""
    lib = cuda_emulation
    dtype, S = torch.bfloat16, 2
    torch.manual_seed(3)
    stride = (1 << 31) // 2
    kv = torch.randn(B, M, 2 * D).to(dtype)
    q = torch.randn(B * S, D).to(dtype)
    d_ctx = torch.randn(B * S, D).to(dtype)
    d_pooled = torch.randn(B * S, M)
    wide = WideBuffer(dtype, M, B, 2 * D, stride)
    for m in range(M):
        wide.block(m).copy_(kv[:, m])
    packed = _desc(dtype, (0, 0), tgt_len=S, q_is_shared=False)
    strided = _desc(dtype, (2 * D, stride), tgt_len=S, q_is_shared=False)
    got = _fwd(lib.aecf_pool_fwd, strided, q.data_ptr(), wide.data_ptr(), B * S, dtype)
    assert _lib.pool_last_kernel() == "multi fwd M=3 J=1 PAD=0 grid=1", _lib.pool_last_kernel()
    want = _fwd(lib.aecf_pool_fwd, packed, q.data_ptr(), kv.data_ptr(), B * S, dtype)

    def bwd(desc, kv_ptr, d_kv_ptr):
        d_q, d_bias = torch.zeros(B * S, D, dtype=dtype), torch.zeros(2 * D)
        ws = torch.zeros(lib.aecf_pool_bwd_workspace_bytes(C.byref(desc)), dtype=torch.uint8)
        rc = lib.aecf_pool_bwd(C.byref(desc), q.data_ptr(), kv_ptr, None, d_ctx.data_ptr(), d_pooled.data_ptr(), None,
                               d_kv_ptr, d_q.data_ptr(), d_bias.data_ptr(), ws.data_ptr(), ws.numel(), None)
        _lib.check(rc, "aecf_pool_bwd (several queries)")
        assert _lib.pool_last_kernel().startswith("multi bwd M=3 J=1 PAD=0 fold=0 "), _lib.pool_last_kernel()
        return dict(d_q=d_q, d_bias_kv=d_bias)

    d_kv = torch.zeros(B, M, 2 * D, dtype=dtype)
    want.update(bwd(packed, kv.data_ptr(), d_kv.data_ptr()))
    d_wide = WideBuffer(dtype, M, B, 2 * D, stride)
    got.update(bwd(strided, wide.data_ptr(), d_wide.data_ptr()))
    got["d_kv"] = torch.stack([d_wide.block(m) for m in range(M)], 1)
    want["d_kv"] = d_kv
    _assert_identical(got, want)
