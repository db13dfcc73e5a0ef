"""Tensor-level wrappers over the C ABI: torch supplies device memory and the stream, nothing else.

Every function enqueues on ``torch.cuda.current_stream()`` of the tensors' device and returns
immediately.  CPU tensors are rejected: the fusion path has no CPU implementation.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib

_DTYPE = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16}

def dtype_code(dtype: torch.dtype) -> int:
    try:
        return _DTYPE[dtype]
    except KeyError:
        raise TypeError(f"aecf_b200 supports float32 and bfloat16 tensors, got {dtype}") from None


def require_cuda(*tensors: Optional[torch.Tensor]) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(
                "aecf_b200 runs only on CUDA tensors (sm_100a kernels, no CPU fallback); "
                f"got a tensor on {t.device}")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"tensors on different devices: {dev} and {t.device}")
    if dev is None:
        raise RuntimeError("no tensor given")
    return dev


def _stream(dev: torch.device) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def _workspace(nbytes: int, dev: torch.device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=dev)


def gemm(a: torch.Tensor, b: torch.Tensor, *, m: int, n: int, k: int, a_layout: int, b_layout: int,
         lda: int, ldb: int, out: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None,
         ldc: Optional[int] = None, bias: Optional[torch.Tensor] = None, accumulate: bool = False,
         impl: int = _lib.GEMM_AUTO, name: str = "gemm") -> torch.Tensor:
    """C[m, n] = sum_k A[m, k] B[n, k] (+ bias[n]); operands addressed as ``include/aecf_b200.h`` says.

    ``a``/``b``/``out`` may be views into larger buffers: only data_ptr and the leading dimension are used.
    """
    dev = require_cuda(a, b, out, bias)
    lib = _lib.load()
    if out is None:
        out = torch.empty((m, n), dtype=out_dtype or a.dtype, device=dev)
        ldc = n
    elif ldc is None:
        ldc = out.stride(0) if out.dim() >= 2 else n
    d = _lib.GemmDesc(device=dev.index or 0, dtype_a=dtype_code(a.dtype), dtype_b=dtype_code(b.dtype),
                      dtype_c=dtype_code(out.dtype), dtype_bias=dtype_code(bias.dtype) if bias is not None else 0,
                      a_layout=a_layout, b_layout=b_layout, accumulate=int(accumulate), impl=impl,
                      m=m, n=n, k=k, lda=lda, ldb=ldb, ldc=ldc)
    ws_bytes = lib.aecf_gemm_workspace_bytes(C.byref(d))
    ws = _workspace(ws_bytes, dev)
    rc = lib.aecf_gemm(C.byref(d), a.data_ptr(), b.data_ptr(), _lib.ptr(bias), out.data_ptr(),
                       ws.data_ptr(), ws.numel(), _stream(dev))
    _lib.check(rc, f"aecf_gemm[{name}] m={m} n={n} k={k}")
    return out


def linear(x2d: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], *, out=None, ldc=None,
           out_dtype=None, name="linear") -> torch.Tensor:
    """x2d [rows, K] (row stride = lda) times weight[N, K]^T (+ bias): torch.nn.functional.linear."""
    rows, k = x2d.shape
    n = weight.shape[0]
    return gemm(x2d, weight, m=rows, n=n, k=k, a_layout=_lib.K_MAJOR, b_layout=_lib.K_MAJOR,
                lda=x2d.stride(0), ldb=weight.stride(0), bias=bias, out=out, ldc=ldc, out_dtype=out_dtype, name=name)


def matmul_nn(x2d: torch.Tensor, weight: torch.Tensor, *, out=None, ldc=None, out_dtype=None, name="matmul_nn"):
    """x2d [rows, K] times weight [K, N] (weight rows are the reduction index): grad wrt a linear's input."""
    rows, k = x2d.shape
    n = weight.shape[1]
    return gemm(x2d, weight, m=rows, n=n, k=k, a_layout=_lib.K_MAJOR, b_layout=_lib.MN_MAJOR,
                lda=x2d.stride(0), ldb=weight.stride(0), out=out, ldc=ldc, out_dtype=out_dtype, name=name)


def matmul_tn(a2d: torch.Tensor, b2d: torch.Tensor, *, out=None, ldc=None, out_dtype=None, name="matmul_tn"):
    """a2d^T b2d for a2d [R, M], b2d [R, N] (reduce over rows): grad wrt a linear's weight."""
    r, m = a2d.shape
    n = b2d.shape[1]
    return gemm(a2d, b2d, m=m, n=n, k=r, a_layout=_lib.MN_MAJOR, b_layout=_lib.MN_MAJOR,
                lda=a2d.stride(0), ldb=b2d.stride(0), out=out, ldc=ldc, out_dtype=out_dtype, name=name)


def colsum(x2d: torch.Tensor, out_dtype: Optional[torch.dtype] = None, name="colsum") -> torch.Tensor:
    dev = require_cuda(x2d)
    lib = _lib.load()
    rows, cols = x2d.shape
    out = torch.empty(cols, dtype=out_dtype or x2d.dtype, device=dev)
    ws = _workspace(lib.aecf_colsum_workspace_bytes(rows, cols), dev)
    rc = lib.aecf_colsum(dev.index or 0, dtype_code(x2d.dtype), dtype_code(out.dtype), x2d.data_ptr(), rows, cols,
                         x2d.stride(0), out.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev))
    _lib.check(rc, "aecf_colsum")
    return out


def param_cast(tensors) -> Tuple[torch.Tensor, list]:
    """bf16 shadows of fp32 parameters, one launch (``aecf_param_cast``): returns the block and, per entry of
    ``tensors`` (``None`` entries stay ``None``), a view of it with that tensor's shape.  Each view starts on a 16-byte
    boundary of the block, so it is a valid GEMM operand."""
    present = [t for t in tensors if t is not None]
    if len(present) > _lib.PARAM_CAST_MAX_SEGMENTS:
        raise ValueError(f"param_cast: at most {_lib.PARAM_CAST_MAX_SEGMENTS} tensors per launch, got {len(present)}")
    dev = require_cuda(*present)
    offsets, total = [], 0
    for t in present:
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise TypeError("param_cast: the parameters must be contiguous float32 tensors")
        offsets.append(total)
        total += (t.numel() + 7) // 8 * 8
    block = torch.empty(max(total, 8), dtype=torch.bfloat16, device=dev)
    if present:
        n = len(present)
        src = (C.c_void_p * n)(*[t.data_ptr() for t in present])
        counts = (C.c_int64 * n)(*[t.numel() for t in present])
        rc = _lib.load().aecf_param_cast(dev.index or 0, n, src, counts, block.data_ptr(), _stream(dev))
        _lib.check(rc, f"aecf_param_cast segments={n}")
    views, i = [], 0
    for t in tensors:
        if t is None:
            views.append(None)
            continue
        views.append(block[offsets[i]:offsets[i] + t.numel()].view(t.shape))
        i += 1
    return block, views


def make_pool_desc(dev: torch.device, dtype: torch.dtype, *, batch: int, num_tokens: int, embed_dim: int,
                   num_heads: int, training: bool, masking: int, min_active: int, q_is_shared: bool,
                   base_mask_prob: float, entropy_target: float, dropout_p: float, seed: int, offset: int,
                   row0: int, bias_strides: Tuple[int, ...] = (0, 0),
                   kv_strides: Tuple[int, int] = (0, 0), fold_key: bool = False,
                   rng_state: Optional[torch.Tensor] = None, tgt_len: int = 1,
                   q_strides: Tuple[int, int] = (0, 0), loss_out: Optional[torch.Tensor] = None,
                   loss_workspace: Optional[torch.Tensor] = None, loss_target: float = 0.0,
                   row_index: Optional[torch.Tensor] = None, src_rows: int = 0,
                   param_grads_f32: bool = False) -> _lib.PoolDesc:
    """``bias_strides`` = (batch, head[, query]) element strides of the additive score bias; ``tgt_len`` > 1 and
    ``q_strides`` (rows of query (b, s): b*q_strides[0] + s*q_strides[1]) describe several queries per sample.
    ``param_grads_f32``: mixed precision (bf16 shadows of fp32 parameters in, fp32 parameter gradients out)."""
    return _lib.PoolDesc(device=dev.index or 0, dtype=dtype_code(dtype), batch=batch, num_tokens=num_tokens,
                         embed_dim=embed_dim, num_heads=num_heads, training=int(training), masking=int(masking),
                         min_active=int(min_active), q_is_shared=int(q_is_shared),
                         base_mask_prob=float(base_mask_prob), entropy_target=float(entropy_target),
                         dropout_p=float(dropout_p), seed=seed & 0xFFFFFFFFFFFFFFFF, offset=offset & 0xFFFFFFFF,
                         row0=row0, bias_stride_b=bias_strides[0], bias_stride_h=bias_strides[1],
                         kv_stride_b=kv_strides[0], kv_stride_m=kv_strides[1], fold_key=int(fold_key),
                         tgt_len=int(tgt_len), rng_state=None if rng_state is None else rng_state.data_ptr(),
                         q_stride_b=q_strides[0], q_stride_s=q_strides[1],
                         bias_stride_s=bias_strides[2] if len(bias_strides) > 2 else 0,
                         loss_out=None if loss_out is None else loss_out.data_ptr(),
                         loss_workspace=None if loss_workspace is None else loss_workspace.data_ptr(),
                         loss_target=float(loss_target),
                         row_index=None if row_index is None else row_index.data_ptr(), src_rows=int(src_rows),
                         param_grads_f32=int(param_grads_f32))


def fold_score_cols(dtype: torch.dtype, num_heads: int) -> Tuple[int, int]:
    """(HS, HSP) of the folded key projection: columns of the fp32 score matrix (heads rounded up to 4) and
    score-gradient columns appended to each d_kv row (heads rounded up to 16 bytes of ``dtype``)."""
    per16 = 8 if dtype == torch.bfloat16 else 4
    return (num_heads + 3) // 4 * 4, (num_heads + per16 - 1) // per16 * per16


def gemm_aux(a: torch.Tensor, b: torch.Tensor, *, m: int, n: int, k: int, aux_cols: int,
             bias: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None,
             impl: int = _lib.GEMM_AUTO) -> Tuple[torch.Tensor, torch.Tensor]:
    """C[m, n] = A B[:n]^T (+ bias) and the fp32 side output aux[m, aux_cols] = A B[n:n+aux_cols]^T, K-major
    operands (``aecf_gemm_aux``).  ``b`` has n + roundup(aux_cols, 16 bytes) rows."""
    dev = require_cuda(a, b, bias)
    lib = _lib.load()
    out = torch.empty((m, n), dtype=out_dtype or a.dtype, device=dev)
    aux_ld = (aux_cols + 3) // 4 * 4
    aux = torch.empty((m, aux_ld), dtype=torch.float32, device=dev)
    d = _lib.GemmDesc(device=dev.index or 0, dtype_a=dtype_code(a.dtype), dtype_b=dtype_code(b.dtype),
                      dtype_c=dtype_code(out.dtype), dtype_bias=dtype_code(bias.dtype) if bias is not None else 0,
                      a_layout=_lib.K_MAJOR, b_layout=_lib.K_MAJOR, accumulate=0, impl=impl,
                      m=m, n=n, k=k, lda=a.stride(0), ldb=b.stride(0), ldc=n)
    ws = _workspace(lib.aecf_gemm_workspace_bytes(C.byref(d)), dev)
    rc = lib.aecf_gemm_aux(C.byref(d), a.data_ptr(), b.data_ptr(), _lib.ptr(bias), out.data_ptr(), aux.data_ptr(),
                           aux_cols, aux_ld, ws.data_ptr(), ws.numel(), _stream(dev))
    _lib.check(rc, f"aecf_gemm_aux m={m} n={n} k={k} aux={aux_cols}")
    return out, aux


def pool_fwd(desc: _lib.PoolDesc, q: torch.Tensor, kv: torch.Tensor, score_bias: Optional[torch.Tensor],
             want_mask_bits: bool = False):
    """Returns ctx [B,D], pooled [B,M], entropy [B], mask_rate [B], masked [B,M], mask_bits [B] or None."""
    dev = require_cuda(q, kv, score_bias)
    lib = _lib.load()
    B, M, D = desc.batch, desc.num_tokens, desc.embed_dim
    ctx = torch.empty((B, D), dtype=kv.dtype, device=dev)
    pooled = torch.empty((B, M), dtype=torch.float32, device=dev)
    entropy = torch.empty((B,), dtype=torch.float32, device=dev)
    mask_rate = torch.empty((B,), dtype=torch.float32, device=dev)
    masked = torch.empty((B, M), dtype=torch.float32, device=dev)
    bits = torch.empty((B,), dtype=torch.uint8, device=dev) if want_mask_bits else None
    rc = lib.aecf_pool_fwd(C.byref(desc), q.data_ptr(), kv.data_ptr(), _lib.ptr(score_bias), ctx.data_ptr(),
                           pooled.data_ptr(), entropy.data_ptr(), mask_rate.data_ptr(), masked.data_ptr(),
                           _lib.ptr(bits), _stream(dev))
    _lib.check(rc, f"aecf_pool_fwd B={B} M={M} D={D} H={desc.num_heads}")
    return ctx, pooled, entropy, mask_rate, masked, bits


def pool_bwd(desc: _lib.PoolDesc, q: torch.Tensor, kv: torch.Tensor, score_bias: Optional[torch.Tensor],
             d_ctx: torch.Tensor, d_pooled: Optional[torch.Tensor], d_entropy: Optional[torch.Tensor]):
    """Returns d_kv [B,M,2D], d_q ([D] fp32 if shared else [B,D]), d_bias_kv [2D] fp32."""
    dev = require_cuda(q, kv, score_bias, d_ctx, d_pooled, d_entropy)
    lib = _lib.load()
    B, M, D = desc.batch, desc.num_tokens, desc.embed_dim
    d_kv = torch.empty((B, M, 2 * D), dtype=kv.dtype, device=dev)
    if desc.q_is_shared:
        d_q = torch.empty((D,), dtype=torch.float32, device=dev)
    else:
        d_q = torch.empty((B, D), dtype=kv.dtype, device=dev)
    d_bias_kv = torch.empty((2 * D,), dtype=torch.float32, device=dev)
    ws = _workspace(lib.aecf_pool_bwd_workspace_bytes(C.byref(desc)), dev)
    rc = lib.aecf_pool_bwd(C.byref(desc), q.data_ptr(), kv.data_ptr(), _lib.ptr(score_bias), d_ctx.data_ptr(),
                           _lib.ptr(d_pooled), _lib.ptr(d_entropy), d_kv.data_ptr(), d_q.data_ptr(),
                           d_bias_kv.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev))
    _lib.check(rc, f"aecf_pool_bwd B={B} M={M} D={D} H={desc.num_heads}")
    return d_kv, d_q, d_bias_kv


def entropy_loss_fwd(entropy: torch.Tensor, target: float) -> torch.Tensor:
    dev = require_cuda(entropy)
    loss = torch.empty((), dtype=torch.float32, device=dev)
    rc = _lib.load().aecf_entropy_loss_fwd(dev.index or 0, entropy.data_ptr(), entropy.numel(), float(target),
                                           loss.data_ptr(), _stream(dev))
    _lib.check(rc, "aecf_entropy_loss_fwd")
    return loss


def entropy_loss_bwd(entropy: torch.Tensor, target: float, d_loss: torch.Tensor) -> torch.Tensor:
    dev = require_cuda(entropy, d_loss)
    d_e = torch.empty_like(entropy)
    rc = _lib.load().aecf_entropy_loss_bwd(dev.index or 0, entropy.data_ptr(), entropy.numel(), float(target),
                                           d_loss.data_ptr(), d_e.data_ptr(), _stream(dev))
    _lib.check(rc, "aecf_entropy_loss_bwd")
    return d_e


def sdpa_fwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    dev = require_cuda(q, k, v)
    B, S, D = q.shape
    T = k.shape[1]
    out = torch.empty_like(q)
    rc = _lib.load().aecf_sdpa_fwd(dev.index or 0, dtype_code(q.dtype), q.data_ptr(), k.data_ptr(), v.data_ptr(),
                                   out.data_ptr(), B, S, T, D, _stream(dev))
    _lib.check(rc, f"aecf_sdpa_fwd B={B} S={S} T={T} D={D}")
    return out


def sdpa_bwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, d_out: torch.Tensor):
    dev = require_cuda(q, k, v, d_out)
    B, S, D = q.shape
    T = k.shape[1]
    d_q, d_k, d_v = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
    ws = torch.empty(2 * B * S, dtype=torch.float32, device=dev)
    rc = _lib.load().aecf_sdpa_bwd(dev.index or 0, dtype_code(q.dtype), q.data_ptr(), k.data_ptr(), v.data_ptr(), d_out.data_ptr(),
                                   d_q.data_ptr(), d_k.data_ptr(), d_v.data_ptr(), ws.data_ptr(), ws.numel() * 4, B, S, T, D,
                                   _stream(dev))
    _lib.check(rc, f"aecf_sdpa_bwd B={B} S={S} T={T} D={D}")
    return d_q, d_k, d_v


def curriculum_mask(weights2d: torch.Tensor, mode: int, *, base_mask_prob: float = 0.15, min_active: int = 1,
                    seed: int = 0, offset: int = 0, row0: int = 0, want_masked: bool = True):
    """Standalone masking stage on fp32 [rows, len] weights.  Returns (masked or None, entropy, mask_rate)."""
    dev = require_cuda(weights2d)
    rows, length = weights2d.shape
    masked = torch.empty_like(weights2d) if want_masked else None
    entropy = torch.empty((rows,), dtype=torch.float32, device=dev)
    mask_rate = torch.empty((rows,), dtype=torch.float32, device=dev)
    rc = _lib.load().aecf_curriculum_mask(dev.index or 0, weights2d.data_ptr(), rows, length, mode,
                                          float(base_mask_prob), int(min_active), seed & 0xFFFFFFFFFFFFFFFF,
                                          offset & 0xFFFFFFFF, row0, _lib.ptr(masked), entropy.data_ptr(),
                                          mask_rate.data_ptr(), _stream(dev))
    _lib.check(rc, f"aecf_curriculum_mask rows={rows} len={length}")
    return masked, entropy, mask_rate


def curriculum_mask_bwd(weights2d: torch.Tensor, d_masked: torch.Tensor, *, base_mask_prob: float, min_active: int, seed: int,
                        offset: int, row0: int = 0) -> torch.Tensor:
    dev = require_cuda(weights2d, d_masked)
    rows, length = weights2d.shape
    d_w = torch.empty_like(weights2d)
    rc = _lib.load().aecf_curriculum_mask_bwd(dev.index or 0, weights2d.data_ptr(), rows, length, float(base_mask_prob),
                                              int(min_active), seed & 0xFFFFFFFFFFFFFFFF, offset & 0xFFFFFFFF, row0,
                                              d_masked.data_ptr(), d_w.data_ptr(), _stream(dev))
    _lib.check(rc, "aecf_curriculum_mask_bwd")
    return d_w


def entropy_bwd(weights2d: torch.Tensor, d_entropy: torch.Tensor) -> torch.Tensor:
    dev = require_cuda(weights2d, d_entropy)
    rows, length = weights2d.shape
    d_w = torch.empty_like(weights2d)
    rc = _lib.load().aecf_entropy_bwd(dev.index or 0, weights2d.data_ptr(), rows, length, d_entropy.data_ptr(),
                                      d_w.data_ptr(), _stream(dev))
    _lib.check(rc, "aecf_entropy_bwd")
    return d_w


def peer_flag_block(dev: torch.device) -> torch.Tensor:
    """A zeroed flag block for ``peer_allreduce`` (one per rank, lives as long as the buckets are mapped)."""
    return torch.zeros(_lib.load().aecf_peer_flag_bytes() // 4, dtype=torch.int32, device=dev)


def peer_allreduce(buckets, flags, rank: int, *, average: bool = False, stream: Optional[int] = None,
                   grid_limit: int = 0, mine: Optional[torch.Tensor] = None) -> None:
    """In-place sum (mean) of ``buckets[rank]`` with every other entry of ``buckets`` -- this process's mappings of
    all ranks' buckets -- over peer memory (``aecf_peer_allreduce``).  Every rank makes the same call with its own
    ``rank``; the call returns at once and completes on the stream when the whole bucket is reduced.  ``buckets`` /
    ``flags`` hold tensors or plain device addresses (IPC mappings); ``mine`` is this rank's bucket tensor when they are
    addresses."""
    mine = buckets[rank] if mine is None else mine
    dev = require_cuda(mine)
    world = len(buckets)
    addr = lambda x: x if isinstance(x, int) else x.data_ptr()
    d = _lib.PeerDesc(device=dev.index or 0, dtype=dtype_code(mine.dtype), world=world, rank=rank,
                      count=mine.numel(), average=int(average), grid_limit=int(grid_limit))
    data = (C.c_void_p * world)(*[addr(b) for b in buckets])
    flag_ptrs = (C.c_void_p * world)(*[addr(f) for f in flags])
    rc = _lib.load().aecf_peer_allreduce(C.byref(d), data, flag_ptrs, _stream(dev) if stream is None else stream)
    _lib.check(rc, f"aecf_peer_allreduce world={world} rank={rank} count={mine.numel()}")


_loss_workspaces: dict = {}


def loss_workspace(dev: torch.device) -> torch.Tensor:
    """The fused entropy_loss term's scratch (per-CTA partial sums and a "CTAs done" counter): zeroed once, re-armed by
    the kernel.  One per device: forwards of one device are expected to be ordered (one stream, or one CUDA graph); it is
    allocated outside any capture (the first eager or warm-up forward)."""
    key = dev.index or 0
    ws = _loss_workspaces.get(key)
    if ws is None:
        ws = torch.zeros(int(_lib.load().aecf_pool_loss_workspace_bytes()), dtype=torch.uint8, device=dev)
        _loss_workspaces[key] = ws
    return ws


def pool_fwd_has_loss(desc: _lib.PoolDesc, folded: bool) -> bool:
    return bool(_lib.load().aecf_pool_fwd_has_loss(C.byref(desc), int(folded)))


def fusion_grad_sums_floats(desc: _lib.PoolDesc) -> int:
    """fp32 elements of one raw-sum buffer of the backward's fused gradient tail (0: this descriptor has none)."""
    return int(_lib.load().aecf_fusion_grad_sums_bytes(C.byref(desc))) // 4


def fusion_workspace(desc: _lib.PoolDesc, dev: torch.device) -> torch.Tensor:
    return _workspace(_lib.load().aecf_fusion_workspace_bytes(C.byref(desc)), dev)


def fusion_fwd(desc: _lib.PoolDesc, tensors: _lib.FusionTensors, dev: torch.device) -> None:
    """Whole forward (q/kv projections, fused pool, out projection) in one C-ABI call."""
    ws = fusion_workspace(desc, dev)
    rc = _lib.load().aecf_fusion_fwd(C.byref(desc), C.byref(tensors), ws.data_ptr(), ws.numel(), _stream(dev))
    _lib.check(rc, f"aecf_fusion_fwd B={desc.batch} M={desc.num_tokens} D={desc.embed_dim} H={desc.num_heads}")


def fusion_bwd(desc: _lib.PoolDesc, tensors: _lib.FusionTensors, grads: _lib.FusionGrads, ws: torch.Tensor,
               dev: torch.device) -> None:
    rc = _lib.load().aecf_fusion_bwd(C.byref(desc), C.byref(tensors), C.byref(grads), ws.data_ptr(), ws.numel(), _stream(dev))
    _lib.check(rc, f"aecf_fusion_bwd B={desc.batch} M={desc.num_tokens} D={desc.embed_dim}")
