"""The projections either side of the pool in the reference's documented callers, on the same GEMM kernels as the pool's
own (``aecf_gemm``: tcgen05 for bf16, SIMT for fp32) instead of ``nn.Linear`` -> cuBLAS.

* ``project_tokens([(x_0, lin_0), (x_1, lin_1), ...])`` replaces ``torch.stack([lin_0(x_0), lin_1(x_1), ...], dim=1)`` of the
  reference README (``README.md:183-186``): each modality's encoder GEMM writes straight into its column block of the
  ``[B, M, D]`` token buffer (the ABI takes a strided C: ``ldc = M * D``), so the stack -- a full copy of every token --
  never happens.  Backward: ``dX_m = g_m W_m`` (only where the input wants a gradient), ``dW_m = g_m^T x_m``,
  ``db_m = colsum(g_m)``, reading ``g_m`` in place out of ``d_tokens`` through the same stride.
* ``linear(x, lin)`` is ``lin(x)`` for a 2-D ``x`` (the classifier head, ``README.md:175``).

``lin`` is any module with ``weight [N, K]`` and ``bias [N] | None`` (``nn.Linear`` as the reference builds it), so
state_dicts stay interchangeable with the reference model's.

Mixed precision: an fp32 ``lin`` applied to a bf16 input runs in bf16 on a bf16 rounding of its weight and bias (one
``aecf_param_cast`` launch per call, never cached) and returns bf16; ``d_weight`` / ``d_bias`` come out fp32, straight from
the fp32 sums the bf16 call would round, and the input gradient is bf16.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import torch

from . import _lib, ops


def _dx(g2d: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
    return ops.matmul_nn(g2d, weight, name="projection d_x")


def _is_mixed(x: torch.Tensor, weight: torch.Tensor) -> bool:
    return x.dtype == torch.bfloat16 and weight.dtype == torch.float32


def _shadows(tensors: Sequence) -> List:
    """bf16 roundings of the given fp32 tensors (``None`` stays ``None``), at most one launch per 8 of them."""
    out: List = []
    step = _lib.PARAM_CAST_MAX_SEGMENTS
    for i in range(0, len(tensors), step):
        out.extend(ops.param_cast(list(tensors[i:i + step]))[1])
    return out


class _ProjectTokens(torch.autograd.Function):
    @staticmethod
    def forward(ctx, count: int, *args):
        xs, weights, biases = args[:count], args[count:2 * count], args[2 * count:]
        dev = ops.require_cuda(*xs, *weights)
        B, D = xs[0].shape[0], weights[0].shape[0]
        tokens = torch.empty((B, count, D), dtype=xs[0].dtype, device=dev)
        mixed = [_is_mixed(x, w) for x, w in zip(xs, weights)]
        if any(mixed):                                              # fp32 weights, bf16 inputs: compute on bf16 shadows
            pick = [t if mixed[m % count] else None for m, t in enumerate((*weights, *biases))]
            cast = _shadows(pick)
            weights = tuple(c if c is not None else w for c, w in zip(cast[:count], weights))
            biases = tuple(c if mixed[m] else b for m, (c, b) in enumerate(zip(cast[count:], biases)))
        for m, (x, w, b) in enumerate(zip(xs, weights, biases)):
            if x.dim() != 2 or x.shape[0] != B or w.shape != (D, x.shape[1]):
                raise ValueError("project_tokens: every modality needs a [B, K_m] input and a [D, K_m] weight")
            ops.linear(x.contiguous(), w, b, out=tokens[:, m, :], ldc=count * D, name=f"token projection {m}")
        ctx.count = count
        ctx.mixed = mixed
        ctx.has_bias = [b is not None for b in biases]
        ctx.save_for_backward(*xs, *weights)
        return tokens

    @staticmethod
    def backward(ctx, d_tokens):
        count = ctx.count
        saved = ctx.saved_tensors
        xs, weights = saved[:count], saved[count:]
        d_tokens = d_tokens.contiguous()
        d_x: List = [None] * count
        d_w: List = [None] * count
        d_b: List = [None] * count
        for m in range(count):
            g = d_tokens[:, m, :]                                   # [B, D], row stride count * D, read in place
            if ctx.needs_input_grad[1 + m]:
                d_x[m] = _dx(g, weights[m])
            grad_dtype = torch.float32 if ctx.mixed[m] else None    # fp32 gradients of fp32 masters
            if ctx.needs_input_grad[1 + count + m]:
                d_w[m] = ops.matmul_tn(g, xs[m].contiguous(), out_dtype=grad_dtype, name=f"token projection {m} d_weight")
            if ctx.has_bias[m] and ctx.needs_input_grad[1 + 2 * count + m]:
                d_b[m] = ops.colsum(g, out_dtype=grad_dtype)
        return (None, *d_x, *d_w, *d_b)


def project_tokens(pairs: Sequence[Tuple[torch.Tensor, torch.nn.Module]]) -> torch.Tensor:
    """``torch.stack([lin(x) for x, lin in pairs], dim=1)`` without the stack (and without cuBLAS): ``[B, M, D]``."""
    xs = [x for x, _ in pairs]
    ws = [lin.weight for _, lin in pairs]
    bs = [getattr(lin, "bias", None) for _, lin in pairs]
    return _ProjectTokens.apply(len(pairs), *xs, *ws, *bs)


class _Linear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias):
        ops.require_cuda(x, weight, bias)
        ctx.mixed = _is_mixed(x, weight)
        if ctx.mixed:                                               # fp32 weight, bf16 input: compute on bf16 shadows
            weight, bias = _shadows([weight, bias])
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return ops.linear(x, weight, bias, name="linear")

    @staticmethod
    def backward(ctx, g):
        x, weight = ctx.saved_tensors
        g = g.contiguous()
        grad_dtype = torch.float32 if ctx.mixed else None          # fp32 gradients of fp32 masters
        d_x = _dx(g, weight) if ctx.needs_input_grad[0] else None
        d_w = ops.matmul_tn(g, x, out_dtype=grad_dtype, name="linear d_weight") if ctx.needs_input_grad[1] else None
        d_b = ops.colsum(g, out_dtype=grad_dtype) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return d_x, d_w, d_b


def linear(x: torch.Tensor, lin: torch.nn.Module) -> torch.Tensor:
    """``lin(x)`` for ``x [rows, K]`` on the library's GEMM."""
    if x.dim() != 2:
        raise ValueError("linear expects a 2-D input")
    return _Linear.apply(x.contiguous(), lin.weight, getattr(lin, "bias", None))
