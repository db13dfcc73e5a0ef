"""autograd glue for the fused fusion pool: every tensor operation below is a C-ABI kernel launch.

Forward  (reference aecf/AECFLayer.py:515-541 over torch/nn/functional.py:5847-5865, 6630-6659):
    q-proj GEMM -> packed KV GEMM -> fused pool kernel (scores, softmax, dropout, value sum,
    head mean, curriculum mask) -> out-proj GEMM            [aecf_fusion_fwd, csrc/fusion.cu]
    With the folded key projection (one shared query, the bf16 default): q-proj -> fold -> ONE GEMM that
    yields the values and, as an fp32 side output, the per-head scores -> pool -> out-proj; K never exists.
Backward (SURVEY.md Appendix B; autograd of the same lines in the reference):
    colsum + dWo GEMM + dctx GEMM -> fused recompute pool backward -> dX GEMM + dWkv GEMM
    -> the small query-side products                        [aecf_fusion_bwd]
Nothing the forward computed is kept except the projected K/V and the context.
Mixed precision (``PoolConfig.mixed``): fp32 parameters, bf16 activations.  The forward first rounds the parameters to one
bf16 block (``aecf_param_cast``), runs the bf16 step on those shadows and keeps them for the backward, which writes the
parameter gradients in fp32 (``aecf_pool_desc::param_grads_f32``).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, Optional

import torch

from . import _lib, ops


@dataclass
class PoolConfig:
    num_heads: int
    dropout_p: float
    training: bool              # attention module in training mode (dropout on)
    masking: int                # 0 none, 1 CurriculumMasking in training mode, 2 in eval mode
    base_mask_prob: float = 0.15
    entropy_target: float = 0.7
    min_active: int = 1
    seed: int = 0
    offset: int = 0
    rng_state: Optional[torch.Tensor] = None    # device int64 {seed, offset} read at run time (CUDA-graph capture)
    row0: int = 0
    q_shared: bool = True
    seq_first: bool = False     # key/value are [M, B, D] (batch_first=False), used in place
    fold: bool = False          # folded key projection (include/aecf_b200.h): shared query, key is value
    want_mask_bits: bool = False
    bias_strides: tuple = (0, 0)        # (batch, head[, query]) element strides of the additive score bias
    tgt_len: int = 1            # fusion queries per sample; > 1: per-row queries [B, S, D] / [S, B, D], rows (b, s)
    # data-parallel hook: called in backward with (name, grad tensor) for each parameter gradient it produced
    grad_ready: Optional[Callable[[str, torch.Tensor], None]] = None
    # data-parallel: {parameter name: tensor} the backward writes that parameter's gradient into
    # (slices of the all-reduce bucket), instead of allocating it
    grad_buffers: Optional[dict] = None
    # fused CurriculumMasking.entropy_loss: the target the module's entropy_loss() would use after this forward; the
    # forward kernel then also produces the loss scalar (None: not wanted / not a training-mode masking forward)
    loss_target: Optional[float] = None
    # where the backward's gradient tail runs (side stream + fork / join events; None: on the compute stream)
    side: Optional["SideStream"] = None
    # data-parallel, folded path: sum the raw gradient sums over the ranks inside the backward (aecf_b200.dp.FusedGradSum)
    dp: Optional[object] = None
    # int64 [nb] device tensor: pool only these samples of the batch, in place (aecf_pool_desc::row_index)
    sample_index: Optional[torch.Tensor] = None
    # mixed precision: fp32 parameters (and shared query), bf16 key / value.  The forward rounds the parameters to a bf16
    # shadow (one launch, every call: never cached) and runs the bf16 step on it; the parameter gradients come out fp32
    mixed: bool = False


class SideStream:
    """A second stream of the pool's device and the events that fork the backward's gradient tail onto it (twice) and join
    it back (``aecf_fusion_grads.side_stream / fork_event / fork_event2 / join_event``).  The tail -- split-K folds, column sums, the
    rank-H key/query terms, with data parallelism the cross-rank sum -- then runs NEXT TO the dX product.  Works eagerly
    and under CUDA-graph capture (the event edges become graph edges)."""

    def __init__(self, device: torch.device):
        self.device = device
        self.stream = torch.cuda.Stream(device=device)
        self.fork, self.fork2, self.join = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
        with torch.cuda.device(device):                 # the handles exist only after a first record
            for event in (self.fork, self.fork2, self.join):
                event.record(self.stream)

    def __deepcopy__(self, memo):                       # a copied module gets a stream and events of its own
        return SideStream(self.device)

    def __reduce__(self):
        return (SideStream, (self.device,))


def _rows(x3d: torch.Tensor) -> torch.Tensor:
    """[A, B, D] contiguous -> [A*B, D] view."""
    return x3d.reshape(x3d.shape[0] * x3d.shape[1], x3d.shape[2])


class FusedPoolFunction(torch.autograd.Function):
    """out, pooled, entropy, mask_rate, masked, mask_bits = f(query, key, value, params...).

    One C-ABI call for the forward (``aecf_fusion_fwd``), one for the backward (``aecf_fusion_bwd``).
    """

    @staticmethod
    def forward(ctx, q_src, key, value, in_w, in_b, out_w, out_b, score_bias, cfg: PoolConfig):
        dev = ops.require_cuda(q_src, key, value, in_w, in_b, out_w, out_b, score_bias)
        dt = key.dtype
        D = key.shape[-1]
        fold = bool(cfg.fold)
        if cfg.seq_first:
            M, B = key.shape[0], key.shape[1]
            kv_strides = (1, B) if fold else (2 * D, B * 2 * D)     # folded: strides in rows of [B*M, .] matrices
        else:
            B, M = key.shape[0], key.shape[1]
            kv_strides = (0, 0)
        H = cfg.num_heads
        hs, hsp = ops.fold_score_cols(dt, H)
        S = int(cfg.tgt_len)
        R = B * S                       # query rows (b, s): b-major for batch-first input, s-major for sequence-first
        index = cfg.sample_index
        NB = B if index is None else int(index.numel())        # rows the pool kernels and the info outputs see
        desc = ops.make_pool_desc(
            dev, dt, batch=NB, num_tokens=M, embed_dim=D, num_heads=cfg.num_heads, training=cfg.training,
            masking=cfg.masking, min_active=cfg.min_active, q_is_shared=cfg.q_shared,
            base_mask_prob=cfg.base_mask_prob, entropy_target=cfg.entropy_target, dropout_p=cfg.dropout_p,
            seed=cfg.seed, offset=cfg.offset, row0=cfg.row0, bias_strides=cfg.bias_strides, kv_strides=kv_strides,
            fold_key=fold, rng_state=cfg.rng_state, tgt_len=S,
            q_strides=(1, B) if (S > 1 and cfg.seq_first) else (0, 0), row_index=index, src_rows=B if index is not None else 0,
            param_grads_f32=cfg.mixed)
        IR = NB * S                                            # rows of the info tensors

        q_in = q_src.reshape(D) if cfg.q_shared else q_src.reshape(R, D)
        if not q_in.is_contiguous():
            q_in = q_in.contiguous()
        if cfg.mixed:                                          # the bf16 shadows stand in for the fp32 parameters from here on
            _, (in_w, in_b, out_w, out_b, q_sh) = ops.param_cast(
                [in_w, in_b, out_w, out_b, q_in if cfg.q_shared else None])
            if cfg.q_shared:
                q_in = q_sh
        qp = torch.empty((D,), dtype=torch.float32, device=dev) if cfg.q_shared else torch.empty((R, D), dtype=dt, device=dev)
        kv = torch.empty((B * M, D if fold else 2 * D), dtype=dt, device=dev)     # folded: the values only
        scores = torch.empty((B * M, hs), dtype=torch.float32, device=dev) if fold else None
        folded_w = torch.empty((D + hsp, D), dtype=dt, device=dev) if fold else None
        attn = torch.empty((R, D), dtype=dt, device=dev)
        out = torch.empty((R, D), dtype=dt, device=dev)
        pooled = torch.empty((IR, M), dtype=torch.float32, device=dev)       # info tensors: rows b*S + s always
        entropy = torch.empty((IR,), dtype=torch.float32, device=dev)
        mask_rate = torch.empty((IR,), dtype=torch.float32, device=dev)
        masked = torch.empty((IR, M), dtype=torch.float32, device=dev)
        bits = torch.empty((IR if cfg.want_mask_bits else 0,), dtype=torch.uint8, device=dev)
        loss = torch.empty((0,), dtype=torch.float32, device=dev)
        if cfg.loss_target is not None and cfg.masking == 1 and ops.pool_fwd_has_loss(desc, fold):
            loss = torch.empty((1,), dtype=torch.float32, device=dev)
            ws = ops.loss_workspace(dev)
            desc.loss_out, desc.loss_workspace, desc.loss_target = loss.data_ptr(), ws.data_ptr(), float(cfg.loss_target)
        p = _lib.ptr
        tensors = _lib.FusionTensors(
            query=p(q_in), key=p(key), value=p(value), in_proj_weight=p(in_w), in_proj_bias=p(in_b),
            out_proj_weight=p(out_w), out_proj_bias=p(out_b), score_bias=p(score_bias),
            q_proj=p(qp), kv=p(kv), ctx=p(attn), out=p(out), pooled=p(pooled), entropy=p(entropy),
            mask_rate=p(mask_rate), masked=p(masked), mask_bits=p(bits) if cfg.want_mask_bits else None,
            scores=p(scores), folded_w=p(folded_w))
        ops.fusion_fwd(desc, tensors, dev)

        ctx.cfg, ctx.desc = cfg, desc
        # gradients of outputs the loss does not use arrive as None instead of freshly zero-filled tensors:
        # no fill kernels, and the backward kernel skips the d_pooled / d_entropy terms altogether
        ctx.set_materialize_grads(False)
        ctx.shape = (B, M, D)
        ctx.query_rows = R
        ctx.info_rows = IR
        ctx.index = index
        ctx.q_shape = q_src.shape
        ctx.save_for_backward(q_in, key, value, in_w, in_b, out_w, out_b, qp, kv, attn, score_bias, scores, folded_w)
        desc.loss_out = desc.loss_workspace = None      # the descriptor is kept for the backward: no dangling pointers
        if cfg.masking != 2:                            # entropy is detached in training mode (reference :278)
            ctx.mark_non_differentiable(mask_rate, masked, bits, entropy, loss)
        else:
            ctx.mark_non_differentiable(mask_rate, masked, bits, loss)
        return out, pooled, entropy, mask_rate, masked, bits, loss

    @staticmethod
    def backward(ctx, g_out, g_pooled, g_entropy, _g_rate, _g_masked, _g_bits, _g_loss):
        cfg: PoolConfig = ctx.cfg
        q_in, key, value, in_w, in_b, out_w, out_b, qp, kv, attn, score_bias, scores, folded_w = ctx.saved_tensors
        B, M, D = ctx.shape
        R = ctx.query_rows
        dev, dt = key.device, key.dtype
        need_q, need_key, need_value, need_in_w, need_in_b, need_out_w, need_out_b = ctx.needs_input_grad[:7]
        notify = cfg.grad_ready

        if g_out is None:
            g = torch.zeros((R, D), dtype=dt, device=dev)
        else:
            g = g_out.reshape(R, D)
            if g.dtype != dt or not g.is_contiguous():
                g = g.to(dt).contiguous()
        d_pooled = None
        if g_pooled is not None:
            d_pooled = g_pooled.reshape(ctx.info_rows, M).to(torch.float32).contiguous()
        d_entropy = None
        if g_entropy is not None and cfg.masking == 2:
            d_entropy = g_entropy.reshape(ctx.info_rows).to(torch.float32).contiguous()
        ctx.desc.row_index = None if ctx.index is None else ctx.index.data_ptr()     # (kept alive by ctx.index)

        new = lambda shape, dtype=dt: torch.empty(shape, dtype=dtype, device=dev)
        # folded: rows of d_kv are [dV (D) | ds (HSP)]
        d_kv_cols = D + ops.fold_score_cols(dt, cfg.num_heads)[1] if cfg.fold else 2 * D
        d_ctx, d_kv = new((R, D)), new((B * M, d_kv_cols))
        d_q_rows = None if cfg.q_shared else new((R, D))
        d_key = new(key.shape) if need_key else None
        d_value = new(value.shape) if (value is not None and need_value) else None
        # fused tail: the folded backward as one call; with cfg.dp the cross-rank sum happens inside it and the
        # gradients come back final, so they go to fresh tensors autograd owns, not into the all-reduce bucket
        fused_dp = cfg.dp if (cfg.fold and cfg.dp is not None and cfg.dp.usable(ctx.desc)) else None
        bufs = {} if fused_dp is not None else (cfg.grad_buffers or {})
        if fused_dp is not None:
            notify = None

        # the parameter gradients: in the parameter dtype -- fp32 in mixed precision, where `like` is the bf16 shadow
        grad_dtype = torch.float32 if cfg.mixed else None

        def grad_like(name, like):
            dtype = grad_dtype or like.dtype
            b = bufs.get(name)
            if b is not None and b.numel() == like.numel() and b.dtype == dtype and b.is_contiguous():
                return b.view(like.shape)
            return torch.empty_like(like, dtype=dtype)

        d_q = (grad_like("query", q_in) if cfg.q_shared else new(q_in.shape, q_in.dtype)) if need_q else None
        d_in_w = grad_like("in_proj_weight", in_w) if need_in_w else None
        d_in_b = grad_like("in_proj_bias", in_b) if (need_in_b and in_b is not None) else None
        d_out_w = grad_like("out_proj.weight", out_w) if need_out_w else None
        d_out_b = grad_like("out_proj.bias", out_b) if (need_out_b and out_b is not None) else None

        p = _lib.ptr
        tensors = _lib.FusionTensors(
            query=p(q_in), key=p(key), value=p(value), in_proj_weight=p(in_w), in_proj_bias=p(in_b),
            out_proj_weight=p(out_w), out_proj_bias=p(out_b), score_bias=p(score_bias),
            q_proj=p(qp), kv=p(kv), ctx=p(attn), scores=p(scores), folded_w=p(folded_w))
        grads = _lib.FusionGrads(
            d_out=p(g), d_pooled=p(d_pooled), d_entropy=p(d_entropy), d_ctx=p(d_ctx), d_kv=p(d_kv), d_q_rows=p(d_q_rows),
            d_key=p(d_key), d_value=p(d_value), d_query=p(d_q), d_in_proj_weight=p(d_in_w), d_in_proj_bias=p(d_in_b),
            d_out_proj_weight=p(d_out_w), d_out_proj_bias=p(d_out_b))
        side = cfg.side
        if side is not None and cfg.fold and side.device == dev:
            grads.side_stream, grads.fork_event, grads.fork_event2, grads.join_event = (
                side.stream.cuda_stream, side.fork.cuda_event, side.fork2.cuda_event, side.join.cuda_event)
        if fused_dp is not None:
            grads.dp = fused_dp.pointer()
            fused_dp.ran = True
        ws = ops.fusion_workspace(ctx.desc, dev)
        ops.fusion_bwd(ctx.desc, tensors, grads, ws, dev)
        if notify is not None:                          # one bucket all-reduce after the backward (GradientSync.finish)
            for name, t in (("out_proj.bias", d_out_b), ("out_proj.weight", d_out_w), ("in_proj_weight", d_in_w),
                            ("in_proj_bias", d_in_b)):
                if t is not None:
                    notify(name, t)
        if d_q is not None:
            d_q = d_q.reshape(ctx.q_shape)
        return d_q, d_key, d_value, d_in_w, d_in_b, d_out_w, d_out_b, None, None


class EntropyLossFunction(torch.autograd.Function):
    """CurriculumMasking.entropy_loss (reference aecf/AECFLayer.py:285-314) as two tiny kernels."""

    @staticmethod
    def forward(ctx, entropy, target: float):
        e = entropy.reshape(-1).to(torch.float32).contiguous()
        ctx.save_for_backward(e)
        ctx.target, ctx.shape, ctx.dtype = target, entropy.shape, entropy.dtype
        return ops.entropy_loss_fwd(e, target).to(entropy.dtype)

    @staticmethod
    def backward(ctx, g):
        (e,) = ctx.saved_tensors
        d = ops.entropy_loss_bwd(e, ctx.target, g.reshape(1).to(torch.float32).contiguous())
        return d.reshape(ctx.shape).to(ctx.dtype), None


class EntropyFunction(torch.autograd.Function):
    """compute_entropy / eval-mode CurriculumMasking entropy on caller-supplied weights
    (reference aecf/AECFLayer.py:101-128, 150-156): clamp(-sum xlogy(w, w), 0, log L), differentiable."""

    @staticmethod
    def forward(ctx, weights):
        w2 = weights.reshape(-1, weights.shape[-1]).to(torch.float32).contiguous()
        _, entropy, _ = ops.curriculum_mask(w2, 3, want_masked=False)
        ctx.save_for_backward(w2)
        ctx.shape, ctx.dtype = weights.shape, weights.dtype
        return entropy.reshape(weights.shape[:-1]).to(weights.dtype)

    @staticmethod
    def backward(ctx, g):
        (w2,) = ctx.saved_tensors
        d = ops.entropy_bwd(w2, g.reshape(-1).to(torch.float32).contiguous())
        return d.reshape(ctx.shape).to(ctx.dtype)


class SdpaFunction(torch.autograd.Function):
    """The projection-free single-head attention of the functional fast path (reference aecf/AECFLayer.py:556-581),
    differentiable like the reference's: the backward recomputes the weights (two kernels, nothing stored)."""

    @staticmethod
    def forward(ctx, q, k, v):
        ctx.save_for_backward(q, k, v)
        return ops.sdpa_fwd(q, k, v)

    @staticmethod
    def backward(ctx, g):
        q, k, v = ctx.saved_tensors
        d_q, d_k, d_v = ops.sdpa_bwd(q, k, v, g.to(q.dtype).contiguous())
        return (d_q if ctx.needs_input_grad[0] else None, d_k if ctx.needs_input_grad[1] else None,
                d_v if ctx.needs_input_grad[2] else None)


class CurriculumMaskFunction(torch.autograd.Function):
    """Stand-alone training-mode CurriculumMasking.forward on user weights (reference aecf/AECFLayer.py:168-283): the
    masked, renormalised weights keep their graph like the reference's ``final_weights``; entropy and mask_rate do not."""

    @staticmethod
    def forward(ctx, weights, base_mask_prob: float, min_active: int, seed: int, offset: int):
        w2 = weights.detach().reshape(-1, weights.shape[-1]).to(torch.float32).contiguous()
        masked, entropy, mask_rate = ops.curriculum_mask(w2, 1, base_mask_prob=base_mask_prob, min_active=min_active,
                                                         seed=seed, offset=offset)
        ctx.save_for_backward(w2)
        ctx.args = (base_mask_prob, min_active, seed, offset)
        ctx.shape, ctx.dtype = weights.shape, weights.dtype
        ctx.mark_non_differentiable(entropy, mask_rate)
        return masked.reshape(weights.shape).to(weights.dtype), entropy, mask_rate

    @staticmethod
    def backward(ctx, g_masked, _g_entropy, _g_rate):
        (w2,) = ctx.saved_tensors
        base_mask_prob, min_active, seed, offset = ctx.args
        g = g_masked.reshape(w2.shape).to(torch.float32).contiguous()
        d = ops.curriculum_mask_bwd(w2, g, base_mask_prob=base_mask_prob, min_active=min_active, seed=seed, offset=offset)
        return d.reshape(ctx.shape).to(ctx.dtype), None, None, None, None
