"""CPU restatement of the AECF fusion hot path -- TEST INFRASTRUCTURE ONLY.

This module restates, in explicit torch-CPU tensor arithmetic, what the reference
computes for ``MultimodalAttentionPool.forward`` + ``CurriculumMasking`` and the
backward that autograd derives from it.  It is the checker for the CUDA kernels
in ``aecf_b200/csrc``; nothing under ``aecf_b200/`` imports it.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may.

Where the arithmetic lives.  The reference delegates attention to
``torch.nn.MultiheadAttention`` (reference ``aecf/AECFLayer.py:399-407``, called
at ``:515-521``); torch is an unpinned dependency (``requirements.txt:1``
``torch>=2.0.0``; installed here: 2.11.0+cu128).  The math restated below is
``torch/nn/functional.py:5847-5865`` (packed in-projection) and ``:6630-6659``
(scale, scores, softmax, dropout, value sum, out-projection, head mean), plus
reference ``aecf/AECFLayer.py:130-283`` (masking) and ``:285-314`` (loss).

Parity pin.  The reference ships no tests or golden vectors (SURVEY.md section 4), so
the pin is the reference itself, run with the shared Philox uniforms injected:
``tests/golden/make_golden.py`` imports the reference checkout that
``AECF_REFERENCE`` names and writes ``tests/golden/*.npz``;
``tests/test_oracle_golden.py`` checks every function here against them.

Random numbers are *inputs* (``u_mask``, ``u_drop``; see ``oracle/philox.py``):
    mask keeps token m   iff u_mask[b, m]    <= keep_prob[b]
    dropout keeps (h, m) iff u_drop[b, h, m] >= p_drop
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, Optional

import torch

Tensor = torch.Tensor


# ----------------------------------------------------------------------------
# CurriculumMasking
# ----------------------------------------------------------------------------

def shannon_entropy(weights: Tensor) -> Tensor:
    """clamp(-sum xlogy(w, w), 0, log L) -- reference aecf/AECFLayer.py:113-128."""
    h = torch.xlogy(weights, weights).sum(dim=-1).neg()
    return h.clamp(0.0, math.log(weights.size(-1)))


def topk_onehot(weights: Tensor, k: int) -> Tensor:
    """One-hot set of the k largest entries, ties to the lowest index.

    Restates the ``topk`` + scatter of reference aecf/AECFLayer.py:213-257 as a
    rank computation (the form the CUDA kernel uses): entry i is selected iff
    fewer than k entries beat it, where j beats i if w[j] > w[i], or w[j] == w[i]
    and j < i.  Checked against ``torch.topk`` in tests/test_oracle_golden.py.
    """
    L = weights.size(-1)
    wi = weights.unsqueeze(-1)            # [..., i, 1]
    wj = weights.unsqueeze(-2)            # [..., 1, j]
    idx = torch.arange(L)
    earlier = idx.view(1, L) < idx.view(L, 1)          # [i, j] : j < i
    beats = (wj > wi) | ((wj == wi) & earlier)
    rank = beats.sum(dim=-1)
    return (rank < k).to(weights.dtype)


def curriculum_mask(pooled: Tensor, u_mask: Optional[Tensor], *, base_mask_prob: float = 0.15,
                    entropy_target: float = 0.7, min_active: int = 1,
                    training: bool = True) -> Dict[str, Tensor]:
    """CurriculumMasking.forward -- reference aecf/AECFLayer.py:130-283.

    ``pooled`` is (..., L); ``u_mask`` the injected uniforms of the same shape.
    Returns masked weights, the 0/1 mask and the info tensors.  ``entropy`` keeps
    its autograd graph only in eval mode (reference :151-156 vs :278).
    """
    L = pooled.size(-1)
    lead = pooled.shape[:-1]
    zeros = torch.zeros(lead, dtype=pooled.dtype)
    if not training:                                             # :150-156
        return {"masked": pooled, "mask": torch.ones_like(pooled),
                "entropy": shannon_entropy(pooled), "mask_rate": zeros}
    if L <= 1:                                                   # :159-167
        return {"masked": pooled, "mask": torch.ones_like(pooled), "entropy": zeros,
                "mask_rate": zeros.clone(), "target_entropy": zeros.clone()}

    eps = torch.tensor(1e-8, dtype=torch.float32)                # the _eps buffer, :96
    w = torch.where(torch.isfinite(pooled), pooled, torch.zeros((), dtype=pooled.dtype))  # :173-176
    total = w.sum(dim=-1, keepdim=True)                          # :170 / :176
    w = torch.where(total < eps, torch.full((), 1.0 / L, dtype=w.dtype), w / total)      # :178-184

    entropy = shannon_entropy(w)                                 # :190
    log_l = math.log(float(L))
    norm_entropy = (entropy / log_l).clamp(0.0, 1.0)             # :191-192
    keep_prob = (1.0 - base_mask_prob * norm_entropy).unsqueeze(-1).clamp(0.0, 1.0)  # :197-201
    mask = (u_mask.to(keep_prob.dtype) <= keep_prob).to(w.dtype)          # :204 with injected draws

    k = min(int(min_active), L)                                  # :207
    short = mask.sum(dim=-1) < k                                 # :208-209
    mask = torch.where(short.unsqueeze(-1), topk_onehot(w, k), mask)      # :211-260 (replace, not OR)

    kept = w * mask                                              # :263
    kept_sum = kept.sum(dim=-1, keepdim=True)                    # :264
    masked = torch.where(kept_sum > eps, kept / kept_sum, w)     # :267-272
    mask_rate = 1.0 - mask.float().mean(dim=-1)                  # :275
    return {"masked": masked, "mask": mask, "renormalised": w,
            "entropy": entropy.detach(), "mask_rate": mask_rate.detach(),
            "keep_prob": keep_prob.squeeze(-1).detach(),
            "target_entropy": torch.full_like(entropy, log_l * entropy_target)}  # :280


def entropy_loss(entropy: Tensor, last_seq_len: int = 2, entropy_target: float = 0.7) -> Tensor:
    """mean((H - target*log L)^2) with the NaN scrub -- reference aecf/AECFLayer.py:285-314."""
    entropy = torch.nan_to_num(entropy, nan=0.0, posinf=1.0, neginf=0.0)  # :295-296 (no-op when finite)
    log_l = math.log(float(last_seq_len)) if last_seq_len > 1 else 0.0    # :307
    diff = entropy - log_l * entropy_target
    return (diff * diff).mean().clamp(min=0.0)


# ----------------------------------------------------------------------------
# Attention pool forward / backward
# ----------------------------------------------------------------------------

@dataclass
class PoolResult:
    out: Tensor                 # [B, S, D]
    pooled: Tensor              # [B, S, M]  head-averaged post-dropout weights
    info: Dict[str, Tensor] = field(default_factory=dict)
    saved: Dict[str, Tensor] = field(default_factory=dict)


def _round(t: Tensor, storage: Optional[torch.dtype]) -> Tensor:
    """Model a tensor that the CUDA path keeps in HBM in ``storage`` precision."""
    if storage is None or storage == t.dtype:
        return t
    return t.to(storage).to(t.dtype)


def pool_forward(query: Tensor, key: Tensor, value: Optional[Tensor],
                 in_proj_weight: Tensor, in_proj_bias: Optional[Tensor],
                 out_proj_weight: Tensor, out_proj_bias: Optional[Tensor], num_heads: int, *,
                 dropout_p: float = 0.0, training: bool = True,
                 u_drop: Optional[Tensor] = None, u_mask: Optional[Tensor] = None,
                 score_bias: Optional[Tensor] = None,
                 masking: Optional[dict] = None,
                 storage: Optional[torch.dtype] = None, fold_key: bool = False,
                 per_row_query_storage: bool = False) -> PoolResult:
    """MultimodalAttentionPool.forward, batch_first -- reference aecf/AECFLayer.py:409-547
    over torch/nn/functional.py:5847-5865 and :6630-6659.

    query [B,S,D] (an expand of [1,1,D] is fine; S > 1 fusion queries per sample are covered, each (b, s)
    pair is a row of its own for the softmax, the dropout draws u_drop [B,H,S,M] and the mask draws
    u_mask [B,S,M]), key/value [B,M,D].
    ``score_bias`` is the additive float mask torch builds from key_padding_mask
    and attn_mask (functional.py:6608-6620), broadcastable to [B,H,S,M].
    ``masking`` = dict(base_mask_prob, entropy_target, min_active) or None.
    ``storage``: if set (e.g. torch.bfloat16) the intermediates the CUDA path
    writes to HBM (projected K/V, context, output) are rounded to that dtype while
    all arithmetic stays in ``query.dtype`` -- the stage-exact model of the bf16 path.
    ``fold_key`` (stage model of the CUDA path's folded key projection, single shared query only): the
    scores are associated as x . (scale * Wk_h^T q_h) with that per-head vector rounded to ``storage``
    and the key bias dropped (it shifts every token of a head alike, so the softmax does not see it);
    mathematically identical to the reference's (x Wk^T + bk) . (scale q_h), the rounding differs.
    ``per_row_query_storage``: with per-row queries the CUDA path keeps the projected queries (and, in the backward,
    their gradients) in ``storage`` too; the one shared fusion query of the hot path stays fp32.
    """
    if value is None:
        value = key
    B, S, D = query.shape
    M = key.shape[1]
    H = num_heads
    hd = D // H
    Wq, Wk, Wv = in_proj_weight[:D], in_proj_weight[D:2 * D], in_proj_weight[2 * D:]
    if in_proj_bias is None:
        bq = bk = bv = None
    else:
        bq, bk, bv = in_proj_bias[:D], in_proj_bias[D:2 * D], in_proj_bias[2 * D:]

    lin = torch.nn.functional.linear
    qp = lin(query, Wq, bq)                                      # functional.py:5854
    if per_row_query_storage:
        qp = _round(qp, storage)
    k = _round(lin(key, Wk, bk), storage)                        # :5855 (K half)
    v = _round(lin(value, Wv, bv), storage)                      # :5855 (V half)

    qh = qp.view(B, S, H, hd).transpose(1, 2)                    # [B,H,S,hd]  (:6554)
    kh = k.view(B, M, H, hd).transpose(1, 2)                     # [B,H,M,hd]
    vh = v.view(B, M, H, hd).transpose(1, 2)
    q_scaled = qh * math.sqrt(1.0 / float(hd))                   # :6632
    scores = q_scaled @ kh.transpose(-2, -1)                     # :6642   [B,H,S,M]
    if fold_key:
        assert S == 1, "the folded association needs one query per sample"
        scale = math.sqrt(1.0 / float(hd))
        qk = torch.einsum("he,hed->hd", qp[0, 0].view(H, hd), Wk.view(H, hd, D)) * scale   # [H, D]
        qk = _round(qk, storage)
        scores = torch.einsum("bmd,hd->bhm", key, qk).unsqueeze(2)                       # [B,H,1,M]
    if score_bias is not None:
        scores = scores + score_bias                             # :6638 baddbmm
    w = torch.softmax(scores, dim=-1)                            # :6643
    if training and dropout_p > 0.0:                             # :6645
        if dropout_p >= 1.0:
            keep = torch.zeros_like(w)
            wd = w * 0.0
        else:
            keep = (u_drop.view(B, H, S, M).to(w.dtype) >= dropout_p).to(w.dtype)
            wd = w * keep / (1.0 - dropout_p)
    else:
        keep = torch.ones_like(w)
        wd = w
    ctx = (wd @ vh).transpose(1, 2).reshape(B, S, D)             # :6647-6652
    ctx = _round(ctx, storage)
    out = _round(lin(ctx, out_proj_weight, out_proj_bias), storage)   # :6653
    pooled = wd.mean(dim=1)                                      # :6657-6659  [B,S,M]

    res = PoolResult(out=out, pooled=pooled)
    res.saved = dict(qp=qp, k=k, v=v, w=w, wd=wd, keep=keep, ctx=ctx)
    res.info["attention_weights"] = pooled                       # AECFLayer.py:538
    if masking is not None:
        cm = curriculum_mask(pooled, None if u_mask is None else u_mask.view(B, S, M),
                             training=training, **masking)       # :534
        for name in ("entropy", "mask_rate", "target_entropy"):
            if name in cm:
                res.info[name] = cm[name]
        res.info["masked_attention_weights"] = cm["masked"].detach()      # :541
        res.info["mask"] = cm["mask"]
        if "keep_prob" in cm:
            res.info["keep_prob"] = cm["keep_prob"]
    return res


def pool_backward(query: Tensor, key: Tensor, value: Optional[Tensor],
                  in_proj_weight: Tensor, out_proj_weight: Tensor, num_heads: int,
                  saved: Dict[str, Tensor], grad_out: Tensor, *,
                  grad_pooled: Optional[Tensor] = None, grad_entropy: Optional[Tensor] = None,
                  dropout_p: float = 0.0, training: bool = True, has_bias: bool = True,
                  storage: Optional[torch.dtype] = None, fold_key: bool = False,
                  per_row_query_storage: bool = False) -> Dict[str, Tensor]:
    """Closed-form backward of pool_forward (SURVEY.md Appendix B).

    The reference has no backward source: it is autograd over
    torch/nn/functional.py:5847-5865, 6630-6659.  tests/test_oracle_golden.py
    checks this against autograd of the reference itself.
    Covers S >= 1 fusion queries per sample (S == 1 is the hot path): dK and dV sum over the queries of a sample.
    ``fold_key``: the association the CUDA path's folded key projection uses (one shared query): dK is never
    formed; with ds the score gradient, Qk[h] = scale * Wk_h^T q_h and R[h] = sum_{b,m} ds[b,h,m] x[b,m],
        dX   = dV Wv + ds Qk            dWk[h*hd + j] = scale * q[h*hd + j] * R[h]
        d q[h*hd + j] = scale * Wk[h*hd + j] . R[h]        (the bk * sum ds term is analytically zero and dropped)
    Same mathematics as autograd of the reference, re-associated; tests/test_oracle_golden.py checks it against
    the reference's own gradients.
    """
    if value is None:
        value = key
    B, S, D = query.shape
    M = key.shape[1]
    H = num_heads
    hd = D // H
    scale = math.sqrt(1.0 / float(hd))
    Wq, Wk, Wv = in_proj_weight[:D], in_proj_weight[D:2 * D], in_proj_weight[2 * D:]
    w, wd, keep = saved["w"], saved["wd"], saved["keep"]              # [B,H,S,M]
    qp = saved["qp"].reshape(B, S, H, hd)
    kh = saved["k"].view(B, M, H, hd)
    vh = saved["v"].view(B, M, H, hd)
    ctx = saved["ctx"].reshape(B * S, D)
    g = grad_out.reshape(B * S, D)

    d_wo = g.t() @ ctx
    d_bo = g.sum(0)
    d_ctx = _round(g @ out_proj_weight, storage).view(B, S, H, hd)
    d_wd = torch.einsum("bshe,bmhe->bhsm", d_ctx, vh)
    d_pooled = None if grad_pooled is None else grad_pooled.reshape(B, S, M)
    if grad_entropy is not None:
        # eval mode only: entropy = clamp(-sum xlogy(p, p), 0, log M) stays attached
        # (reference aecf/AECFLayer.py:151-156).  Autograd's chain term by term: the clamp passes the gradient inside
        # its range and 0 outside; xlogy(p, p) contributes xlogy(p != 0, p) + p / p, which is 0 / 0 = NaN at p = 0
        # whatever the clamp passed.
        pooled = wd.mean(dim=1)                                       # [B,S,M]
        raw = -torch.xlogy(pooled, pooled).sum(-1, keepdim=True)
        inside = (raw >= 0.0) & (raw <= math.log(M))
        g_raw = torch.where(inside, grad_entropy.reshape(B, S, 1), torch.zeros((), dtype=pooled.dtype))
        d_h = -g_raw * (torch.xlogy((pooled != 0).to(pooled.dtype), pooled) + pooled / pooled)
        d_pooled = d_h if d_pooled is None else d_pooled + d_h
    if d_pooled is not None:
        d_wd = d_wd + d_pooled.reshape(B, 1, S, M) / H
    d_v = torch.einsum("bhsm,bshe->bmhe", wd, d_ctx)
    if training and dropout_p > 0.0:
        d_w = d_wd * keep * (0.0 if dropout_p >= 1.0 else 1.0 / (1.0 - dropout_p))
    else:
        d_w = d_wd
    d_s = w * (d_w - (w * d_w).sum(-1, keepdim=True))
    if fold_key:
        assert S == 1, "the folded association needs one query per sample"
        return _folded_input_grads(query, key, in_proj_weight, saved, d_s[:, :, 0], d_v, d_wo, d_bo, scale, H,
                                   has_bias, storage)
    d_qh = scale * torch.einsum("bhsm,bmhe->bshe", d_s, kh)
    d_k = scale * torch.einsum("bhsm,bshe->bmhe", d_s, qp)
    d_k = _round(d_k.reshape(B, M, D), storage)
    d_v = _round(d_v.reshape(B, M, D), storage)
    d_qp = d_qh.reshape(B * S, D)
    if per_row_query_storage:
        d_qp = _round(d_qp, storage)

    grads = {
        "out_proj.weight": d_wo, "out_proj.bias": d_bo,
        "key": d_k @ Wk, "value": d_v @ Wv,
        "query": (d_qp @ Wq).view(B, S, D),
    }
    if value is key:
        grads["key"] = grads["key"] + grads.pop("value")
    x_q = query.reshape(B * S, D)
    d_wq = d_qp.t() @ x_q
    d_wk = d_k.reshape(B * M, D).t() @ key.reshape(B * M, D)
    d_wv = d_v.reshape(B * M, D).t() @ value.reshape(B * M, D)
    grads["in_proj_weight"] = torch.cat([d_wq, d_wk, d_wv], 0)
    if has_bias:
        grads["in_proj_bias"] = torch.cat([d_qp.sum(0), d_k.sum((0, 1)), d_v.sum((0, 1))], 0)
    return grads


def _folded_input_grads(query, key, in_proj_weight, saved, d_s, d_v, d_wo, d_bo, scale, H, has_bias, storage):
    """Input / in-projection gradients of pool_backward in the folded association (see its docstring)."""
    B, _, D = query.shape
    M = key.shape[1]
    hd = D // H
    Wq, Wk, Wv = in_proj_weight[:D], in_proj_weight[D:2 * D], in_proj_weight[2 * D:]
    q0 = saved["qp"][0, 0]                                         # the one projected query, [D]
    qk = _round(torch.einsum("he,hed->hd", q0.view(H, hd), Wk.view(H, hd, D)) * scale, storage)     # [H, D]
    d_s = _round(d_s, storage)                                     # stored next to dV in the storage dtype
    d_v = _round(d_v.reshape(B, M, D), storage)
    x = key.reshape(B * M, D)
    r = torch.einsum("bhm,bmd->hd", d_s, key)                      # R[h] = sum ds x
    d_wk = (scale * q0).view(H, hd, 1) * r.view(H, 1, D)           # [H, hd, D]
    d_q0 = scale * torch.einsum("hed,hd->he", Wk.view(H, hd, D), r).reshape(D)
    d_wq = torch.outer(d_q0, query[0, 0])
    d_wv = d_v.reshape(B * M, D).t() @ x
    grads = {
        "out_proj.weight": d_wo, "out_proj.bias": d_bo,
        "key": d_v @ Wv + torch.einsum("bhm,hd->bmd", d_s, qk),
        # the caller sums the per-row query gradient over the batch: put the whole (already reduced) gradient in row 0
        "query": torch.cat([(d_q0 @ Wq).view(1, 1, D), torch.zeros(B - 1, 1, D, dtype=query.dtype)], 0),
        "in_proj_weight": torch.cat([d_wq, d_wk.reshape(D, D), d_wv], 0),
    }
    if has_bias:
        d_bk = (scale * q0).view(H, hd) * d_s.sum((0, 2)).view(H, 1)
        grads["in_proj_bias"] = torch.cat([d_q0, d_bk.reshape(D), d_v.sum((0, 1))], 0)
    return grads


# ----------------------------------------------------------------------------
# Projection-free fast path of the functional API
# ----------------------------------------------------------------------------

def sdpa_single_head(query: Tensor, key: Tensor, value: Tensor) -> Tensor:
    """softmax(Q K^T / sqrt(D)) V -- reference aecf/AECFLayer.py:573-581."""
    scores = torch.bmm(query, key.transpose(-2, -1)) * (query.size(-1) ** -0.5)
    return torch.bmm(torch.softmax(scores, dim=-1), value)


# ----------------------------------------------------------------------------
# A whole training step, used as the timed CPU baseline ("port")
# ----------------------------------------------------------------------------

def training_step(query0: Tensor, x: Tensor, params: Dict[str, Tensor], num_heads: int, *,
                  u_mask: Tensor, masking: dict, last_seq_len: Optional[int] = None,
                  loss_weight: float = 0.01) -> Dict[str, Tensor]:
    """forward(return_info) + entropy_loss + closed-form backward of
    ``out.pow(2).mean() + loss_weight * entropy_loss`` (SURVEY.md section 8d step).

    In training mode the entropy term carries no gradient (reference :278), so the
    upstream gradient is 2*out/numel.
    """
    B, M, D = x.shape
    q = query0.expand(B, 1, D)
    fwd = pool_forward(q, x, None, params["in_proj_weight"], params["in_proj_bias"],
                       params["out_proj.weight"], params["out_proj.bias"], num_heads,
                       training=True, u_mask=u_mask, masking=masking)
    ent = entropy_loss(fwd.info["entropy"], M if last_seq_len is None else last_seq_len,
                       masking.get("entropy_target", 0.7))
    loss = fwd.out.pow(2).mean() + loss_weight * ent
    g = 2.0 * fwd.out / fwd.out.numel()
    grads = pool_backward(q, x, None, params["in_proj_weight"], params["out_proj.weight"],
                          num_heads, fwd.saved, g)
    grads["query0"] = grads.pop("query").sum(0, keepdim=True)
    return {"loss": loss, "out": fwd.out, "grads": grads, "info": fwd.info}
