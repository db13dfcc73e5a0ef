"""Several fusion queries per sample (target length S > 1; csrc/pool_multi.cuh) against the oracle and the
reference's own outputs (tests/golden/s*.npz).
"""
import os

import numpy as np
import pytest
import torch

import aecf_b200
from oracle import aecf_oracle as oracle
from tests.golden.cases import MULTI_QUERY_CASES, PHILOX_SEED, Case, build_inputs, masking_kwargs
from tests.helpers import assert_close, finite_scale, load_golden, run_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FP32_TOL = 1e-5
BF16_TOL = 2e-2


def expected_bits(mask: torch.Tensor) -> np.ndarray:
    m = (mask.reshape(-1, mask.shape[-1]) > 0).numpy().astype(np.int64)
    return (m * (1 << np.arange(m.shape[1]))).sum(1).astype(np.uint8)


def run_cuda(case: Case, inp: dict, dtype: torch.dtype, batch_first: bool = True, rows=None, attn_mask=None):
    """Forward + backward through the public API.  ``rows``: (first, count) runs that shard of the batch with
    ``row_offset`` set, as a data-parallel rank would."""
    first, count = rows if rows is not None else (0, case.B)
    sl = slice(first, first + count)
    cm = aecf_b200.CurriculumMasking(**masking_kwargs(case))
    pool = aecf_b200.MultimodalAttentionPool(case.D, num_heads=case.H, dropout=case.dropout, curriculum_masking=cm,
                                             batch_first=batch_first, device=DEV, dtype=dtype)
    with torch.no_grad():
        pool.attention.in_proj_weight.copy_(inp["in_proj_weight"])
        pool.attention.in_proj_bias.copy_(inp["in_proj_bias"])
        pool.attention.out_proj.weight.copy_(inp["out_proj.weight"])
        pool.attention.out_proj.bias.copy_(inp["out_proj.bias"])
    pool.train(case.training)
    pool.row_offset = case.row0 + first
    pool._want_mask_bits = True
    query = inp["query"][sl].to(DEV, dtype)
    x = inp["x"][sl].to(DEV, dtype)
    if not batch_first:
        query, x = query.transpose(0, 1).contiguous(), x.transpose(0, 1).contiguous()
    query.requires_grad_(True)
    x.requires_grad_(True)
    kpm = inp["key_padding_mask"][sl].to(DEV) if case.kpm else None
    aecf_b200.set_rng_state(PHILOX_SEED, case.offset)
    try:
        out, info = pool(query, x, key_padding_mask=kpm, attn_mask=attn_mask, return_info=True)
        ent_loss = cm.entropy_loss(info["entropy"])
    finally:
        aecf_b200.set_rng_state(None)
    g_out = inp["grad_out"][sl].to(DEV)
    loss = (out.float() * (g_out if batch_first else g_out.transpose(0, 1))).sum()
    if case.pooled_grad:
        loss = loss + (info["attention_weights"] * inp["grad_pooled"][sl].to(DEV)).sum()
    if not case.training:
        loss = loss + 0.5 * info["entropy"].sum()
    loss.backward()
    torch.cuda.synchronize()
    to_bf = (lambda t: t) if batch_first else (lambda t: t.transpose(0, 1))
    grads = {
        "key": to_bf(x.grad), "query": to_bf(query.grad),
        "in_proj_weight": pool.attention.in_proj_weight.grad, "in_proj_bias": pool.attention.in_proj_bias.grad,
        "out_proj.weight": pool.attention.out_proj.weight.grad, "out_proj.bias": pool.attention.out_proj.bias.grad,
    }
    return to_bf(out), info, ent_loss, grads, cm


def check_against_oracle(case, out, info, ent_loss, grads, ref, ref_grads, tol, exact_masks=True):
    B, S, M = case.B, case.S, case.M
    assert out.shape == (B, S, case.D)
    assert info["attention_weights"].shape == (B, S, M) and info["entropy"].shape == (B, S)
    assert info["mask_rate"].shape == (B, S) and info["masked_attention_weights"].shape == (B, S, M)
    assert_close("out", out.float().cpu(), ref.out, tol)
    assert_close("attention_weights", info["attention_weights"].cpu(), ref.info["attention_weights"], tol, atol=tol)
    assert_close("entropy", info["entropy"].cpu(), ref.info["entropy"], tol, atol=tol * max(float(np.log(max(M, 2))), 1.0))
    if exact_masks:
        assert np.array_equal(info["mask_bits"].cpu().numpy().reshape(-1), expected_bits(ref.info["mask"])), "mask bits differ"
        assert torch.equal(info["mask_rate"].cpu(), ref.info["mask_rate"].float()), "mask_rate differs"
    assert_close("masked_attention_weights", info["masked_attention_weights"].cpu(),
                 ref.info["masked_attention_weights"], tol, atol=tol)
    last = M if (case.training and M > 1) else 2
    assert_close("entropy_loss", ent_loss.cpu(), oracle.entropy_loss(ref.info["entropy"], last, case.entropy_target), tol, atol=tol)
    for name in ("key", "query", "out_proj.bias", "out_proj.weight", "in_proj_weight"):
        assert_close(f"grad {name}", grads[name].float().cpu(), ref_grads[name], tol)
    scale = finite_scale(ref_grads["in_proj_bias"])        # the K-bias third is analytically zero
    assert_close("grad in_proj_bias", grads["in_proj_bias"].float().cpu(), ref_grads["in_proj_bias"], tol, atol=tol * scale)


@pytest.mark.parametrize("batch_first", [True, False], ids=["batch_first", "seq_first"])
@pytest.mark.parametrize("case", MULTI_QUERY_CASES, ids=lambda c: c.name)
def test_fp32_matches_oracle(case, batch_first):
    inp = build_inputs(case)
    ref, ref_grads = run_oracle(case, inp)
    out, info, ent_loss, grads, cm = run_cuda(case, inp, torch.float32, batch_first=batch_first)
    assert cm._last_seq_len == (case.M if (case.training and case.M > 1) else 2)
    check_against_oracle(case, out, info, ent_loss, grads, ref, ref_grads, FP32_TOL)


@pytest.mark.parametrize("case", MULTI_QUERY_CASES, ids=lambda c: c.name)
def test_fp32_matches_reference_golden(case):
    """Directly against what the unmodified reference produced on the same inputs and draws."""
    g = load_golden(case)
    out, info, ent_loss, grads, _ = run_cuda(case, build_inputs(case), torch.float32)
    tol = 2e-5
    assert_close("out", out.cpu(), g["out"], tol)
    assert_close("attention_weights", info["attention_weights"].cpu(), g["attention_weights"], tol, atol=tol)
    assert_close("entropy", info["entropy"].cpu(), g["entropy"], tol, atol=tol)
    assert np.array_equal(info["mask_rate"].cpu().numpy(), g["mask_rate"])
    assert_close("masked_attention_weights", info["masked_attention_weights"].cpu(), g["masked_attention_weights"], tol, atol=tol)
    assert_close("entropy_loss", ent_loss.cpu(), g["entropy_loss"], tol, atol=tol)
    assert_close("grad_x", grads["key"].cpu(), g["grad_x"], tol)
    assert_close("grad_query", grads["query"].cpu(), g["grad_query"], tol)
    assert_close("grad_out_proj_bias", grads["out_proj.bias"].cpu(), g["grad_out_proj_bias"], tol)
    scale = finite_scale(g["grad_in_proj_bias"])
    assert_close("grad_in_proj_bias", grads["in_proj_bias"].cpu(), g["grad_in_proj_bias"], tol, atol=tol * scale)
    if case.full_grads:
        assert_close("grad_in_proj_weight", grads["in_proj_weight"].cpu(), g["grad_in_proj_weight"], tol)
        assert_close("grad_out_proj_weight", grads["out_proj.weight"].cpu(), g["grad_out_proj_weight"], tol)
    else:
        assert_close("grad_in_proj_weight_rowsum", grads["in_proj_weight"].cpu().sum(1), g["grad_in_proj_weight_rowsum"], tol)
        assert_close("grad_out_proj_weight_rowsum", grads["out_proj.weight"].cpu().sum(1), g["grad_out_proj_weight_rowsum"], tol)


@pytest.mark.parametrize("case", MULTI_QUERY_CASES, ids=lambda c: c.name)
def test_bf16_masks_exact_against_stage_rounded_oracle(case):
    """bf16 storage: against the oracle that rounds K/V, ctx and out where the CUDA path stores them."""
    inp = build_inputs(case)
    for k in ("in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias", "query", "x", "grad_out"):
        inp[k] = inp[k].bfloat16().float()
    ref, ref_grads = run_oracle(case, inp, storage=torch.bfloat16)
    out, info, ent_loss, grads, _ = run_cuda(case, inp, torch.bfloat16)
    assert np.array_equal(info["mask_bits"].cpu().numpy().reshape(-1), expected_bits(ref.info["mask"])), "mask bits differ"
    assert torch.equal(info["mask_rate"].cpu(), ref.info["mask_rate"].float())
    assert_close("attention_weights", info["attention_weights"].cpu(), ref.info["attention_weights"], 1e-4, atol=1e-5)
    assert_close("entropy", info["entropy"].cpu(), ref.info["entropy"], 1e-4, atol=1e-5)
    assert_close("out", out.float().cpu(), ref.out, 1e-2)
    for name in ("key", "query", "in_proj_weight", "out_proj.weight"):
        assert_close(f"grad {name}", grads[name].float().cpu(), ref_grads[name], BF16_TOL)


def test_batch_shards_reproduce_the_full_batch():
    """Rows (b, s) draw from Philox row (row0 + b) * S + s: two half batches with row_offset reproduce the masks of
    the full batch bit for bit and their parameter gradients add up to it."""
    case = MULTI_QUERY_CASES[0]
    inp = build_inputs(case)
    out, info, _, grads, _ = run_cuda(case, inp, torch.float32)
    half = case.B // 2
    parts = [run_cuda(case, inp, torch.float32, rows=(0, half)), run_cuda(case, inp, torch.float32, rows=(half, case.B - half))]
    assert torch.equal(torch.cat([p[0] for p in parts]), out)
    for key in ("mask_bits", "entropy", "attention_weights", "masked_attention_weights"):
        assert torch.equal(torch.cat([p[1][key] for p in parts]), info[key]), key
    assert torch.equal(torch.cat([p[3]["key"] for p in parts]), grads["key"])
    for name in ("in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias"):
        assert_close(name, (parts[0][3][name] + parts[1][3][name]).cpu(), grads[name].cpu(), 1e-5)


def test_attn_mask_per_query():
    """A 2D [S, M] additive attn_mask and the 3D [B*H, S, M] form (torch/nn/functional.py:6608-6620)."""
    case = MULTI_QUERY_CASES[0]
    inp = build_inputs(case)
    B, S, M, H = case.B, case.S, case.M, case.H
    am2 = torch.zeros(S, M)
    am2[0, 1] = float("-inf")
    am2[1, 2] = -1.5
    q, x = inp["query"], inp["x"]
    for am in (am2, am2.view(1, S, M).expand(B * H, S, M).contiguous()):
        bias = am2.view(1, 1, S, M)
        ref = oracle.pool_forward(q, x, None, inp["in_proj_weight"], inp["in_proj_bias"], inp["out_proj.weight"],
                                  inp["out_proj.bias"], H, dropout_p=case.dropout, training=True, u_drop=inp["u_drop"],
                                  u_mask=inp["u_mask"], score_bias=bias, masking=masking_kwargs(case))
        out, info, _, _, _ = run_cuda(case, inp, torch.float32, attn_mask=am.to(DEV))
        assert_close("out", out.cpu(), ref.out, FP32_TOL)
        assert_close("attention_weights", info["attention_weights"].cpu(), ref.info["attention_weights"], FP32_TOL, atol=FP32_TOL)
        assert np.array_equal(info["mask_bits"].cpu().numpy().reshape(-1), expected_bits(ref.info["mask"]))
        assert float(info["attention_weights"][:, 0, 1].abs().max()) == 0.0
