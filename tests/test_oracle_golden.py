"""Pin the oracle: every function of oracle/aecf_oracle.py against the reference's own outputs
(tests/golden/*.npz, written by tests/golden/make_golden.py from the reference checkout that AECF_REFERENCE names)."""
import math

import numpy as np
import pytest
import torch

from oracle import aecf_oracle as oracle
from oracle import philox
from tests.golden.cases import CASES, MULTI_QUERY_CASES, build_inputs, masking_kwargs
from tests.helpers import assert_close, finite_scale, load_golden, run_oracle


def _tol(case):
    return 1e-12 if case.dtype == "float64" else 2e-6


@pytest.mark.parametrize("case", CASES + MULTI_QUERY_CASES, ids=lambda c: c.name)
def test_forward_matches_reference(case):
    g = load_golden(case)
    fwd, _ = run_oracle(case)
    tol = _tol(case)
    assert_close("out", fwd.out, g["out"], tol)
    assert_close("attention_weights", fwd.info["attention_weights"], g["attention_weights"], tol)
    assert_close("entropy", fwd.info["entropy"], g["entropy"], tol, atol=tol)
    # mask-derived outputs are exact: same draws, same threshold arithmetic
    assert np.array_equal(fwd.info["mask_rate"].numpy(), g["mask_rate"])
    ref_mask = g["masked_attention_weights"] > 0
    got = fwd.info["masked_attention_weights"].numpy()
    if case.training and case.M > 1:
        # a kept token whose weight is exactly 0 (padded key) also shows 0 in the reference output
        live = g["attention_weights"] > 0
        assert np.array_equal((fwd.info["mask"].numpy() > 0) & live, ref_mask)
    assert_close("masked_attention_weights", got, g["masked_attention_weights"], tol, atol=tol)
    if "target_entropy" in g:
        assert_close("target_entropy", fwd.info["target_entropy"], g["target_entropy"], tol, atol=tol)
    else:
        assert "target_entropy" not in fwd.info                  # eval mode: key absent (:153-156)
    last = case.M if (case.training and case.M > 1) else 2       # _last_seq_len side effect (:99, :187)
    assert int(g["last_seq_len"]) == last
    assert_close("entropy_loss", oracle.entropy_loss(fwd.info["entropy"], last, case.entropy_target),
                 g["entropy_loss"], tol, atol=tol)


FOLDABLE = [c for c in CASES if not c.separate_value]


@pytest.mark.parametrize("case", FOLDABLE, ids=lambda c: c.name)
def test_folded_key_projection_matches_reference(case):
    """The association the CUDA path's folded key projection uses (scores = x . (scale Wk_h^T q_h), rank-H key-side
    gradients through R = sum ds x) against the reference's own outputs and autograd gradients: identical masks,
    everything else to rounding."""
    g = load_golden(case)
    fwd, grads = run_oracle(case, fold_key=True)
    f64 = case.dtype == "float64"
    tol, gtol = (1e-11, 1e-10) if f64 else (1e-5, 3e-5)
    assert_close("out", fwd.out, g["out"], tol)
    assert_close("attention_weights", fwd.info["attention_weights"], g["attention_weights"], tol, atol=tol)
    assert_close("entropy", fwd.info["entropy"], g["entropy"], tol, atol=tol)
    assert np.array_equal(fwd.info["mask_rate"].numpy(), g["mask_rate"])
    if case.training and case.M > 1:
        live = g["attention_weights"] > 0
        assert np.array_equal((fwd.info["mask"].numpy() > 0) & live, g["masked_attention_weights"] > 0)
    assert_close("grad_x", grads["key"], g["grad_x"], gtol)
    assert_close("grad_query0", grads["query0"], g["grad_query0"], gtol)
    scale = float(np.abs(g["grad_in_proj_bias"]).max())
    assert_close("grad_in_proj_bias", grads["in_proj_bias"], g["grad_in_proj_bias"], gtol, atol=gtol * scale)
    if case.full_grads:
        assert_close("grad_in_proj_weight", grads["in_proj_weight"], g["grad_in_proj_weight"], gtol)
    else:
        assert_close("grad_in_proj_weight_rowsum", grads["in_proj_weight"].sum(1), g["grad_in_proj_weight_rowsum"], gtol)


@pytest.mark.parametrize("case", CASES + MULTI_QUERY_CASES, ids=lambda c: c.name)
def test_backward_matches_reference_autograd(case):
    g = load_golden(case)
    _, grads = run_oracle(case)
    tol = 1e-11 if case.dtype == "float64" else 2e-5
    assert_close("grad_x", grads["key"], g["grad_x"], tol)
    if case.separate_value:
        assert_close("grad_value", grads["value"], g["grad_value"], tol)
    if case.S > 1:
        assert_close("grad_query", grads["query"], g["grad_query"], tol)
    else:
        assert_close("grad_query0", grads["query0"], g["grad_query0"], tol)
    assert_close("grad_out_proj_bias", grads["out_proj.bias"], g["grad_out_proj_bias"], tol)
    # the K-bias gradient is analytically zero (softmax shift invariance): compare on the V/Q scale
    scale = finite_scale(g["grad_in_proj_bias"])
    assert_close("grad_in_proj_bias", grads["in_proj_bias"], g["grad_in_proj_bias"], tol, atol=tol * scale)
    for name, key in (("in_proj_weight", "in_proj_weight"), ("out_proj_weight", "out_proj.weight")):
        got = grads[key]
        if case.full_grads:
            assert_close(f"grad_{name}", got, g[f"grad_{name}"], tol)
        else:
            assert_close(f"grad_{name}_rowsum", got.sum(1), g[f"grad_{name}_rowsum"], tol)
            assert_close(f"grad_{name}_colsum", got.sum(0), g[f"grad_{name}_colsum"], tol)
            assert_close(f"grad_{name}_strided", got.flatten()[::97], g[f"grad_{name}_strided"], tol)


def test_topk_onehot_matches_torch_topk():
    """Tie rule.  torch's CPU topk (ATen TopKImpl.h: std::nth_element for these sizes) is stable
    only up to 3 entries (libstdc++ falls to insertion sort); for L >= 4 its pick among EXACT ties
    is an artefact of introselect and differs again on CUDA (radix select).  The contract here is
    lowest index: identical to the reference for L <= 3 and for tie-free rows of any L, and for
    tied rows with L >= 4 the selected VALUES are identical (only which twin is picked differs)."""
    torch.manual_seed(0)
    for L in range(2, 9):
        w = torch.softmax(torch.randn(500, L), -1)
        tied = torch.zeros(500, dtype=torch.bool)
        w[::7] = 1.0 / L                                  # exact ties
        tied[::7] = True
        w[1::11, : L // 2] = w[1::11, L // 2: 2 * (L // 2)]  # partial ties
        tied[1::11] = True
        for k in range(1, L + 1):
            idx = w.topk(k, dim=-1).indices
            want = torch.zeros_like(w).scatter_(-1, idx, 1.0)
            got = oracle.topk_onehot(w, k)
            assert (got.sum(-1) == k).all()
            exact = torch.ones(500, dtype=torch.bool) if L <= 3 else ~tied
            assert torch.equal(got[exact], want[exact]), (L, k)
            assert torch.equal((got * w).sort(-1).values, (want * w).sort(-1).values), (L, k)


def test_readme_validation_snippet():
    """reference README.md:300-317: masking returns the three info keys and finite output."""
    u = torch.from_numpy(philox.mask_uniforms(1, 0, 0, 100, 8))
    w = torch.softmax(torch.from_numpy(philox.normal(3, (100, 8))).float(), -1)
    r = oracle.curriculum_mask(w, u)
    assert {"entropy", "mask_rate", "target_entropy"} <= set(r)
    edge = torch.tensor([[1.0, 0.0, 0.0], [0.33, 0.33, 0.34]])
    r = oracle.curriculum_mask(edge, torch.full((2, 3), 0.5))
    assert torch.isfinite(r["masked"]).all()
    assert torch.allclose(r["masked"].sum(-1), torch.ones(2))


def test_masking_properties():
    for M in (2, 3, 5, 8):
        for min_active in (1, 2, 9):
            u = torch.from_numpy(philox.mask_uniforms(5, M, 0, 4096, M))
            w = torch.softmax(3 * torch.from_numpy(philox.normal(M, (4096, M))).float(), -1)
            r = oracle.curriculum_mask(w, u, base_mask_prob=1.0, min_active=min_active)
            assert (r["mask"].sum(-1) >= min(min_active, M)).all()
            assert torch.allclose(r["masked"].sum(-1), torch.ones(4096), atol=1e-6)
            assert (r["entropy"] >= 0).all() and (r["entropy"] <= math.log(M) + 1e-6).all()


def test_masking_scrubs_non_finite_rows():
    w = torch.tensor([[float("nan"), 0.5, 0.5], [float("inf"), 0.0, 0.0], [0.0, 0.0, 0.0]])
    r = oracle.curriculum_mask(w, torch.full((3, 3), 0.5))
    assert torch.isfinite(r["masked"]).all()
    assert torch.allclose(r["renormalised"][2], torch.full((3,), 1 / 3))


def test_sdpa_fast_path():
    q = torch.from_numpy(philox.normal(1, (4, 2, 16))).float()
    k = torch.from_numpy(philox.normal(2, (4, 5, 16))).float()
    out = oracle.sdpa_single_head(q, k, k)
    want = torch.nn.functional.scaled_dot_product_attention(q, k, k)
    assert torch.allclose(out, want, atol=1e-6)


def test_stage_rounded_oracle_stays_close_to_fp32():
    """The bf16 storage model perturbs outputs well inside the 2e-2 budget of north_star."""
    case = CASES[1]
    inp = build_inputs(case)
    for k in ("in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias", "query0", "x", "grad_out"):
        inp[k] = inp[k].bfloat16().float()
    ref, _ = run_oracle(case, inp)
    got, _ = run_oracle(case, inp, storage=torch.bfloat16)
    assert_close("out", got.out, ref.out, 2e-2)


@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("name,S", [("d64_h4_m4_kpm", 1), ("s2_d64_h4_m4_kpm_eval", 2)])
def test_fully_padded_samples_match_torch_autograd(name, S, training):
    """The NaN pattern of the oracle on fully padded samples (and, in eval mode, the entropy gradient at the padded
    tokens' zero weights) is torch's own: autograd through torch.nn.functional.multi_head_attention_forward and the
    oracle's masking stage, in fp64."""
    import dataclasses

    from tests.golden.cases import CASES_BY_NAME
    case = dataclasses.replace(CASES_BY_NAME[name], training=training, dropout=0.0, pooled_grad=True, name=name + "_pad")
    inp = build_inputs(case, torch.float64)
    padded = [0, 5, case.B - 1]
    inp["key_padding_mask"][padded, :] = True
    ref, ref_grads = run_oracle(case, inp)

    B, M, D = case.B, case.M, case.D
    leaf = {k: inp[k].clone().requires_grad_(True)
            for k in ("in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias", "x", "query" if S > 1 else "query0")}
    q = leaf["query"] if S > 1 else leaf["query0"].expand(B, 1, D)
    x = leaf["x"]
    out, pooled = torch.nn.functional.multi_head_attention_forward(
        q.transpose(0, 1), x.transpose(0, 1), x.transpose(0, 1), D, case.H, leaf["in_proj_weight"], leaf["in_proj_bias"],
        None, None, False, 0.0, leaf["out_proj.weight"], leaf["out_proj.bias"], training=training,
        key_padding_mask=inp["key_padding_mask"], need_weights=True, average_attn_weights=True)
    out = out.transpose(0, 1)
    cm = oracle.curriculum_mask(pooled, inp["u_mask"].reshape(pooled.shape), training=training, **masking_kwargs(case))
    loss = (out * inp["grad_out"].reshape(out.shape)).sum() + (pooled * inp["grad_pooled"].reshape(pooled.shape)).sum()
    if not training:
        loss = loss + 0.5 * cm["entropy"].sum()
    loss.backward()
    assert bool(torch.isnan(out[padded]).all())
    assert_close("out", ref.out, out.detach(), 1e-12)
    assert_close("attention_weights", ref.info["attention_weights"], pooled.detach(), 1e-12)
    assert_close("entropy", ref.info["entropy"], cm["entropy"].detach(), 1e-12, atol=1e-12)
    assert_close("mask_rate", ref.info["mask_rate"], cm["mask_rate"], 0.0, atol=0.0)
    for name_g, key in (("key", "x"), ("in_proj_weight", "in_proj_weight"), ("in_proj_bias", "in_proj_bias"),
                        ("out_proj.weight", "out_proj.weight"), ("out_proj.bias", "out_proj.bias")):
        assert_close(f"grad {name_g}", ref_grads[name_g], leaf[key].grad, 1e-10)
    if S > 1:
        assert_close("grad query", ref_grads["query"], leaf["query"].grad, 1e-10)
    else:
        assert_close("grad query0", ref_grads["query0"], leaf["query0"].grad, 1e-10)
    assert bool(torch.isnan(ref_grads["in_proj_weight"]).all())          # a padded sample reaches every batch sum
