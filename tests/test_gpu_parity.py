"""Parity of the CUDA path (through the public module API -> C ABI) with the oracle and with the
reference's own outputs (tests/golden).  Run on the B200 box:  pytest tests -m gpu

Tolerances (BASELINE.json north_star): fp32 1e-5 relative, bf16 2e-2 relative, masks and the
active-token set bit-exact.
"""
import json
import math

import numpy as np
import pytest
import torch

import aecf_b200
from aecf_b200 import _lib, ops
from oracle import aecf_oracle as oracle
from oracle import philox
from tests.golden.cases import CASES, CASES_BY_NAME, PHILOX_SEED, Case, build_inputs, masking_kwargs
from tests.helpers import assert_close, finite_scale, load_golden, run_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FP32_TOL = 1e-5
BF16_TOL = 2e-2


def make_pool(case: Case, inp: dict, dtype: torch.dtype, fold=None):
    """fold: None = the module's automatic choice (folded key projection for bf16 with a shared query), True/False
    force it on (wherever it applies) / off."""
    cm = aecf_b200.CurriculumMasking(**masking_kwargs(case))
    pool = aecf_b200.MultimodalAttentionPool(case.D, num_heads=case.H, dropout=case.dropout,
                                             curriculum_masking=cm, device=DEV, dtype=dtype)
    with torch.no_grad():
        pool.attention.in_proj_weight.copy_(inp["in_proj_weight"])
        pool.attention.in_proj_bias.copy_(inp["in_proj_bias"])
        pool.attention.out_proj.weight.copy_(inp["out_proj.weight"])
        pool.attention.out_proj.bias.copy_(inp["out_proj.bias"])
    pool.train(case.training)
    pool.row_offset = case.row0
    pool._want_mask_bits = True
    pool.fold_key_projection = fold
    return pool, cm


def run_cuda(case: Case, inp: dict, dtype: torch.dtype, fold=None):
    """Forward + backward through the public API with the case's Philox (seed, offset, row0)."""
    pool, cm = make_pool(case, inp, dtype, fold)
    query0 = torch.nn.Parameter(inp["query0"].to(DEV, dtype))
    x = inp["x"].to(DEV, dtype).requires_grad_(True)
    value = inp["value"].to(DEV, dtype).requires_grad_(True) if case.separate_value else None
    kpm = inp["key_padding_mask"].to(DEV) if case.kpm else None
    aecf_b200.set_rng_state(PHILOX_SEED, case.offset)
    try:
        out, info = pool(query0.expand(case.B, -1, -1), x, value, key_padding_mask=kpm, return_info=True)
        ent_loss = cm.entropy_loss(info["entropy"])
    finally:
        aecf_b200.set_rng_state(None)
    loss = (out.float() * inp["grad_out"].to(DEV)).sum()
    if case.pooled_grad:
        loss = loss + (info["attention_weights"] * inp["grad_pooled"].to(DEV)).sum()
    if not case.training:
        loss = loss + 0.5 * info["entropy"].sum()
    loss.backward()
    torch.cuda.synchronize()
    grads = {
        "key": x.grad, "query0": query0.grad,
        "in_proj_weight": pool.attention.in_proj_weight.grad, "in_proj_bias": pool.attention.in_proj_bias.grad,
        "out_proj.weight": pool.attention.out_proj.weight.grad, "out_proj.bias": pool.attention.out_proj.bias.grad,
    }
    if value is not None:
        grads["value"] = value.grad
    return out, info, ent_loss, grads, cm


def expected_bits(mask: torch.Tensor) -> np.ndarray:
    m = (mask.reshape(mask.shape[0], -1) > 0).numpy().astype(np.int64)
    return (m * (1 << np.arange(m.shape[1]))).sum(1).astype(np.uint8)


def check_forward(case, out, info, ent_loss, ref, ref_loss, tol, exact_masks=True):
    assert_close("out", out.cpu(), ref.out, tol)
    assert_close("attention_weights", info["attention_weights"].cpu(), ref.info["attention_weights"], tol, atol=tol)
    assert_close("entropy", info["entropy"].cpu(), ref.info["entropy"], tol, atol=tol * max(math.log(max(case.M, 2)), 1))
    if exact_masks:
        assert np.array_equal(info["mask_bits"].cpu().numpy(), expected_bits(ref.info["mask"])), "mask bits differ"
        assert torch.equal(info["mask_rate"].cpu(), ref.info["mask_rate"].float()), "mask_rate differs"
    assert_close("masked_attention_weights", info["masked_attention_weights"].cpu(),
                 ref.info["masked_attention_weights"], tol, atol=tol)
    assert_close("entropy_loss", ent_loss.cpu(), ref_loss, tol, atol=tol)
    if case.training:
        assert "target_entropy" in info
        assert_close("target_entropy", info["target_entropy"].cpu(), ref.info["target_entropy"], 1e-6, atol=1e-6)
        assert not info["entropy"].requires_grad                       # detached in training (reference :278)
    else:
        assert "target_entropy" not in info and info["entropy"].requires_grad
    assert info["attention_weights"].requires_grad                      # keeps its graph (reference :538)
    assert not info["masked_attention_weights"].requires_grad


def check_grads(case, grads, ref_grads, tol):
    assert_close("grad key", grads["key"].cpu(), ref_grads["key"], tol)
    if case.separate_value:
        assert_close("grad value", grads["value"].cpu(), ref_grads["value"], tol)
    assert_close("grad query0", grads["query0"].cpu(), ref_grads["query0"], tol)
    assert_close("grad out_proj.bias", grads["out_proj.bias"].cpu(), ref_grads["out_proj.bias"], tol)
    assert_close("grad out_proj.weight", grads["out_proj.weight"].cpu(), ref_grads["out_proj.weight"], tol)
    assert_close("grad in_proj_weight", grads["in_proj_weight"].cpu(), ref_grads["in_proj_weight"], tol)
    scale = finite_scale(ref_grads["in_proj_bias"])        # the K-bias third is analytically zero
    assert_close("grad in_proj_bias", grads["in_proj_bias"].cpu(), ref_grads["in_proj_bias"], tol, atol=tol * scale)


FP32_CASES = [c for c in CASES if c.dtype == "float32"]


@pytest.mark.parametrize("case", FP32_CASES, ids=lambda c: c.name)
def test_fp32_matches_oracle(case):
    inp = build_inputs(case)
    ref, ref_grads = run_oracle(case, inp)
    last = case.M if (case.training and case.M > 1) else 2
    ref_loss = oracle.entropy_loss(ref.info["entropy"], last, case.entropy_target)
    out, info, ent_loss, grads, cm = run_cuda(case, inp, torch.float32)
    assert cm._last_seq_len == last
    check_forward(case, out, info, ent_loss, ref, ref_loss, FP32_TOL)
    check_grads(case, grads, ref_grads, FP32_TOL)


@pytest.mark.parametrize("case", FP32_CASES, ids=lambda c: c.name)
def test_fp32_matches_reference_golden(case):
    """Directly against what the unmodified reference produced on the same inputs and draws."""
    g = load_golden(case)
    inp = build_inputs(case)
    out, info, ent_loss, grads, _ = run_cuda(case, inp, torch.float32)
    tol = 2e-5       # the reference's own fp32 rounding (MKL summation order) is part of this distance
    assert_close("out", out.cpu(), g["out"], tol)
    assert_close("attention_weights", info["attention_weights"].cpu(), g["attention_weights"], tol, atol=tol)
    assert_close("entropy", info["entropy"].cpu(), g["entropy"], tol, atol=tol)
    assert np.array_equal(info["mask_rate"].cpu().numpy(), g["mask_rate"]), "mask_rate differs from the reference"
    live = g["attention_weights"] > 0
    bits = info["mask_bits"].cpu().numpy()[:, None] >> np.arange(case.M)[None, :] & 1
    if case.training and case.M > 1:
        assert np.array_equal((bits.reshape(g["attention_weights"].shape) > 0) & live,
                              g["masked_attention_weights"] > 0), "active-token set differs from the reference"
    assert_close("masked", info["masked_attention_weights"].cpu(), g["masked_attention_weights"], tol, atol=tol)
    assert_close("entropy_loss", ent_loss.cpu(), g["entropy_loss"], tol, atol=tol)
    assert sorted(k for k in info if k != "mask_bits") == sorted(json.loads(str(g["info_keys"])))
    assert_close("grad_x", grads["key"].cpu(), g["grad_x"], tol)
    assert_close("grad_query0", grads["query0"].cpu(), g["grad_query0"], tol)
    assert_close("grad_out_proj_bias", grads["out_proj.bias"].cpu(), g["grad_out_proj_bias"], tol)
    if case.full_grads:
        assert_close("grad_in_proj_weight", grads["in_proj_weight"].cpu(), g["grad_in_proj_weight"], tol)
        assert_close("grad_out_proj_weight", grads["out_proj.weight"].cpu(), g["grad_out_proj_weight"], tol)
    else:
        assert_close("grad_in_proj_weight_rowsum", grads["in_proj_weight"].cpu().sum(1), g["grad_in_proj_weight_rowsum"], tol)
        assert_close("grad_out_proj_weight_strided", grads["out_proj.weight"].cpu().flatten()[::97],
                     g["grad_out_proj_weight_strided"], tol)


FOLDABLE_FP32_CASES = [c for c in FP32_CASES if not c.separate_value]


@pytest.mark.parametrize("case", FOLDABLE_FP32_CASES, ids=lambda c: c.name)
def test_fp32_folded_key_projection_matches_oracle(case):
    """The folded key projection (scores = x . (scale Wk_h^T q_h) out of the value GEMM's side output, ds stored
    next to dV, rank-H key-side gradients through the GEMMs' extra columns) in fp32 against the UNFOLDED oracle:
    same tolerance as the unfolded path, masks and active sets bit-exact."""
    inp = build_inputs(case)
    ref, ref_grads = run_oracle(case, inp)
    last = case.M if (case.training and case.M > 1) else 2
    ref_loss = oracle.entropy_loss(ref.info["entropy"], last, case.entropy_target)
    out, info, ent_loss, grads, _ = run_cuda(case, inp, torch.float32, fold=True)
    check_forward(case, out, info, ent_loss, ref, ref_loss, FP32_TOL)
    check_grads(case, grads, ref_grads, FP32_TOL)


BF16_CASES = [c for c in FP32_CASES if c.name in (
    "config1_d512_h1_m3", "d64_h8_m3", "d64_h8_m3_dropout", "xray_d256_h4_m2", "d128_h4_m8_minactive2",
    "d64_h4_m4_kpm", "d64_h2_m3_separate_value", "d256_h16_m6")]


def _bf16_inputs(case):
    inp = build_inputs(case)
    for k in ("in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias", "query0", "x", "value", "grad_out"):
        if k in inp:
            inp[k] = inp[k].bfloat16().float()
    return inp


@pytest.mark.parametrize("fold", [True, False], ids=["folded", "unfolded"])
@pytest.mark.parametrize("case", BF16_CASES, ids=lambda c: c.name)
def test_bf16_matches_fp32_math_oracle(case, fold):
    """north_star: bf16 within 2e-2 of fp32 math on the bf16-rounded inputs (SURVEY.md section 0 item 8),
    with the folded key projection (the bf16 default) and without it."""
    inp = _bf16_inputs(case)
    ref, ref_grads = run_oracle(case, inp)
    last = case.M if (case.training and case.M > 1) else 2
    ref_loss = oracle.entropy_loss(ref.info["entropy"], last, case.entropy_target)
    out, info, ent_loss, grads, _ = run_cuda(case, inp, torch.bfloat16, fold=fold)
    check_forward(case, out.float(), info, ent_loss, ref, ref_loss, BF16_TOL, exact_masks=False)
    check_grads(case, {k: v.float() for k, v in grads.items()}, ref_grads, BF16_TOL)
    flips = int((torch.from_numpy(np.unpackbits(info["mask_bits"].cpu().numpy()[:, None], axis=1, bitorder="little")
                                  [:, :case.M]) != (ref.info["mask"].reshape(case.B, case.M) > 0)).sum())
    assert flips <= max(1, case.B * case.M // 50), f"{flips} mask flips against fp32 math"


@pytest.mark.parametrize("fold", [True, False], ids=["folded", "unfolded"])
@pytest.mark.parametrize("case", BF16_CASES, ids=lambda c: c.name)
def test_bf16_masks_exact_against_stage_rounded_oracle(case, fold):
    """With the oracle rounding K/V, ctx and out to bf16 where the CUDA path stores them (folded: the per-head
    score vector Qk instead of K), the masks and the active-token sets are bit-exact and everything else is far
    inside the bf16 budget."""
    inp = _bf16_inputs(case)
    folded = fold and not case.separate_value            # with a separate value tensor the module keeps K
    ref, ref_grads = run_oracle(case, inp, storage=torch.bfloat16, fold_key=folded)
    out, info, _, grads, _ = run_cuda(case, inp, torch.bfloat16, fold=fold)
    assert np.array_equal(info["mask_bits"].cpu().numpy(), expected_bits(ref.info["mask"])), "mask bits differ"
    assert torch.equal(info["mask_rate"].cpu(), ref.info["mask_rate"].float())
    assert_close("attention_weights", info["attention_weights"].cpu(), ref.info["attention_weights"], 1e-4, atol=1e-5)
    assert_close("entropy", info["entropy"].cpu(), ref.info["entropy"], 1e-4, atol=1e-5)
    assert_close("out", out.float().cpu(), ref.out, 1e-2)
    assert_close("grad key", grads["key"].float().cpu(), ref_grads["key"], BF16_TOL)


# ---------------------------------------------------------------------------------------------
# rows wider than one warp's slice: several warps share a sample (pool_core.cuh, WPS > 1)
# ---------------------------------------------------------------------------------------------
WIDE_CASES = [
    Case("wide_d1024_h8_m3", B=24, M=3, D=1024, H=8, dropout=0.1, pooled_grad=True, data_seed=31, offset=2),
    Case("wide_d2048_h16_m2", B=12, M=2, D=2048, H=16, data_seed=32, base_mask_prob=0.5),
    Case("wide_d1024_h4_m4_eval", B=10, M=4, D=1024, H=4, training=False, pooled_grad=True, data_seed=33),
    Case("wide_d512_h8_m5_kpm", B=20, M=5, D=512, H=8, kpm=True, min_active=2, base_mask_prob=0.8, data_seed=34),
]


@pytest.mark.parametrize("case", WIDE_CASES, ids=lambda c: c.name)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_wide_rows_span_several_warps(case, dtype):
    if dtype == torch.float32:
        inp = build_inputs(case)
        ref, ref_grads = run_oracle(case, inp)
        tol = FP32_TOL
    else:
        inp = _bf16_inputs(case)
        ref, ref_grads = run_oracle(case, inp, storage=torch.bfloat16, fold_key=True)   # bf16 folds by default
        tol = BF16_TOL
    out, info, _, grads, _ = run_cuda(case, inp, dtype)
    assert np.array_equal(info["mask_bits"].cpu().numpy(), expected_bits(ref.info["mask"])), "mask bits differ"
    assert torch.equal(info["mask_rate"].cpu(), ref.info["mask_rate"].float())
    assert_close("out", out.float().cpu(), ref.out, tol)
    assert_close("attention_weights", info["attention_weights"].cpu(), ref.info["attention_weights"],
                 tol if dtype == torch.float32 else 1e-4, atol=1e-5)
    assert_close("entropy", info["entropy"].cpu(), ref.info["entropy"], tol if dtype == torch.float32 else 1e-4, atol=1e-5)
    check_grads(case, {k: v.float() for k, v in grads.items()}, ref_grads, tol)


# rows of 3 * 2^k sixteen-byte slices (D = 768 / 640 in fp32, 1536 in bf16): the plan widens the warp slices to J = 4
# so that the row still splits over a power-of-two number of warps (api.cu make_plan); the last warp is partly idle
THREE_SLICE_CASES = [
    Case("d768_h12_m3", B=9, M=3, D=768, H=12, dropout=0.1, pooled_grad=True, data_seed=301),
    Case("d768_h6_m4_kpm", B=17, M=4, D=768, H=6, kpm=True, min_active=2, base_mask_prob=0.9, data_seed=302),
    Case("d640_h5_m7", B=10, M=7, D=640, H=5, dropout=0.5, data_seed=303),
    Case("d1536_h12_m2", B=6, M=2, D=1536, H=12, data_seed=304),
]


@pytest.mark.parametrize("case", THREE_SLICE_CASES, ids=lambda c: c.name)
def test_rows_of_three_slices(case):
    if case.D <= 768:
        test_fp32_matches_oracle(case)
        test_fp32_folded_key_projection_matches_oracle(case)
    for fold in (True, False):
        test_bf16_masks_exact_against_stage_rounded_oracle(case, fold)


@pytest.mark.parametrize("case", WIDE_CASES, ids=lambda c: c.name)
def test_wide_rows_folded_fp32(case):
    inp = build_inputs(case)
    ref, ref_grads = run_oracle(case, inp)
    out, info, _, grads, _ = run_cuda(case, inp, torch.float32, fold=True)
    assert np.array_equal(info["mask_bits"].cpu().numpy(), expected_bits(ref.info["mask"])), "mask bits differ"
    assert_close("out", out.cpu(), ref.out, FP32_TOL)
    assert_close("attention_weights", info["attention_weights"].cpu(), ref.info["attention_weights"], FP32_TOL, atol=1e-5)
    check_grads(case, grads, ref_grads, FP32_TOL)


def test_folded_sequence_first_and_large_batch_against_unfolded():
    """bf16, B large enough for the tcgen05 GEMMs (192-wide tiles with the fp32 score side output, K = D + 8
    contractions in the backward): folded and unfolded paths agree within the bf16 budget, in both layouts,
    and the folded path is bit-identical between the batch-first and the sequence-first layout."""
    torch.manual_seed(5)
    B, M, D, H = 1000, 3, 512, 8
    q, pool = aecf_b200.create_fusion_pool(D, M, 0.3, num_heads=H, dropout=0.1, device=DEV, dtype=torch.bfloat16)
    with torch.no_grad():
        pool.attention.in_proj_bias.normal_(0, 0.1)
        q.mul_(8.0)
    pool._want_mask_bits = True
    x = (torch.randn(B, M, D, device=DEV) * 2).bfloat16()
    g = torch.randn(B, 1, D, device=DEV).bfloat16()
    res = {}
    for name, fold, seq_first in (("folded", True, False), ("unfolded", False, False), ("folded_seq", True, True)):
        pool.fold_key_projection = fold
        pool.batch_first = not seq_first
        xs = (x.transpose(0, 1).contiguous() if seq_first else x.clone()).requires_grad_(True)
        qq = q.expand(-1, B, -1) if seq_first else q.expand(B, -1, -1)
        aecf_b200.set_rng_state(31, 2)
        out, info = pool(qq, xs, return_info=True)
        (out.reshape(B, D).float() * g.reshape(B, D).float()).sum().backward()
        res[name] = dict(out=out.detach().reshape(B, D).float(), pooled=info["attention_weights"].detach().reshape(B, M),
                         bits=info["mask_bits"].clone(), gx=(xs.grad.transpose(0, 1) if seq_first else xs.grad).float(),
                         gw=pool.attention.in_proj_weight.grad.float().clone(), gb=pool.attention.in_proj_bias.grad.float().clone(),
                         gq=q.grad.float().clone())
        pool.zero_grad(); q.grad = None
    aecf_b200.set_rng_state(None)
    pool.batch_first = True
    a, b, c = res["folded"], res["unfolded"], res["folded_seq"]
    for k in ("out", "gx", "gw", "gq"):
        assert_close(f"folded vs unfolded {k}", a[k].cpu(), b[k].cpu(), BF16_TOL)
    assert_close("pooled", a["pooled"].cpu(), b["pooled"].cpu(), 1e-2, atol=2e-3)
    assert_close("bias grad (value third)", a["gb"][2 * D:].cpu(), b["gb"][2 * D:].cpu(), BF16_TOL)
    flips = int((a["bits"] != b["bits"]).sum())
    assert flips <= B // 50, f"{flips} rows with different masks between the folded and the unfolded path"
    for k in ("out", "pooled", "bits", "gx"):
        assert torch.equal(a[k], c[k]), f"sequence-first folded path differs in {k}"
    assert_close("seq-first gw", a["gw"].cpu(), c["gw"].cpu(), 1e-2)


@pytest.mark.parametrize("shape", [(640, 512, 512, 8), (300, 256, 128, 4), (1024, 1024, 256, 16), (96, 64, 64, 1)],
                         ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_gemm_with_side_output(shape, dtype):
    """aecf_gemm_aux: C = A B[:n]^T + bias and the fp32 side output A B[n:n+aux]^T in one call (one tcgen05 launch
    with 192-wide tiles when bf16 and m, n >= 128; two SIMT launches otherwise)."""
    m, n, k, aux = shape
    torch.manual_seed(m + n)
    per16 = 8 if dtype == torch.bfloat16 else 4
    rows = n + (aux + per16 - 1) // per16 * per16
    a = torch.randn(m, k, device=DEV).to(dtype)
    b = torch.randn(rows, k, device=DEV).to(dtype)
    b[n + aux:] = 0
    bias = torch.randn(n, device=DEV).to(dtype)
    c, side = ops.gemm_aux(a, b, m=m, n=n, k=k, aux_cols=aux, bias=bias, out_dtype=torch.float32)
    want = a.double() @ b.double().t()
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    assert_close("C", c.cpu(), (want[:, :n] + bias.double()).cpu(), tol)
    assert_close("side", side[:, :aux].cpu(), want[:, n:n + aux].cpu(), 1e-5 if dtype == torch.float32 else 1e-5)
    assert float(side[:, aux:].abs().max()) == 0.0 if side.shape[1] > aux else True


# ---------------------------------------------------------------------------------------------
# full-size, size-independent properties (BASELINE.json configs[1]: B=65536, M=3, D=512, H=8 bf16)
# ---------------------------------------------------------------------------------------------
def _headline(B=65536, M=3, D=512, H=8, dtype=torch.bfloat16, dropout=0.0, seed=0):
    torch.manual_seed(seed)
    q, pool = aecf_b200.create_fusion_pool(D, M, 0.15, num_heads=H, dropout=dropout, device=DEV, dtype=dtype)
    x = torch.randn(B, M, D, device=DEV, dtype=dtype)
    return q, pool, x


# The headline configuration ITSELF against the oracle (VERDICT r1, weak 1): every product on the tcgen05 kernels, the
# streaming pool kernels, the folded key projection -- the path that produces the benchmark number.  Inputs are *peaked*
# (SURVEY.md section 8d) so that keep_prob really depends on the entropy.  The oracle (fp32 math, bf16 where the CUDA path
# stores bf16, folded like it) takes ~3 s at B = 65 536; building the Philox inputs ~25 s.
FULL_SIZE_CASES = [
    Case("headline_b65536_d512_h8_m3", B=65536, M=3, D=512, H=8, data_seed=41, offset=1),
    Case("b4096_d512_h8_m3_dropout", B=4096, M=3, D=512, H=8, dropout=0.1, pooled_grad=True, data_seed=42, offset=4, row0=4096),
]


@pytest.mark.parametrize("case", FULL_SIZE_CASES, ids=lambda c: c.name)
def test_full_size_bf16_folded_against_oracle(case):
    inp = _bf16_inputs(case)
    ref, ref_grads = run_oracle(case, inp, storage=torch.bfloat16, fold_key=True)
    ref32, _ = run_oracle(case, inp)                                   # fp32 math on the same inputs, unfolded
    out, info, ent_loss, grads, _ = run_cuda(case, inp, torch.bfloat16, fold=True)
    B, M = case.B, case.M
    if B >= 4096:
        assert _lib.gemm_last_kernel().startswith("tcgen05"), _lib.gemm_last_kernel()
    # peaked inputs: the entropy -> keep_prob dependence is exercised (flat attention would give mask_rate = base = 0.15)
    ne = ref.info["entropy"].reshape(-1) / math.log(M)
    assert float(ne.quantile(0.1)) < 0.3 and float(ne.quantile(0.9)) > 0.8
    assert np.array_equal(info["mask_bits"].cpu().numpy(), expected_bits(ref.info["mask"])), "mask bits differ"
    assert torch.equal(info["mask_rate"].cpu(), ref.info["mask_rate"].float()), "mask_rate differs"
    assert_close("attention_weights", info["attention_weights"].cpu(), ref.info["attention_weights"], 1e-4, atol=1e-5)
    assert_close("masked_attention_weights", info["masked_attention_weights"].cpu(), ref.info["masked_attention_weights"], 1e-4, atol=1e-5)
    assert_close("entropy", info["entropy"].cpu(), ref.info["entropy"], 1e-4, atol=1e-5)
    assert_close("entropy_loss", ent_loss.cpu(), oracle.entropy_loss(ref.info["entropy"], M, case.entropy_target), 1e-4)
    assert_close("out", out.float().cpu(), ref.out, 1e-2)
    # ... and per ROW, so that no small-norm row hides behind the tensor's largest entry
    err = (out.float().cpu().reshape(B, -1) - ref.out.reshape(B, -1)).abs().amax(1)
    row_scale = ref.out.reshape(B, -1).abs().amax(1)
    assert bool((err <= BF16_TOL * row_scale + 1e-3).all()), f"worst row: {float((err / row_scale).max()):.3e}"
    check_grads(case, {k: v.float() for k, v in grads.items()}, ref_grads, BF16_TOL)
    gx_err = (grads["key"].float().cpu().reshape(B * M, -1) - ref_grads["key"].reshape(B * M, -1)).abs().amax(1)
    gx_scale = ref_grads["key"].reshape(B * M, -1).abs().amax(1)
    assert bool((gx_err <= BF16_TOL * gx_scale + BF16_TOL * float(gx_scale.median())).all())
    # north_star: within 2e-2 of fp32 math too; bf16 storage moves keep_prob by ~1e-3, so a few draws may flip
    assert_close("out vs fp32 math", out.float().cpu(), ref32.out, BF16_TOL)
    flips = int((torch.from_numpy(np.unpackbits(info["mask_bits"].cpu().numpy()[:, None], axis=1, bitorder="little")[:, :M])
                 != (ref32.info["mask"].reshape(B, M) > 0)).sum())
    assert flips <= B * M // 50, f"{flips} mask flips against fp32 math"


def test_headline_shape_properties_and_determinism():
    q, pool, x = _headline(dropout=0.1)
    pool._want_mask_bits = True
    B, M = x.shape[0], x.shape[1]
    runs = []
    for _ in range(2):
        aecf_b200.set_rng_state(123, 7)
        xg = x.clone().requires_grad_(True)
        out, info = pool(q.expand(B, -1, -1), xg, return_info=True)
        (out.float().pow(2).mean() + 0.01 * pool.curriculum_masking.entropy_loss(info["entropy"])).backward()
        runs.append((out.detach(), info, xg.grad, pool.attention.in_proj_weight.grad.clone(), q.grad.clone()))
        pool.zero_grad(); q.grad = None
    aecf_b200.set_rng_state(None)
    (o1, i1, gx1, gw1, gq1), (o2, i2, gx2, gw2, gq2) = runs
    # bit-reproducible run to run (no atomics anywhere on the path)
    assert torch.equal(o1, o2) and torch.equal(gx1, gx2) and torch.equal(gw1, gw2) and torch.equal(gq1, gq2)
    assert torch.equal(i1["mask_bits"], i2["mask_bits"])
    masked = i1["masked_attention_weights"]
    assert torch.allclose(masked.sum(-1), torch.ones_like(masked.sum(-1)), atol=1e-5)
    bits = i1["mask_bits"].long()
    active = sum((bits >> m) & 1 for m in range(M))
    assert int(active.min()) >= 1
    assert torch.equal(i1["mask_rate"].reshape(-1), 1.0 - active.float() / M)
    ent = i1["entropy"]
    assert float(ent.min()) >= 0.0 and float(ent.max()) <= math.log(M) + 1e-6
    assert ((masked > 0).reshape(B, M) <= (((bits[:, None] >> torch.arange(M, device=DEV)) & 1) > 0)).all()
    for t in (o1, gx1, gw1, gq1):
        assert torch.isfinite(t.float()).all()
    # mask statistics: with flat attention keep_prob ~ 0.85 per token
    assert not i1["mask_rate"].requires_grad and not i1["entropy"].requires_grad
    assert abs(float(i1["mask_rate"].mean()) - 0.15) < 0.01


def test_torch_manual_seed_reproduces_masks():
    """Without set_rng_state the Philox (seed, offset) follow torch's CUDA generator: re-seeding replays
    the same masks, the next call draws new ones."""
    q, pool, x = _headline(B=4096)
    pool._want_mask_bits = True

    def masks():
        return pool(q.expand(x.shape[0], -1, -1), x, return_info=True)[1]["mask_bits"].clone()

    torch.manual_seed(11)
    a1, a2 = masks(), masks()
    torch.manual_seed(11)
    b1 = masks()
    assert torch.equal(a1, b1) and not torch.equal(a1, a2)


def test_batch_sharding_reproduces_masks_and_sums_gradients():
    """Rows are independent and Philox is keyed on the GLOBAL row: two half-batches with
    row_offset = 0 / B/2 give the full-batch outputs and masks bit for bit, and parameter gradients
    that add up to the full-batch ones (the data-parallel contract, SURVEY.md section 8e)."""
    q, pool, x = _headline(B=8192, dropout=0.1)
    pool._want_mask_bits = True
    B = x.shape[0]

    def step(xs, row0):
        pool.row_offset = row0
        aecf_b200.set_rng_state(99, 3)
        xs = xs.clone().requires_grad_(True)
        out, info = pool(q.expand(xs.shape[0], -1, -1), xs, return_info=True)
        out.float().pow(2).sum().backward()
        res = (out.detach(), info["mask_bits"].clone(), xs.grad, pool.attention.in_proj_weight.grad.float().clone(),
               q.grad.float().clone())
        pool.zero_grad(); q.grad = None
        return res

    full = step(x, 0)
    lo, hi = step(x[: B // 2], 0), step(x[B // 2:], B // 2)
    aecf_b200.set_rng_state(None); pool.row_offset = 0
    assert torch.equal(torch.cat([lo[0], hi[0]]), full[0])
    assert torch.equal(torch.cat([lo[1], hi[1]]), full[1])
    assert torch.equal(torch.cat([lo[2], hi[2]]), full[2])
    assert_close("in_proj_weight grad", (lo[3] + hi[3]).cpu(), full[3].cpu(), 2e-2)
    assert_close("query grad", (lo[4] + hi[4]).cpu(), full[4].cpu(), 2e-2)


# ---------------------------------------------------------------------------------------------
# API surface on the device
# ---------------------------------------------------------------------------------------------
def test_sequence_first_layout_matches_batch_first():
    case = CASES_BY_NAME["d64_h8_m3"]
    inp = build_inputs(case)
    pool_b, _ = make_pool(case, inp, torch.float32)
    pool_s, _ = make_pool(case, inp, torch.float32)
    pool_s.batch_first = False
    q = inp["query0"].to(DEV)
    x = inp["x"].to(DEV)
    outs = []
    for pool, qq, xx in ((pool_b, q.expand(case.B, -1, -1), x),
                         (pool_s, q.expand(-1, case.B, -1), x.transpose(0, 1).contiguous())):
        aecf_b200.set_rng_state(PHILOX_SEED, 0)
        xx = xx.clone().requires_grad_(True)
        out, info = pool(qq, xx, return_info=True)
        out.pow(2).sum().backward()
        outs.append((out, info, xx.grad))
    aecf_b200.set_rng_state(None)
    assert outs[1][0].shape == (1, case.B, case.D)
    assert torch.equal(outs[0][0].reshape(case.B, case.D), outs[1][0].reshape(case.B, case.D))
    assert torch.equal(outs[0][1]["mask_bits"], outs[1][1]["mask_bits"])
    assert torch.equal(outs[0][2], outs[1][2].transpose(0, 1))


def test_per_row_queries_match_oracle():
    case = CASES_BY_NAME["d64_h8_m3_dropout"]
    inp = build_inputs(case)
    queries = torch.from_numpy(philox.normal(4242, (case.B, 1, case.D))).float() * 0.3
    fwd = oracle.pool_forward(queries, inp["x"], None, inp["in_proj_weight"], inp["in_proj_bias"],
                              inp["out_proj.weight"], inp["out_proj.bias"], case.H, dropout_p=case.dropout,
                              training=True, u_drop=inp["u_drop"], u_mask=inp["u_mask"], masking=masking_kwargs(case))
    grads = oracle.pool_backward(queries, inp["x"], None, inp["in_proj_weight"], inp["out_proj.weight"], case.H,
                                 fwd.saved, inp["grad_out"], dropout_p=case.dropout, training=True)
    pool, _ = make_pool(case, inp, torch.float32)
    qd = queries.to(DEV).requires_grad_(True)
    xd = inp["x"].to(DEV).requires_grad_(True)
    aecf_b200.set_rng_state(PHILOX_SEED, case.offset)
    out, info = pool(qd, xd, return_info=True)
    aecf_b200.set_rng_state(None)
    (out * inp["grad_out"].to(DEV)).sum().backward()
    assert_close("out", out.cpu(), fwd.out, FP32_TOL)
    assert np.array_equal(info["mask_bits"].cpu().numpy(), expected_bits(fwd.info["mask"]))
    assert_close("grad query", qd.grad.cpu(), grads["query"], FP32_TOL)
    assert_close("grad key", xd.grad.cpu(), grads["key"], FP32_TOL)
    assert_close("grad in_proj_weight", pool.attention.in_proj_weight.grad.cpu(), grads["in_proj_weight"], FP32_TOL)
    scale = finite_scale(grads["in_proj_bias"])
    assert_close("grad in_proj_bias", pool.attention.in_proj_bias.grad.cpu(), grads["in_proj_bias"], FP32_TOL,
                 atol=FP32_TOL * scale)


def test_attn_mask_forms_match_oracle():
    """attn_mask as torch accepts it for one target token: (1, M) bool, (1, M) float, (B*H, 1, M) float,
    alone or merged with a key_padding_mask (torch/nn/functional.py:6608-6620)."""
    case = CASES_BY_NAME["d64_h4_m4_kpm"]
    inp = build_inputs(case)
    B, M, H, D = case.B, case.M, case.H, case.D
    kpm = inp["key_padding_mask"]
    per_head = torch.from_numpy(philox.normal(77, (B * H, 1, M))).float()
    per_head[::5, 0, 1] = float("-inf")
    masks = {
        "bool_2d": (torch.tensor([[False, False, True, False]]), None),
        "float_2d": (torch.tensor([[0.0, -1.5, 0.5, float("-inf")]]), None),
        "float_3d": (per_head, None),
        "float_3d_plus_kpm": (per_head, kpm),
    }
    q = inp["query0"].expand(B, 1, D)
    for name, (am, pad) in masks.items():
        bias = am.float() if am.dtype != torch.bool else torch.zeros(am.shape).masked_fill(am, float("-inf"))
        bias = bias.reshape(1, 1, 1, M) if bias.dim() == 2 else bias.reshape(B, H, 1, M)
        if pad is not None:
            bias = bias + torch.zeros(B, 1, 1, M).masked_fill(pad.view(B, 1, 1, M), float("-inf"))
        ref = oracle.pool_forward(q, inp["x"], None, inp["in_proj_weight"], inp["in_proj_bias"], inp["out_proj.weight"],
                                  inp["out_proj.bias"], H, training=True, u_mask=inp["u_mask"], u_drop=inp["u_drop"],
                                  score_bias=bias, masking=masking_kwargs(case))
        grads = oracle.pool_backward(q, inp["x"], None, inp["in_proj_weight"], inp["out_proj.weight"], H, ref.saved,
                                     inp["grad_out"])
        pool, _ = make_pool(case, inp, torch.float32)
        x = inp["x"].to(DEV).requires_grad_(True)
        aecf_b200.set_rng_state(PHILOX_SEED, case.offset)
        out, info = pool(q.to(DEV), x, attn_mask=am.to(DEV), key_padding_mask=None if pad is None else pad.to(DEV),
                         return_info=True)
        aecf_b200.set_rng_state(None)
        (out * inp["grad_out"].to(DEV)).sum().backward()
        assert_close(f"{name}: out", out.cpu(), ref.out, FP32_TOL)
        assert_close(f"{name}: weights", info["attention_weights"].cpu(), ref.info["attention_weights"], FP32_TOL, atol=1e-6)
        assert np.array_equal(info["mask_bits"].cpu().numpy(), expected_bits(ref.info["mask"])), name
        assert_close(f"{name}: grad x", x.grad.cpu(), grads["key"], FP32_TOL)


def test_no_masking_module_and_plain_output():
    case = CASES_BY_NAME["d64_h8_m3"]
    inp = build_inputs(case)
    pool, _ = make_pool(case, inp, torch.float32)
    pool.curriculum_masking = None                                  # runtime toggle (xrays/train_xrays_example.py:179-187)
    q, x = inp["query0"].to(DEV).expand(case.B, -1, -1), inp["x"].to(DEV)
    out = pool(q, x)
    assert isinstance(out, torch.Tensor) and out.shape == (case.B, 1, case.D)
    out2, info = pool(q, x, return_info=True, use_checkpoint=True)
    assert set(info) == {"attention_weights"} and torch.equal(out, out2)
    ref, _ = run_oracle(case, inp)
    assert_close("out", out.cpu(), ref.out, FP32_TOL)


@pytest.mark.parametrize("dtype,fold", [(torch.float32, False), (torch.float32, True), (torch.bfloat16, True), (torch.bfloat16, False)],
                         ids=["fp32_unfolded", "fp32_folded", "bf16_folded", "bf16_unfolded"])
def test_module_without_biases(dtype, fold):
    """bias=False (reference aecf/AECFLayer.py:377): no in_proj_bias / out_proj.bias, null bias pointers through the ABI."""
    case = CASES_BY_NAME["d64_h8_m3_dropout"]
    inp = build_inputs(case)
    if dtype == torch.bfloat16:
        inp = {k: (v.bfloat16().float() if v.is_floating_point() and k not in ("u_mask", "u_drop") else v) for k, v in inp.items()}
    pool = aecf_b200.MultimodalAttentionPool(case.D, num_heads=case.H, dropout=case.dropout, bias=False,
                                             curriculum_masking=aecf_b200.CurriculumMasking(**masking_kwargs(case)),
                                             device=DEV, dtype=dtype)
    assert pool.attention.in_proj_bias is None and pool.attention.out_proj.bias is None
    with torch.no_grad():
        pool.attention.in_proj_weight.copy_(inp["in_proj_weight"])
        pool.attention.out_proj.weight.copy_(inp["out_proj.weight"])
    pool.fold_key_projection, pool._want_mask_bits = fold, True
    query0 = torch.nn.Parameter(inp["query0"].to(DEV, dtype))
    x = inp["x"].to(DEV, dtype).requires_grad_(True)
    aecf_b200.set_rng_state(PHILOX_SEED, case.offset)
    try:
        out, info = pool(query0.expand(case.B, -1, -1), x, return_info=True)
    finally:
        aecf_b200.set_rng_state(None)
    (out.float() * inp["grad_out"].to(DEV)).sum().backward()
    storage = torch.bfloat16 if dtype == torch.bfloat16 else None
    q = inp["query0"].expand(case.B, 1, case.D)
    ref = oracle.pool_forward(q, inp["x"], None, inp["in_proj_weight"], None, inp["out_proj.weight"], None, case.H,
                              dropout_p=case.dropout, training=True, u_drop=inp["u_drop"], u_mask=inp["u_mask"],
                              masking=masking_kwargs(case), storage=storage, fold_key=fold and storage is not None)
    grads = oracle.pool_backward(q, inp["x"], None, inp["in_proj_weight"], inp["out_proj.weight"], case.H, ref.saved, inp["grad_out"],
                                 dropout_p=case.dropout, training=True, has_bias=False, storage=storage,
                                 fold_key=fold and storage is not None)
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    assert np.array_equal(info["mask_bits"].cpu().numpy(), expected_bits(ref.info["mask"])), "mask bits differ"
    assert_close("out", out.float().cpu(), ref.out, tol)
    assert_close("grad key", x.grad.float().cpu(), grads["key"], tol)
    assert_close("grad in_proj_weight", pool.attention.in_proj_weight.grad.float().cpu(), grads["in_proj_weight"], tol)
    assert_close("grad out_proj.weight", pool.attention.out_proj.weight.grad.float().cpu(), grads["out_proj.weight"], tol)
    assert_close("grad query0", query0.grad.float().cpu(), grads["query"].sum(0, keepdim=True), tol)


def test_entropy_loss_comes_out_of_the_forward_kernel():
    """The per-sample entropy_loss term is fused into the streaming forward kernel (aecf_pool_desc::loss_out): for the
    info['entropy'] tensor of a training forward, CurriculumMasking.entropy_loss returns the kernel's scalar; a copy of the
    tensor, a modified tensor or another target take the stand-alone kernels -- all equal the oracle's value."""
    case = CASES_BY_NAME["d64_h8_m3_dropout"]
    inp = build_inputs(case)
    for dtype, fold in ((torch.float32, False), (torch.float32, True), (torch.bfloat16, True)):
        pool, cm = make_pool(case, inp, dtype, fold)
        launched = []
        plain = ops.entropy_loss_fwd
        try:
            ops.entropy_loss_fwd = lambda e, t: (launched.append(1), plain(e, t))[1]
            q = inp["query0"].to(DEV, dtype)
            aecf_b200.set_rng_state(PHILOX_SEED, case.offset)
            _, info = pool(q.expand(case.B, -1, -1), inp["x"].to(DEV, dtype), return_info=True)
            aecf_b200.set_rng_state(None)
            entropy = info["entropy"]
            fused = cm.entropy_loss(entropy)
            assert not launched and fused.shape == () and not fused.requires_grad
            want = oracle.entropy_loss(entropy.detach().float().cpu(), case.M, case.entropy_target)
            assert_close("fused entropy_loss", fused.float().cpu(), want, 1e-6, atol=1e-7)
            separate = cm.entropy_loss(entropy.clone())                    # not the forward's tensor object
            assert launched == [1]
            assert_close("stand-alone entropy_loss", separate.float().cpu(), want, 1e-6, atol=1e-7)
            cm.entropy_target = 0.5                                        # another target: the kernels again
            assert_close("other target", cm.entropy_loss(entropy).float().cpu(),
                         oracle.entropy_loss(entropy.detach().float().cpu(), case.M, 0.5), 1e-6, atol=1e-7)
            cm.entropy_target = case.entropy_target
            entropy.add_(1.0)                                              # modified in place since the forward
            assert_close("modified entropy", cm.entropy_loss(entropy).float().cpu(),
                         oracle.entropy_loss(entropy.detach().float().cpu(), case.M, case.entropy_target), 1e-6, atol=1e-7)
            assert len(launched) == 3
        finally:
            ops.entropy_loss_fwd = plain


@pytest.mark.parametrize("dtype,fold", [(torch.float32, False), (torch.float32, True), (torch.bfloat16, True), (torch.bfloat16, False)],
                         ids=["fp32_unfolded", "fp32_folded", "bf16_folded", "bf16_unfolded"])
def test_sample_index_pools_the_listed_rows_in_place(dtype, fold):
    """pool(query, x, sample_index=idx) against pool(query[idx], x[idx]) -- the reference x-ray model's gather -> pool ->
    scatter (xrays/train_xrays_example.py:202-222): same Philox rows, same info tensors, the same output rows at their places
    in the full batch, the same input gradients there and none anywhere else, the same parameter gradients."""
    case = CASES_BY_NAME["d64_h8_m3_dropout"]
    inp = build_inputs(case)
    B = case.B
    idx = torch.tensor([b for b in range(B) if (b * 7 + 3) % 5 not in (0, 1)], device=DEV)       # an irregular 3/5 of the rows
    g = inp["grad_out"].to(DEV, dtype)
    runs = {}
    for mode in ("gathered", "in_place"):
        pool, cm = make_pool(case, inp, dtype, fold)
        q = torch.nn.Parameter(inp["query0"].to(DEV, dtype))
        x = inp["x"].to(DEV, dtype).requires_grad_(True)
        aecf_b200.set_rng_state(PHILOX_SEED, case.offset)
        if mode == "gathered":
            out, info = pool(q.expand(idx.numel(), -1, -1), x[idx], return_info=True)
            loss = (out.float() * g[idx].float()).sum()
        else:
            out, info = pool(q.expand(B, -1, -1), x, return_info=True, sample_index=idx)
            assert out.shape == (B, 1, case.D)
            out = out[idx]                                       # (the test looks at the listed rows; a model would mask)
            loss = (out.float() * g[idx].float()).sum()
        (loss + (info["attention_weights"] * 0.3).sum()).backward()
        aecf_b200.set_rng_state(None)
        torch.cuda.synchronize()
        runs[mode] = dict(out=out.detach(), info={k: v.detach() for k, v in info.items()}, gx=x.grad,
                          gw=pool.attention.in_proj_weight.grad, gb=pool.attention.in_proj_bias.grad,
                          gwo=pool.attention.out_proj.weight.grad, gbo=pool.attention.out_proj.bias.grad, gq=q.grad)
    a, b = runs["gathered"], runs["in_place"]
    assert torch.equal(a["out"], b["out"])
    for k in a["info"]:
        assert a["info"][k].shape == b["info"][k].shape and torch.equal(a["info"][k], b["info"][k]), k
    assert torch.equal(a["gx"][idx], b["gx"][idx])
    others = torch.ones(B, dtype=torch.bool, device=DEV)
    others[idx] = False
    assert float(b["gx"][others].abs().max()) == 0.0
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    for k in ("gw", "gb", "gwo", "gbo", "gq"):
        scale = finite_scale(a[k].float())
        assert_close(k, b[k].float().cpu(), a[k].float().cpu(), tol, atol=tol * scale)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_in_projection_bias_gradient_both_ways(dtype):
    """The folded backward forms the value / key thirds of in_proj_bias.grad in one of two ways (csrc/pool_bwd.cuh): without
    dropout from the column sums of d_out (the softmax weights of a sample sum to one: d_bias_v = Wo^T colsum(d_out),
    d_bias_k = 0), otherwise from per-sample head sums and a walk over d_ctx.  sample_index=arange(B) forces the second way on
    a case without dropout: both must agree with each other, and the plain run with the oracle (the parity tests above)."""
    case = Case("bias_both_ways", B=200, M=3, D=128, H=8, pooled_grad=True, data_seed=77, offset=2)
    inp = build_inputs(case)
    g = inp["grad_out"].to(DEV, dtype)
    grads = {}
    for mode in ("column_sums", "per_sample_sums"):
        pool, cm = make_pool(case, inp, dtype, True)
        q = torch.nn.Parameter(inp["query0"].to(DEV, dtype))
        x = inp["x"].to(DEV, dtype).requires_grad_(True)
        aecf_b200.set_rng_state(PHILOX_SEED, case.offset)
        kw = {} if mode == "column_sums" else {"sample_index": torch.arange(case.B, device=DEV)}
        out, info = pool(q.expand(case.B, -1, -1), x, return_info=True, **kw)
        ((out.float() * g.float()).sum() + (info["attention_weights"] * 0.3).sum()).backward()
        aecf_b200.set_rng_state(None)
        grads[mode] = pool.attention.in_proj_bias.grad.float().cpu()
    a, b = grads["column_sums"], grads["per_sample_sums"]
    D = case.D
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    scale = finite_scale(b)
    assert_close("query third", a[:D], b[:D], tol, atol=tol * scale)
    assert_close("value third", a[2 * D:], b[2 * D:], tol, atol=tol * scale)
    assert float(a[D:2 * D].abs().max()) == 0.0                    # analytically zero, and written as such
    assert float(b[D:2 * D].abs().max()) <= tol * scale            # ... where the other way leaves rounding noise


def test_unsupported_shapes_fail_loudly():
    pool = aecf_b200.MultimodalAttentionPool(64, num_heads=4, device=DEV)
    x = torch.randn(4, 3, 64, device=DEV)
    assert pool(torch.randn(4, 2, 64, device=DEV), x).shape == (4, 2, 64)            # two queries per sample: supported
    with pytest.raises(_lib.UnsupportedShapeError):
        pool(torch.randn(4, 1, 64, device=DEV), torch.randn(4, 9, 64, device=DEV))   # 9 tokens > 8
    odd = aecf_b200.MultimodalAttentionPool(60, num_heads=4, device=DEV)             # head_dim 15
    with pytest.raises(_lib.UnsupportedShapeError):
        odd(torch.randn(4, 1, 60, device=DEV), torch.randn(4, 3, 60, device=DEV))
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        pool(torch.randn(4, 1, 64), torch.randn(4, 3, 64))          # CPU tensors: no fallback


def test_functional_fast_path_and_module_path():
    q = torch.from_numpy(philox.normal(1, (6, 2, 64))).float()
    k = torch.from_numpy(philox.normal(2, (6, 5, 64))).float()
    out = aecf_b200.multimodal_attention_pool(q.to(DEV), k.to(DEV))
    assert_close("sdpa", out.cpu(), oracle.sdpa_single_head(q, k, k), FP32_TOL)
    out_bf = aecf_b200.multimodal_attention_pool(q.to(DEV).bfloat16(), k.to(DEV).bfloat16())
    assert_close("sdpa bf16", out_bf.float().cpu(), oracle.sdpa_single_head(q.bfloat16().float(), k.bfloat16().float(),
                                                                           k.bfloat16().float()), BF16_TOL)
    cm = aecf_b200.CurriculumMasking(0.15)
    y = aecf_b200.multimodal_attention_pool(torch.randn(8, 1, 64, device=DEV), torch.randn(8, 3, 64, device=DEV),
                                            num_heads=4, curriculum_masking=cm, training=True)
    assert y.shape == (8, 1, 64) and y.is_cuda and torch.isfinite(y).all()


@pytest.mark.parametrize("shape", [(6, 2, 5, 64), (3, 1, 3, 512), (4, 7, 9, 136)], ids=lambda s: "x".join(map(str, s)))
def test_functional_fast_path_is_differentiable(shape):
    """reference aecf/AECFLayer.py:573-581 is plain torch, so gradients flow to query, key and value; here a recompute
    backward (aecf_sdpa_bwd) against autograd through the oracle's restatement -- also with key is value."""
    B, S, T, D = shape
    qc = torch.from_numpy(philox.normal(11, (B, S, D))).float()
    kc = torch.from_numpy(philox.normal(12, (B, T, D))).float()
    vc = torch.from_numpy(philox.normal(13, (B, T, D))).float()
    gc = torch.from_numpy(philox.normal(14, (B, S, D))).float()
    for dtype, tol in ((torch.float32, FP32_TOL), (torch.bfloat16, BF16_TOL)):
        if dtype == torch.bfloat16 and D % 8:
            continue
        ref_in = [t.to(dtype).float().clone().requires_grad_(True) for t in (qc, kc, vc)]     # clones: fresh leaves
        (oracle.sdpa_single_head(*ref_in) * gc.to(dtype).float()).sum().backward()
        ours = [t.detach().to(DEV, dtype).clone().requires_grad_(True) for t in (qc, kc, vc)]
        out = aecf_b200.multimodal_attention_pool(ours[0], ours[1], ours[2])
        assert out.requires_grad
        (out.float() * gc.to(DEV, dtype).float()).sum().backward()
        for name, a, b in zip(("d_query", "d_key", "d_value"), ours, ref_in):
            assert_close(name, a.grad.float().cpu(), b.grad, tol)
        kv = kc.detach().to(DEV, dtype).clone().requires_grad_(True)  # value=None: key is value, the two gradients add up
        q2 = qc.detach().to(DEV, dtype).clone().requires_grad_(True)
        (aecf_b200.multimodal_attention_pool(q2, kv).float() * gc.to(DEV, dtype).float()).sum().backward()
        rk = kc.to(dtype).float().clone().requires_grad_(True)
        (oracle.sdpa_single_head(qc.to(dtype).float(), rk, rk) * gc.to(dtype).float()).sum().backward()
        assert_close("d_key (key is value)", kv.grad.float().cpu(), rk.grad, tol)


def test_standalone_masking_and_entropy():
    cm = aecf_b200.CurriculumMasking(base_mask_prob=0.9, min_active=2).to(DEV)
    w = torch.softmax(2 * torch.from_numpy(philox.normal(5, (257, 10))).float(), -1)
    aecf_b200.set_rng_state(77, 5)
    masked, info = cm(w.to(DEV))
    aecf_b200.set_rng_state(None)
    u = torch.from_numpy(philox.mask_uniforms(77, 5, 0, 257, 10))
    ref = oracle.curriculum_mask(w, u, base_mask_prob=0.9, min_active=2)
    assert set(info) == {"entropy", "mask_rate", "target_entropy"}
    assert torch.equal(info["mask_rate"].cpu(), ref["mask_rate"])
    assert torch.equal(masked.cpu() > 0, ref["masked"] > 0)
    assert_close("masked", masked.cpu(), ref["masked"], FP32_TOL, atol=1e-6)
    assert_close("entropy", info["entropy"].cpu(), ref["entropy"], FP32_TOL, atol=1e-6)
    assert cm._last_seq_len == 10
    # the masked weights keep their graph (reference :262-272: final_weights = weights * mask / sum); mask and entropy do not
    g = torch.from_numpy(philox.normal(6, (257, 10))).float()
    wg = (w * 3.0).to(DEV).requires_grad_(True)                  # unnormalised rows: the first renormalisation matters too
    aecf_b200.set_rng_state(77, 5)
    mg, ig = cm(wg)
    aecf_b200.set_rng_state(None)
    assert mg.requires_grad and not ig["entropy"].requires_grad and not ig["mask_rate"].requires_grad
    (mg * g.to(DEV)).sum().backward()
    wr = (w * 3.0).clone().requires_grad_(True)
    keep = (ref["masked"] > 0).float()
    wn = wr / wr.sum(-1, keepdim=True)
    ((wn * keep / (wn * keep).sum(-1, keepdim=True)) * g).sum().backward()
    assert_close("d masked / d weights", wg.grad.cpu(), wr.grad, FP32_TOL, atol=1e-6)
    # eval mode: weights pass through, entropy stays differentiable (reference :150-156)
    cm.eval()
    wd = w.to(DEV).requires_grad_(True)
    same, einfo = cm(wd)
    assert same is wd and set(einfo) == {"entropy", "mask_rate"}
    einfo["entropy"].sum().backward()
    wc = w.clone().requires_grad_(True)
    oracle.shannon_entropy(wc).sum().backward()
    assert_close("d entropy", wd.grad.cpu(), wc.grad, FP32_TOL)
    assert_close("compute_entropy", cm.compute_entropy(w.to(DEV)).cpu(), oracle.shannon_entropy(w), FP32_TOL, atol=1e-6)
    edge = torch.tensor([[1.0, 0.0, 0.0], [0.33, 0.33, 0.34]], device=DEV)          # README.md:311-316
    cm.train()
    out, _ = cm(edge)
    assert torch.isfinite(out).all()


def test_entropy_loss_gradient_in_eval_mode():
    cm = aecf_b200.CurriculumMasking().to(DEV)
    e = (torch.rand(1000, 1, device=DEV) * 1.1).requires_grad_(True)
    loss = cm.entropy_loss(e)
    loss.backward()
    ec = e.detach().cpu().requires_grad_(True)
    ref = oracle.entropy_loss(ec, 2, 0.7)
    ref.backward()
    assert_close("loss", loss.cpu(), ref, FP32_TOL)
    assert_close("d loss", e.grad.cpu(), ec.grad, FP32_TOL)
    bad = torch.tensor([float("nan"), float("inf"), float("-inf"), 0.3], device=DEV)
    assert_close("scrubbed", cm.entropy_loss(bad).cpu(), oracle.entropy_loss(bad.cpu(), 2, 0.7), FP32_TOL)


# ---------------------------------------------------------------------------------------------
# the projection GEMM on its own, every operand layout the path uses
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("impl", [_lib.GEMM_SIMT, _lib.GEMM_AUTO], ids=["simt", "auto"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("shape", [(384, 256, 128), (200, 136, 72), (1024, 512, 2048), (1, 512, 512), (512, 512, 1)],
                         ids=lambda s: "x".join(map(str, s)))
def test_gemm_layouts(impl, dtype, shape):
    m, n, k = shape
    torch.manual_seed(m + n + k)
    a = torch.randn(m, k, device=DEV).to(dtype)
    b = torch.randn(n, k, device=DEV).to(dtype)
    bias = torch.randn(n, device=DEV).to(dtype)
    want = a.double() @ b.double().t()
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    for a_lay, a_mem in ((_lib.K_MAJOR, a), (_lib.MN_MAJOR, a.t().contiguous())):
        for b_lay, b_mem in ((_lib.K_MAJOR, b), (_lib.MN_MAJOR, b.t().contiguous())):
            for use_bias in (False, True):
                out = ops.gemm(a_mem, b_mem, m=m, n=n, k=k, a_layout=a_lay, b_layout=b_lay,
                               lda=a_mem.shape[1], ldb=b_mem.shape[1], bias=bias if use_bias else None,
                               out_dtype=torch.float32, impl=impl)
                ref = want + (bias.double() if use_bias else 0.0)
                assert_close(f"gemm a_layout={a_lay} b_layout={b_lay} bias={use_bias}", out.cpu(), ref.cpu(), tol)
    # strided output (the separate-value path writes K and V into the halves of one buffer)
    buf = torch.zeros(m, 2 * n, device=DEV, dtype=dtype)
    ops.gemm(a, b, m=m, n=n, k=k, a_layout=_lib.K_MAJOR, b_layout=_lib.K_MAJOR, lda=k, ldb=k, out=buf[:, n:], ldc=2 * n,
             impl=impl)
    assert_close("strided C", buf[:, n:].float().cpu(), want.cpu(), 2e-2 if dtype == torch.bfloat16 else tol)
    assert float(buf[:, :n].abs().max()) == 0.0


def test_colsum():
    for dtype in (torch.float32, torch.bfloat16):
        x = torch.randn(5000, 512, device=DEV).to(dtype)
        assert_close("colsum", ops.colsum(x, out_dtype=torch.float32).cpu(), x.double().sum(0).cpu(), 1e-5)
