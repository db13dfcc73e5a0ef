"""The kernel schedules that only large calls select, on a 148-SM B200, each checked against a high-precision reference.

Most parity tests run at B <= 64, where every projection takes the SIMT GEMM and every pool kernel makes one pass over one
small grid.  The rows below are sized so that the plans of gemm_tcgen05.cu (make_plan) and of the pool launches (api.cu,
pool_*_inst.inc) pick the other schedules: tcgen05 tile loops (a CTA or CTA pair works through several tiles), CTA pairs with
an odd number of row blocks (a filler tile), split-K, the 192-wide side-output tiles, streaming pool forwards with more than
32 rows per warp, grid-stride pool backwards with several passes per CTA, the chunked folded backward, several queries per
sample, and sequence-first K/V with token offsets past 2^31 bytes.  Every case asserts the kernel string the library reports
(aecf_gemm_last_kernel / aecf_pool_last_kernel), so a change of plan cannot quietly turn a row into a copy of another.
The schedule arithmetic assumes 148 SMs: on any other device the file skips.
"""
import math
import re

import numpy as np
import pytest
import torch

import aecf_b200
from aecf_b200 import _lib, ops
from oracle import aecf_oracle as oracle
from oracle import philox
from tests.golden.cases import PHILOX_SEED
from tests.helpers import assert_close, finite_scale

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BF16_TOL = 2e-2
FP32_TOL = 1e-5


@pytest.fixture(autouse=True, scope="module")
def _b200_with_148_sms():
    if not torch.cuda.is_available() or torch.cuda.get_device_properties(0).multi_processor_count != 148:
        pytest.skip("the schedules below are worked out for the 148 SMs of a B200")


# ---------------------------------------------------------------------------------------------------------------------
# tcgen05 GEMM plans
# ---------------------------------------------------------------------------------------------------------------------
K, MN = _lib.K_MAJOR, _lib.MN_MAJOR
ALL_LAYOUTS = [(K, K), (K, MN), (MN, MN), (MN, K)]

# (m, n, k), the kernel GEMM_AUTO must report, and why the row is here
GEMM_PLANS = [
    ((128, 200, 72), "tcgen05 1sm bn128 cluster1 splits1", "one row block, ragged n and k"),
    ((128, 38920, 136), "tcgen05 1sm bn256 cluster1 splits1", "153 column tiles on 148 CTAs: tile loop without a cluster"),
    ((16384, 512, 512), "tcgen05 1sm bn256 cluster2 splits1", "128 tiles per 74 pairs: 2 tiles per pair"),
    ((12416, 512, 520), "tcgen05 2sm bn256 splits1", "97 row blocks (a filler tile), 9 k-blocks, 2 tiles per pair"),
    ((520, 512, 393216), "tcgen05 2sm bn256 splits12", "[dWv ; R] at B = 131 072: 5 row blocks, 12 splits of 512 k-blocks"),
    ((128, 512, 8160), "tcgen05 1sm bn256 cluster1 splits16", "split-K without a cluster, ragged k tail"),
    ((1000, 200, 4104), "tcgen05 1sm bn128 cluster2 splits8", "split-K on 128-wide tiles, ragged rows and k"),
]
SPLIT_K_ROWS = {shape for shape, kernel, _ in GEMM_PLANS if "splits1" not in kernel}


def _bf16_round_ulp(x: torch.Tensor) -> torch.Tensor:
    """One bf16 ulp at each element of x (x already bf16-representable)."""
    _, e = torch.frexp(x)
    return torch.ldexp(torch.ones_like(x), (e - 8).to(torch.int32)).clamp_min(2.0 ** -133)


def _gemm_ok(got: torch.Tensor, want: torch.Tensor, out_dtype, k: int) -> bool:
    """fp32 C: within 1e-5 of the tensor's scale for reductions up to k = 4096; beyond, the allowance grows like sqrt(k / 4096),
    as the rounding error of an fp32 accumulation does (k = 393 216 measured 4e-5 of the scale).  bf16 C: within one bf16
    ulp of the fp64 result rounded to bf16, plus the same fp32 allowance (an element far below the tensor's scale can carry
    more fp32 rounding than its own ulp)."""
    got, want = got.double(), want.double()
    fp32_budget = FP32_TOL * max(1.0, math.sqrt(k / 4096)) * float(want.abs().max())
    if out_dtype == torch.float32:
        return bool(((got - want).abs() <= fp32_budget).all())
    rounded = want.to(torch.bfloat16).double()
    return bool(((got - rounded).abs() <= _bf16_round_ulp(rounded) + fp32_budget).all())


def _operands(m, n, k, a_layout, b_layout, seed, extra_b_rows=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    a = torch.randn(m, k, device=DEV, generator=g).bfloat16()
    b = torch.randn(n + extra_b_rows, k, device=DEV, generator=g).bfloat16()
    bias = torch.randn(n, device=DEV, generator=g).bfloat16()
    a_mem = a if a_layout == K else a.t().contiguous()
    b_mem = b if b_layout == K else b.t().contiguous()
    return a, b, bias, a_mem, b_mem


def _sentinel_output(m, n, dtype):
    """C with ldc = n + 8 inside a buffer with 3 spare rows, all NaN: the kernel may write only C[:m, :n]."""
    buf = torch.full((m + 3, n + 8), float("nan"), device=DEV, dtype=dtype)
    return buf, n + 8


def _assert_sentinels(buf, m, n, what):
    assert bool(buf[:m, n:].isnan().all()), f"{what}: wrote past n into the ldc padding"
    assert bool(buf[m:].isnan().all()), f"{what}: wrote below row m"


@pytest.mark.parametrize("layouts", ALL_LAYOUTS, ids=["aK_bK", "aK_bMN", "aMN_bMN", "aMN_bK"])
@pytest.mark.parametrize("row", GEMM_PLANS, ids=lambda r: "x".join(map(str, r[0])))
def test_gemm_plan(row, layouts):
    (m, n, k), kernel, _ = row
    a_layout, b_layout = layouts
    a, b, bias, a_mem, b_mem = _operands(m, n, k, a_layout, b_layout, m + 3 * n + 7 * k)
    prod = a.double() @ b.double().t()
    lda, ldb = a_mem.shape[1], b_mem.shape[1]
    combos = [(torch.float32, None), (torch.bfloat16, bias)]
    if layouts == (K, K):
        combos += [(torch.float32, bias), (torch.bfloat16, None)]
    for out_dtype, use_bias in combos:
        what = f"{(m, n, k)} a={a_layout} b={b_layout} out={out_dtype} bias={use_bias is not None}"
        buf, ldc = _sentinel_output(m, n, out_dtype)
        ops.gemm(a_mem, b_mem, m=m, n=n, k=k, a_layout=a_layout, b_layout=b_layout, lda=lda, ldb=ldb, bias=use_bias,
                 out=buf, ldc=ldc)
        assert _lib.gemm_last_kernel() == kernel, (what, _lib.gemm_last_kernel())
        print(f"{what}: {_lib.gemm_last_kernel()}")
        torch.cuda.synchronize()
        want = prod + (use_bias.double() if use_bias is not None else 0.0)
        got = buf[:m, :n]
        assert torch.isfinite(got).all(), what
        assert _gemm_ok(got, want, out_dtype, k), f"{what}: max |err| {float((got.double() - want).abs().max()):.3e}"
        _assert_sentinels(buf, m, n, what)
        if (m, n, k) in SPLIT_K_ROWS:
            # the bound is tight enough to see one missing 64-wide k-block (a split's partial dropped or doubled)
            kb = (k // 64) // 2
            dropped = want - a[:, kb * 64:(kb + 1) * 64].double() @ b[:, kb * 64:(kb + 1) * 64].double().t()
            assert not _gemm_ok(got, dropped, out_dtype, k), f"{what}: the check cannot see a missing k-block"


# aecf_gemm_aux: 192-wide tiles with the fp32 side output; B is K-major by contract
AUX_PLANS = [((128, 1280, 960), aux, "tcgen05 1sm bn192 cluster1 splits1") for aux in (5, 12, 20, 32)] + [
    ((12416, 512, 520), aux, "tcgen05 1sm bn192 cluster2 splits1") for aux in (5, 12, 32)] + [
    ((49152, 1280, 1280), 20, "tcgen05 1sm bn192 cluster2 splits1")]     # 1344 tiles on 74 pairs: up to 19 per pair


@pytest.mark.parametrize("row", AUX_PLANS, ids=lambda r: "x".join(map(str, r[0])) + f"_aux{r[1]}")
def test_gemm_side_output_plan(row):
    (m, n, k), aux, kernel = row
    aux_rows = (aux + 7) // 8 * 8
    a, b, bias, _, _ = _operands(m, n, k, K, K, m + n + aux, extra_b_rows=aux_rows)
    b[n + aux:] = 0
    prod = a.double() @ b.double().t()
    for out_dtype, use_bias in ((torch.float32, None), (torch.bfloat16, bias), (torch.float32, bias), (torch.bfloat16, None)):
        what = f"{(m, n, k)} aux={aux} out={out_dtype} bias={use_bias is not None}"
        c, side = ops.gemm_aux(a, b, m=m, n=n, k=k, aux_cols=aux, bias=use_bias, out_dtype=out_dtype)
        assert _lib.gemm_last_kernel() == kernel, (what, _lib.gemm_last_kernel())
        print(f"{what}: {_lib.gemm_last_kernel()}")
        torch.cuda.synchronize()
        want = prod[:, :n] + (use_bias.double() if use_bias is not None else 0.0)
        assert _gemm_ok(c, want, out_dtype, k), f"{what}: C, max |err| {float((c.double() - want).abs().max()):.3e}"
        assert _gemm_ok(side[:, :aux], prod[:, n:n + aux], torch.float32, k), f"{what}: side output"
        assert float(side[:, aux:].abs().max()) == 0.0 if side.shape[1] > aux else True


@pytest.mark.parametrize("shape", [(200, 136, 256), (200, 136, 4096)], ids=["direct", "split_k"])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_gemm_accumulate(shape, out_dtype):
    """accumulate = 1 (C += A B^T + bias) runs on the SIMT kernel, directly and through the split-K reduce; the tcgen05
    kernels do not take it."""
    m, n, k = shape
    a, b, bias, _, _ = _operands(m, n, k, K, K, 17 + k)
    c0 = torch.randn(m, n, device=DEV).to(out_dtype)
    for use_bias in (None, bias):
        buf, ldc = _sentinel_output(m, n, out_dtype)
        buf[:m, :n] = c0
        ops.gemm(a, b, m=m, n=n, k=k, a_layout=K, b_layout=K, lda=k, ldb=k, bias=use_bias, out=buf, ldc=ldc, accumulate=True)
        assert _lib.gemm_last_kernel() == "simt"
        torch.cuda.synchronize()
        want = c0.double() + a.double() @ b.double().t() + (use_bias.double() if use_bias is not None else 0.0)
        assert _gemm_ok(buf[:m, :n], want, out_dtype, k), f"accumulate {shape} {out_dtype} bias={use_bias is not None}"
        _assert_sentinels(buf, m, n, "accumulate")
        assert not _gemm_ok(buf[:m, :n], want - c0.double(), out_dtype, k), "the check cannot tell accumulate from overwrite"
    with pytest.raises(_lib.UnsupportedShapeError):
        ops.gemm(a, b, m=m, n=n, k=k, a_layout=K, b_layout=K, lda=k, ldb=k, out=buf, ldc=ldc, accumulate=True,
                 impl=_lib.GEMM_TCGEN05)


# ---------------------------------------------------------------------------------------------------------------------
# pool schedules: whole training steps through the module API against the stage-rounded oracle
# ---------------------------------------------------------------------------------------------------------------------
def _inputs(B, M, D, H, *, S=1, seed, dtype, separate_value=False, per_row_query=False, offset=0, row0=0, device="cpu"):
    """Parameters and data drawn with torch.randn on the GPU, rounded to the storage dtype, returned as fp32 on `device`
    (the CPU for the oracle); attention made peaked along one direction as tests/golden/cases.py does, so that keep_prob
    really depends on the entropy; the Philox uniforms of the kernels' draws."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    rnd = lambda *shape: torch.randn(*shape, device=DEV, generator=g)        # noqa: E731
    Wi, bi = rnd(3 * D, D) * math.sqrt(2.0 / (4 * D)), rnd(3 * D) * 0.05
    Wo, bo = rnd(D, D) / math.sqrt(D), rnd(D) * 0.05
    q0 = rnd(1, 1, D) * math.sqrt(2.0 / D)
    direction = Wi[D:2 * D].t() @ (q0.reshape(D) @ Wi[:D].t() + bi[:D])
    per_unit = float(direction.norm()) / (H * math.sqrt(D // H))
    x = rnd(B, M, D) + rnd(B, M, 1) * (2.0 / per_unit) * (direction / direction.norm())
    inp = {"in_proj_weight": Wi, "in_proj_bias": bi, "out_proj.weight": Wo, "out_proj.bias": bo, "query0": q0, "x": x,
           "grad_out": rnd(B, S, D), "grad_pooled": rnd(B, S, M)}
    if separate_value:
        inp["value"] = rnd(B, M, D)
    if per_row_query or S > 1:
        inp["query"] = q0 + rnd(B, S, D) * math.sqrt(2.0 / D)
    for k_ in inp:
        if k_ != "grad_pooled":
            inp[k_] = inp[k_].to(dtype).float()
        inp[k_] = inp[k_].to(device)
    inp["u_mask"] = torch.from_numpy(philox.mask_uniforms(PHILOX_SEED, offset, row0 * S, B * S, M)).reshape(B, S, M)
    inp["u_drop"] = torch.from_numpy(np.ascontiguousarray(
        philox.dropout_uniforms(PHILOX_SEED, offset, row0 * S, B * S, H, M).reshape(B, S, H, M).transpose(0, 2, 1, 3)))
    return inp


def _run_module(inp, H, dtype, *, fold, dropout, offset=0, row0=0, seq_first=False):
    """One training step (forward with return_info, entropy_loss, backward of out . grad_out + pooled . grad_pooled).
    Returns the results and the pool kernel strings of the forward and (read on autograd's thread) the backward."""
    B, M, D = inp["x"].shape
    S = inp["grad_out"].shape[1]
    cm = aecf_b200.CurriculumMasking(base_mask_prob=0.15, entropy_target=0.7, min_active=1)
    pool = aecf_b200.MultimodalAttentionPool(D, num_heads=H, dropout=dropout, curriculum_masking=cm, device=DEV, dtype=dtype)
    with torch.no_grad():
        pool.attention.in_proj_weight.copy_(inp["in_proj_weight"])
        pool.attention.in_proj_bias.copy_(inp["in_proj_bias"])
        pool.attention.out_proj.weight.copy_(inp["out_proj.weight"])
        pool.attention.out_proj.bias.copy_(inp["out_proj.bias"])
    pool.train(True)
    pool.row_offset = row0
    pool._want_mask_bits = True
    pool.fold_key_projection = fold
    pool.batch_first = not seq_first
    per_row = "query" in inp
    query = torch.nn.Parameter((inp["query"] if per_row else inp["query0"]).to(DEV, dtype))
    x = inp["x"].to(DEV, dtype)
    value = inp["value"].to(DEV, dtype) if "value" in inp else None
    if seq_first:
        x = x.transpose(0, 1).contiguous()
        value = value.transpose(0, 1).contiguous() if value is not None else None
    x.requires_grad_(True)
    if value is not None:
        value.requires_grad_(True)
    q_in = query if per_row else query.expand(B, -1, -1)
    if seq_first:
        q_in = q_in.transpose(0, 1)
    seen = {}

    def note_backward_kernel(grad):         # runs on autograd's thread, right after the fused backward produced d x
        seen.setdefault("bwd", _lib.pool_last_kernel())

    x.register_hook(note_backward_kernel)
    aecf_b200.set_rng_state(PHILOX_SEED, offset)
    try:
        out, info = pool(q_in, x, value, return_info=True)
        seen["fwd"] = _lib.pool_last_kernel()
        ent_loss = cm.entropy_loss(info["entropy"])
    finally:
        aecf_b200.set_rng_state(None)
    if seq_first:
        out = out.transpose(0, 1)
    loss = (out.float() * inp["grad_out"].to(DEV)).sum() + (info["attention_weights"].reshape(B, S, M)
                                                              * inp["grad_pooled"].to(DEV)).sum()
    loss.backward()
    torch.cuda.synchronize()
    grads = {"key": x.grad.transpose(0, 1) if seq_first else x.grad, "query": query.grad,
             "in_proj_weight": pool.attention.in_proj_weight.grad, "in_proj_bias": pool.attention.in_proj_bias.grad,
             "out_proj.weight": pool.attention.out_proj.weight.grad, "out_proj.bias": pool.attention.out_proj.bias.grad}
    if value is not None:
        grads["value"] = value.grad.transpose(0, 1) if seq_first else value.grad
    return out, info, ent_loss, grads, seen


def _run_oracle(inp, H, *, storage, fold_key, dropout):
    B, M, D = inp["x"].shape
    S = inp["grad_out"].shape[1]
    per_row = "query" in inp
    q = inp["query"] if per_row else inp["query0"].expand(B, 1, D)
    u_mask = inp["u_mask"] if S > 1 else inp["u_mask"].reshape(B, M)
    u_drop = inp["u_drop"] if S > 1 else inp["u_drop"].reshape(B, H, M)
    fwd = oracle.pool_forward(q, inp["x"], inp.get("value"), inp["in_proj_weight"], inp["in_proj_bias"],
                              inp["out_proj.weight"], inp["out_proj.bias"], H, dropout_p=dropout, training=True,
                              u_drop=u_drop, u_mask=u_mask, masking=dict(base_mask_prob=0.15, entropy_target=0.7, min_active=1),
                              storage=storage, fold_key=fold_key, per_row_query_storage=per_row)
    grads = oracle.pool_backward(q, inp["x"], inp.get("value"), inp["in_proj_weight"], inp["out_proj.weight"], H, fwd.saved,
                                 inp["grad_out"], grad_pooled=inp["grad_pooled"], dropout_p=dropout, training=True,
                                 storage=storage, fold_key=fold_key, per_row_query_storage=per_row)
    if not per_row:
        grads["query"] = grads["query"].sum(0, keepdim=True)
    return fwd, grads


def _rowwise(name, got, want, rows, tol):
    """Every row within tol of its own scale (plus tol of the median row scale), so no small row hides behind a large one."""
    got, want = got.float().cpu().reshape(rows, -1).double(), want.reshape(rows, -1).double()
    err = (got - want).abs().amax(1)
    scale = want.abs().amax(1)
    bad = err > tol * scale + tol * float(scale.median())
    assert not bool(bad.any()), f"{name}: {int(bad.sum())} rows off, first {int(bad.nonzero()[0])}, worst {float((err / scale).max()):.3e}"


def _check(inp, H, dtype, res, ref, folded):
    out, info, ent_loss, grads, _ = res
    fwd, ref_grads = ref
    B, M, D = inp["x"].shape
    S = inp["grad_out"].shape[1]
    rows = B * S
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    bits = ((fwd.info["mask"].reshape(rows, M) > 0).numpy() * (1 << np.arange(M))).sum(1).astype(np.uint8)
    assert np.array_equal(info["mask_bits"].reshape(-1).cpu().numpy(), bits), "mask bits differ"
    assert torch.equal(info["mask_rate"].reshape(-1).cpu(), fwd.info["mask_rate"].reshape(-1).float()), "mask_rate differs"
    # The unfolded bf16 path stores K in bf16: where the kernel's and the oracle's fp32 projections round a K element to
    # neighbouring bf16 values, the weights move by ~1e-4 (B = 131 109 measured 1.3e-4 on a few dozen rows).  The folded
    # path keeps its scores in fp32.
    aw_tol, aw_atol = (FP32_TOL, 1e-5) if dtype == torch.float32 else (1e-4, 1e-5) if folded else (1e-3, 2e-4)
    assert_close("attention_weights", info["attention_weights"].cpu(), fwd.info["attention_weights"], aw_tol, atol=aw_atol)
    assert_close("masked_attention_weights", info["masked_attention_weights"].cpu(), fwd.info["masked_attention_weights"],
                 aw_tol, atol=aw_atol)
    assert_close("entropy", info["entropy"].cpu(), fwd.info["entropy"], aw_tol, atol=aw_atol)
    assert_close("entropy_loss", ent_loss.cpu(), oracle.entropy_loss(fwd.info["entropy"], M, 0.7), aw_tol)
    _rowwise("out", out, fwd.out, rows, tol)
    _rowwise("grad key", grads["key"], ref_grads["key"], B * M, tol)
    if "value" in grads:
        _rowwise("grad value", grads["value"], ref_grads["value"], B * M, tol)
    if "query" in inp:
        _rowwise("grad query", grads["query"], ref_grads["query"], rows, tol)
    else:
        assert_close("grad query0", grads["query"].float().cpu(), ref_grads["query"], tol)
    # batch sums (the grid-stride backward's partials and their finalize, the weight-gradient products)
    for k_ in ("out_proj.bias", "out_proj.weight", "in_proj_weight"):
        assert_close(f"grad {k_}", grads[k_].float().cpu(), ref_grads[k_], tol)
    assert_close("grad in_proj_bias", grads["in_proj_bias"].float().cpu(), ref_grads["in_proj_bias"], tol,
                 atol=tol * finite_scale(ref_grads["in_proj_bias"]))


# name: (B, M, D, H, dict(options), forward kernel pattern, backward kernel pattern, schedule condition)
POOL_PLANS = {
    # 131 109 rows on 148 x 24 warps: 37 rows per warp (a partial second 32-row group), the last CTA partly idle
    "folded_b131109_d512_m3": (131109, 3, 512, 8, dict(fold=True),
                               r"dense stream M=3 J=2 PAD=0 fold=1 warps=24 rows_per_warp=37 ctas=148",
                               r"bwd chunked M=3 J=2 PAD=0 fold=1 grid=8195 chunk=16", None),
    "unfolded_b131109_d512_m3": (131109, 3, 512, 8, dict(fold=False),
                                 r"stream M=3 J=2 PAD=0 fold=0 warps=16 rows_per_warp=56 ctas=147",
                                 r"bwd grid-stride M=3 J=2 PAD=0 fold=0 grid=(\d+) passes=(\d+)", "passes"),
    # 32 KB rings: 6 warps per CTA, 33 rows per warp
    "unfolded_b28417_d512_m8": (28417, 8, 512, 8, dict(fold=False),
                                r"stream M=8 J=2 PAD=0 fold=0 warps=6 rows_per_warp=33 ctas=144",
                                r"bwd grid-stride M=8 J=2 PAD=0 fold=0 grid=(\d+) passes=(\d+)", "passes"),
    # one head of 1024 (J = 4): the README's head_dim table
    "folded_b64_d1024_h1": (64, 3, 1024, 1, dict(fold=True), r"dense stream M=3 J=4 PAD=0 fold=1 warps=16 rows_per_warp=1 ctas=4",
                            r"bwd chunked M=3 J=4 PAD=0 fold=1 grid=4 chunk=16", None),
    "folded_b65536_d1024_h1": (65536, 3, 1024, 1, dict(fold=True),
                               r"dense stream M=3 J=4 PAD=0 fold=1 warps=16 rows_per_warp=28 ctas=147",
                               r"bwd chunked M=3 J=4 PAD=0 fold=1 grid=4096 chunk=16", None),
    "unfolded_b64_d1024_h1": (64, 3, 1024, 1, dict(fold=False), r"stream M=3 J=4 PAD=0 fold=0 warps=8 rows_per_warp=1 ctas=8",
                              r"bwd grid-stride M=3 J=4 PAD=0 fold=0 grid=(\d+) passes=(\d+)", None),
    "unfolded_b65536_d1024_h1": (65536, 3, 1024, 1, dict(fold=False),
                                 r"stream M=3 J=4 PAD=0 fold=0 warps=8 rows_per_warp=56 ctas=147",
                                 r"bwd grid-stride M=3 J=4 PAD=0 fold=0 grid=(\d+) passes=(\d+)", "passes"),
    # grid-stride backward, several passes per CTA, in each of its modes
    "fp32_b65539_d512": (65539, 3, 512, 8, dict(fold=False, dtype=torch.float32), r"slice M=3 J=2 PAD=0 fold=0 grid=16385",
                         r"bwd grid-stride M=3 J=2 PAD=0 fold=0 grid=(\d+) passes=(\d+)", "passes"),
    "per_row_query_b65539_d512": (65539, 3, 512, 8, dict(fold=False, per_row_query=True, dropout=0.1),
                                  r"stream M=3 J=2 PAD=0 fold=0 warps=16 rows_per_warp=28 ctas=147",
                                  r"bwd grid-stride M=3 J=2 PAD=0 fold=0 grid=(\d+) passes=(\d+)", "passes"),
    "separate_value_b65539_d512": (65539, 3, 512, 8, dict(fold=None, separate_value=True),
                                   r"stream M=3 J=2 PAD=0 fold=0 warps=16 rows_per_warp=28 ctas=147",
                                   r"bwd grid-stride M=3 J=2 PAD=0 fold=0 grid=(\d+) passes=(\d+)", "passes"),
    # chunked folded backward with B not a multiple of the chunk; with dropout it hands per-sample sums to the tail
    "chunked_b65541": (65541, 3, 512, 8, dict(fold=True), r"dense stream M=3 J=2 PAD=0 fold=1 warps=24 rows_per_warp=19 ctas=144",
                       r"bwd chunked M=3 J=2 PAD=0 fold=1 grid=4097 chunk=16", None),
    "chunked_b65541_dropout": (65541, 3, 512, 8, dict(fold=True, dropout=0.1, offset=3, row0=4096),
                               r"dense stream M=3 J=2 PAD=0 fold=1 warps=24 rows_per_warp=19 ctas=144",
                               r"bwd chunked M=3 J=2 PAD=0 fold=1 grid=4097 chunk=16", None),
    # two queries per sample: 28 passes of the one-CTA-per-SM backward
    "multi_query_s2_b32771": (32771, 3, 512, 8, dict(fold=False, S=2, dropout=0.1), r"multi fwd M=3 J=2 PAD=0 grid=8193",
                              r"multi bwd M=3 J=2 PAD=0 fold=0 grid=148 passes=28", None),
}


@pytest.mark.parametrize("name", list(POOL_PLANS))
def test_pool_schedule_against_oracle(name):
    B, M, D, H, opt, fwd_kernel, bwd_kernel, condition = POOL_PLANS[name]
    dtype = opt.get("dtype", torch.bfloat16)
    dropout = opt.get("dropout", 0.0)
    offset, row0 = opt.get("offset", 0), opt.get("row0", 0)
    inp = _inputs(B, M, D, H, S=opt.get("S", 1), seed=B + M + D, dtype=dtype, separate_value=opt.get("separate_value", False),
                  per_row_query=opt.get("per_row_query", False), offset=offset, row0=row0)
    res = _run_module(inp, H, dtype, fold=opt["fold"], dropout=dropout, offset=offset, row0=row0)
    seen = res[4]
    print(f"{name}: forward {seen['fwd']} | backward {seen['bwd']}")
    assert re.fullmatch(fwd_kernel, seen["fwd"]), seen["fwd"]
    match = re.fullmatch(bwd_kernel, seen["bwd"])
    assert match, seen["bwd"]
    if condition == "passes":
        assert int(match.group(2)) >= 2, f"{seen['bwd']}: one pass per CTA, the grid-stride loop is not exercised"
    folded = opt["fold"] is not False and dtype == torch.bfloat16 and "value" not in inp and "query" not in inp
    storage = torch.bfloat16 if dtype == torch.bfloat16 else None
    ref = _run_oracle(inp, H, storage=storage, fold_key=folded, dropout=dropout)
    _check(inp, H, dtype, res, ref, folded)


# Sequence-first K/V at B = 98 304: the token stride is B * 2D (unfolded) or B rows of D (folded) elements, 402 MB, so tokens
# 6 and 7 of every sample sit past 2^31 bytes from token 0.  The same step batch-first must give the same bits.
SEQ_FIRST = {
    "unfolded_m8_d1024_h8": (98304, 8, 1024, 8, False, r"slice M=8 J=2 PAD=0 fold=0 grid=24576",
                             r"bwd grid-stride M=8 J=2 PAD=0 fold=0 grid=(\d+) passes=(\d+)"),
    "folded_m8_d2048_h16": (98304, 8, 2048, 16, True, r"slice M=8 J=2 PAD=0 fold=1 grid=\d+",
                            r"bwd chunked M=8 J=2 PAD=0 fold=1 grid=\d+ chunk=\d+"),
}


@pytest.mark.parametrize("name", list(SEQ_FIRST))
def test_sequence_first_past_2gb_matches_batch_first(name):
    B, M, D, H, fold, fwd_kernel, bwd_kernel = SEQ_FIRST[name]
    assert (M - 2) * B * (2 if not fold else 1) * D * 2 >= 2 ** 31
    inp = _inputs(B, M, D, H, seed=7, dtype=torch.bfloat16, device=DEV)       # no oracle here: the data stays on the GPU
    runs = {}
    for seq_first in (False, True):
        out, info, _, grads, seen = _run_module(inp, H, torch.bfloat16, fold=fold, dropout=0.1, offset=2, seq_first=seq_first)
        print(f"{name} {'sequence' if seq_first else 'batch'}-first: forward {seen['fwd']} | backward {seen['bwd']}")
        assert re.fullmatch(fwd_kernel, seen["fwd"]), seen["fwd"]
        assert re.fullmatch(bwd_kernel, seen["bwd"]), seen["bwd"]
        runs[seq_first] = (out.reshape(B, D), info, grads)
    (ob, ib, gb), (os_, is_, gs) = runs[False], runs[True]
    assert torch.equal(ob, os_), "out differs between the layouts"
    for k_ in ("attention_weights", "mask_bits", "entropy", "masked_attention_weights"):
        assert torch.equal(ib[k_].reshape(B, -1), is_[k_].reshape(B, -1)), f"{k_} differs between the layouts"
    assert torch.equal(gb["key"], gs["key"]), "grad key differs between the layouts"
    for k_ in ("in_proj_weight", "in_proj_bias", "out_proj.weight", "query"):   # batch sums: the row order may differ
        assert_close(f"grad {k_}", gs[k_].float().cpu(), gb[k_].float().cpu(), 1e-2)
