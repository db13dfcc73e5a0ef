"""Rows where the reference itself produces -inf scores, NaN weights and NaN gradients, against the oracle (fp64 / autograd
where noted) with tests/helpers.py::assert_close, which requires NaN and +-inf exactly where the reference has them.

- A fully padded sample (key_padding_mask all True) has softmax(-inf, ..., -inf) = NaN: torch returns NaN for its output,
  its attention weights and every gradient it touches -- the batch sums over samples (weight and bias gradients) are NaN
  as a whole.  The other samples must be unaffected, in their outputs and in their input gradients.
- The eval-mode entropy -sum xlogy(p, p) has the gradient 0 / 0 = NaN at p = 0 in torch (a padded token).
- The small stand-alone kernels at the edges of their launch geometry.

tests/test_emu_nonfinite.py runs the same bodies on the host emulation.
"""
import dataclasses
import math

import numpy as np
import pytest
import torch

import aecf_b200
from aecf_b200 import ops
from oracle import aecf_oracle as oracle
from oracle import philox
from tests import test_gpu_multi_query as MQ
from tests import test_gpu_parity as P
from tests.golden.cases import CASES_BY_NAME, MULTI_QUERY_CASES, PHILOX_SEED, Case, build_inputs
from tests.helpers import assert_close, finite_scale, run_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FP32_TOL = 1e-5
BF16_TOL = 2e-2

# Which samples are padded: the first, several, and the first / last sample of a backward CTA's chunk of 16 samples
# (POOL_BWD_CHUNK) -- with B = 32 that is both chunk boundaries and the batch's last sample.
PADDINGS = {"first": [0], "several": [0, 5, 6, 21], "chunk_edges": [15, 16, 31]}
# (training, d_pooled): the training step, with the attention-weights gradient, and eval mode, where info['entropy']
# keeps its graph and the loss takes 0.5 * its sum too
MODES = {"train": (True, False), "train_dpooled": (True, True), "eval_dpooled": (False, True)}


def padded_case(pad, mode):
    training, pooled_grad = MODES[mode]
    return dataclasses.replace(CASES_BY_NAME["d64_h4_m4_kpm"], training=training, pooled_grad=pooled_grad,
                               name=f"d64_h4_m4_kpm_pad_{pad}_{mode}")


def padded_inputs(case, rows, bf16=False):
    inp = P._bf16_inputs(case) if bf16 else build_inputs(case)
    inp["key_padding_mask"][rows, :] = True
    return inp


def check_padded_run(case, rows, kpm, out, info, ent_loss, grads, ref, ref_grads, tol):
    B, M = case.B, case.M
    # the oracle's own pattern: NaN in the padded samples' outputs and weights, nowhere else
    bad = torch.zeros(B, dtype=torch.bool)
    bad[rows] = True
    assert bool(torch.isnan(ref.out.reshape(B, -1)[bad]).all()) and bool(torch.isfinite(ref.out.reshape(B, -1)[~bad]).all())
    assert_close("out", out.float().cpu(), ref.out, tol)
    assert_close("attention_weights", info["attention_weights"].cpu(), ref.info["attention_weights"], tol, atol=tol)
    assert_close("entropy", info["entropy"].cpu(), ref.info["entropy"], tol, atol=tol * math.log(M))
    assert_close("masked_attention_weights", info["masked_attention_weights"].cpu(), ref.info["masked_attention_weights"],
                 tol, atol=tol)
    assert torch.equal(info["mask_rate"].cpu(), ref.info["mask_rate"].float()), "mask_rate differs"
    assert np.array_equal(info["mask_bits"].cpu().numpy(), P.expected_bits(ref.info["mask"])), "mask bits differ"
    last = M if case.training else 2
    assert_close("entropy_loss", ent_loss.float().cpu(), oracle.entropy_loss(ref.info["entropy"], last, case.entropy_target),
                 tol, atol=tol)
    for name in ("key", "query0", "out_proj.bias", "out_proj.weight", "in_proj_weight"):
        assert_close(f"grad {name}", grads[name].float().cpu(), ref_grads[name], tol)
    assert_close("grad in_proj_bias", grads["in_proj_bias"].float().cpu(), ref_grads["in_proj_bias"], tol,
                 atol=tol * finite_scale(ref_grads["in_proj_bias"]))
    # a padded sample leaks into no other row: the other samples' input gradients are finite, except in eval mode where
    # a padded token (pooled weight 0) gives its own sample the NaN of the entropy gradient
    gx = grads["key"].float().cpu().reshape(B, -1)
    nan_rows = kpm.any(1) if not case.training else bad
    assert bool(torch.isfinite(gx[~nan_rows]).all()) and bool(torch.isnan(gx[bad]).all())


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("pad", list(PADDINGS))
@pytest.mark.parametrize("fold", [False, True], ids=["unfolded", "folded"])
def test_fp32_fully_padded_samples(pad, mode, fold):
    case = padded_case(pad, mode)
    inp = padded_inputs(case, PADDINGS[pad])
    ref, ref_grads = run_oracle(case, inp)
    out, info, ent_loss, grads, _ = P.run_cuda(case, inp, torch.float32, fold=fold)
    check_padded_run(case, PADDINGS[pad], inp["key_padding_mask"], out, info, ent_loss, grads, ref, ref_grads, FP32_TOL)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("pad", ["several", "chunk_edges"])
@pytest.mark.parametrize("fold", [False, True], ids=["unfolded", "folded"])
def test_bf16_fully_padded_samples(pad, mode, fold):
    """Against the oracle that rounds to bf16 where the CUDA path stores bf16 (folded like it)."""
    case = padded_case(pad, mode)
    inp = padded_inputs(case, PADDINGS[pad], bf16=True)
    ref, ref_grads = run_oracle(case, inp, storage=torch.bfloat16, fold_key=fold)
    out, info, ent_loss, grads, _ = P.run_cuda(case, inp, torch.bfloat16, fold=fold)
    check_padded_run(case, PADDINGS[pad], inp["key_padding_mask"], out, info, ent_loss, grads, ref, ref_grads, BF16_TOL)


def test_fully_padded_sample_leaves_the_others_key_gradients_alone():
    """d64_h4_m4_kpm, one fully padded sample, fp32, folded: every other sample's d key equals the oracle's."""
    case = dataclasses.replace(CASES_BY_NAME["d64_h4_m4_kpm"], pooled_grad=True, name="d64_h4_m4_kpm_pad0")
    inp = padded_inputs(case, [0])
    _, ref_grads = run_oracle(case, inp)
    for fold in (False, True, True):                 # the second folded run: nothing carries over from an earlier call
        grads = P.run_cuda(case, inp, torch.float32, fold=fold)[3]
        got, want = grads["key"].cpu().reshape(case.B, -1), ref_grads["key"].reshape(case.B, -1)
        assert bool(torch.isnan(got[0]).all())
        assert_close(f"d key of samples 1.. (fold={fold})", got[1:], want[1:], FP32_TOL)


# ---- several queries per sample (csrc/pool_multi.cuh), batch-first and sequence-first -------------------------------
MQ_PADDED = [dataclasses.replace(MULTI_QUERY_CASES[2], name="s2_d64_h4_m4_kpm_eval_pad"),
             dataclasses.replace(MULTI_QUERY_CASES[2], training=True, dropout=0.1, name="s2_d64_h4_m4_kpm_train_pad")]


@pytest.mark.parametrize("batch_first", [True, False], ids=["batch_first", "seq_first"])
@pytest.mark.parametrize("case", MQ_PADDED, ids=lambda c: c.name)
def test_multi_query_fully_padded_samples(case, batch_first):
    inp = build_inputs(case)
    inp["key_padding_mask"][[0, 7, case.B - 1], :] = True
    ref, ref_grads = run_oracle(case, inp)
    assert bool(torch.isnan(ref.out[0]).all()) and bool(torch.isfinite(ref.out[1]).all())
    out, info, ent_loss, grads, _ = MQ.run_cuda(case, inp, torch.float32, batch_first=batch_first)
    MQ.check_against_oracle(case, out, info, ent_loss, grads, ref, ref_grads, FP32_TOL)


@pytest.mark.parametrize("case", MQ_PADDED, ids=lambda c: c.name)
def test_multi_query_bf16_fully_padded_samples(case):
    inp = build_inputs(case)
    for k in ("in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias", "query", "x", "grad_out"):
        inp[k] = inp[k].bfloat16().float()
    inp["key_padding_mask"][[0, 7, case.B - 1], :] = True
    ref, ref_grads = run_oracle(case, inp, storage=torch.bfloat16)
    out, info, _, grads, _ = MQ.run_cuda(case, inp, torch.bfloat16)
    assert np.array_equal(info["mask_bits"].cpu().numpy().reshape(-1), MQ.expected_bits(ref.info["mask"]))
    assert torch.equal(info["mask_rate"].cpu(), ref.info["mask_rate"].float())
    assert_close("attention_weights", info["attention_weights"].cpu(), ref.info["attention_weights"], 1e-4, atol=1e-5)
    assert_close("entropy", info["entropy"].cpu(), ref.info["entropy"], 1e-4, atol=1e-5)
    assert_close("out", out.float().cpu(), ref.out, 1e-2)
    for name in ("key", "query", "in_proj_weight", "out_proj.weight"):
        assert_close(f"grad {name}", grads[name].float().cpu(), ref_grads[name], BF16_TOL)


# ---- sample_index: a non-finite sample among the listed rows and one among the others ----------------------------------
@pytest.mark.parametrize("dtype,fold", [(torch.float32, False), (torch.float32, True), (torch.bfloat16, True)],
                         ids=["fp32_unfolded", "fp32_folded", "bf16_folded"])
def test_sample_index_with_non_finite_samples(dtype, fold):
    """pool(x, sample_index=idx) against pool(x[idx]): a listed sample with an infinite token gives the NaN the gathered
    call gives, bit for bit, and an unlisted one with NaN tokens changes nothing -- every gradient stays as without it."""
    case = CASES_BY_NAME["d64_h8_m3_dropout"]
    inp = build_inputs(case)
    B = case.B
    idx = torch.tensor([b for b in range(B) if (b * 7 + 3) % 5 not in (0, 1)])
    listed, unlisted = int(idx[4]), next(b for b in range(B) if b not in set(idx.tolist()))
    inp["x"][listed, 1, :] = float("inf")
    inp["x"][unlisted] = float("nan")
    runs = {}
    for mode in ("gathered", "in_place"):
        pool, _ = P.make_pool(case, inp, dtype, fold)
        q = torch.nn.Parameter(inp["query0"].to(DEV, dtype))
        x = inp["x"].to(DEV, dtype).requires_grad_(True)
        g = inp["grad_out"].to(DEV, dtype)[idx.to(DEV)].float()
        aecf_b200.set_rng_state(PHILOX_SEED, case.offset)
        if mode == "gathered":
            out, info = pool(q.expand(idx.numel(), -1, -1), x[idx.to(DEV)], return_info=True)
        else:
            out, info = pool(q.expand(B, -1, -1), x, return_info=True, sample_index=idx.to(DEV))
            out = out[idx.to(DEV)]
        aecf_b200.set_rng_state(None)
        ((out.float() * g).sum() + (info["attention_weights"] * 0.3).sum()).backward()
        runs[mode] = dict(out=out.detach(), gx=x.grad[idx.to(DEV)], gw=pool.attention.in_proj_weight.grad,
                          gb=pool.attention.in_proj_bias.grad, gwo=pool.attention.out_proj.weight.grad, gq=q.grad,
                          **{k: v.detach() for k, v in info.items()}, others=x.grad[unlisted])
    a, b = runs["gathered"], runs["in_place"]
    row = int((idx == listed).nonzero())
    assert bool(torch.isnan(a["out"][row]).all()) and bool(torch.isfinite(a["out"][:row]).all())
    for k in ("out", "gx", "attention_weights", "entropy", "mask_rate", "masked_attention_weights", "mask_bits"):
        assert_close(k, b[k].float().cpu(), a[k].float().cpu(), 0.0, atol=0.0)
    assert float(b["others"].abs().max()) == 0.0
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    for k in ("gw", "gb", "gwo", "gq"):
        assert_close(k, b[k].float().cpu(), a[k].float().cpu(), tol)


# ---- the eval-mode entropy gradient at zero weights ---------------------------------------------------------------------
# S = 1 twin of s2_d64_h4_m4_kpm_eval: padded tokens have pooled weight 0, where torch's d entropy / d p is NaN
EVAL_KPM = Case("d64_h4_m4_kpm_eval", B=12, M=4, D=64, H=4, kpm=True, training=False, pooled_grad=True, data_seed=25)


@pytest.mark.parametrize("fold", [False, True], ids=["unfolded", "folded"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_eval_entropy_gradient_at_padded_tokens(dtype, fold):
    case = EVAL_KPM
    bf16 = dtype == torch.bfloat16
    inp = P._bf16_inputs(case) if bf16 else build_inputs(case)
    assert bool(inp["key_padding_mask"].any(1).any()) and not bool(inp["key_padding_mask"].all(1).any())
    ref, ref_grads = run_oracle(case, inp, storage=torch.bfloat16 if bf16 else None, fold_key=fold and bf16)
    assert bool(torch.isnan(ref_grads["key"]).any())        # the case does reach the NaN of the entropy gradient
    out, info, ent_loss, grads, _ = P.run_cuda(case, inp, dtype, fold=fold)
    tol = BF16_TOL if bf16 else FP32_TOL
    assert_close("out", out.float().cpu(), ref.out, tol)
    assert_close("entropy", info["entropy"].cpu(), ref.info["entropy"], 1e-4 if bf16 else tol, atol=1e-5)
    for name in ("key", "query0", "out_proj.bias", "out_proj.weight", "in_proj_weight"):
        assert_close(f"grad {name}", grads[name].float().cpu(), ref_grads[name], tol)
    assert_close("grad in_proj_bias", grads["in_proj_bias"].float().cpu(), ref_grads["in_proj_bias"], tol,
                 atol=tol * finite_scale(ref_grads["in_proj_bias"]))


def _weights_with_zeros():
    w = torch.softmax(2 * torch.from_numpy(philox.normal(31, (64, 6))).float(), -1)
    w[::3, 1] = 0.0                                   # zero weights in normalised rows
    w[::3] /= w[::3].sum(-1, keepdim=True)
    w[1] = torch.tensor([1.0, 0.0, 0.0, 0.0, 0.0, 0.0])       # entropy 0: at the lower end of the clamp
    w[2] = 1.0 / 6                                             # the upper end
    w[4::5] *= 3.0                                             # unnormalised: the clamp saturates
    w[5, 2] = 0.0                                              # ... with a zero weight
    return w


def test_standalone_entropy_gradient_at_zero_weights():
    """CurriculumMasking in eval mode and compute_entropy: d entropy / d w against autograd of torch's own formula."""
    w = _weights_with_zeros()
    g = torch.from_numpy(philox.normal(32, (64,))).float()
    wr = w.clone().requires_grad_(True)
    (oracle.shannon_entropy(wr) * g).sum().backward()
    assert bool(torch.isnan(wr.grad[0]).any()) and bool(torch.isnan(wr.grad[5]).any())
    cm = aecf_b200.CurriculumMasking().to(DEV)
    cm.eval()
    wd = w.to(DEV).requires_grad_(True)
    _, info = cm(wd)
    (info["entropy"] * g.to(DEV)).sum().backward()
    assert_close("d entropy / d w (eval forward)", wd.grad.cpu(), wr.grad, FP32_TOL, atol=1e-6)
    wc = w.to(DEV).requires_grad_(True)
    (cm.compute_entropy(wc) * g.to(DEV)).sum().backward()
    assert_close("d compute_entropy / d w", wc.grad.cpu(), wr.grad, FP32_TOL, atol=1e-6)
    assert_close("d entropy / d w (ops)", ops.entropy_bwd(w.to(DEV), g.to(DEV)).cpu(), wr.grad, FP32_TOL, atol=1e-6)


# ---- the small kernels at their edges -------------------------------------------------------------------------------------
def _mask_rows(L):
    w = torch.softmax(3 * torch.from_numpy(philox.normal(40 + L, (300, L))).float(), -1)
    w[::7] = 1.0 / L                                           # exact ties everywhere: the top-k repair's lowest-index rule
    w[1::11, : min(L, 3)] = 0.5                                # ties at the top
    w[3, 0] = float("nan")
    w[4, L - 1] = float("inf")
    w[6, 0] = float("-inf")
    w[5] = 0.0                                                 # all zero: degenerate, uniform weights
    w[8] = 1e-10                                               # total < 1e-8: degenerate too
    w[9] = 0.0
    w[9, L - 1] = 1e-9                                         # one tiny weight
    w[10] = 0.0
    w[10, 0] = 1.0                                             # a one-hot row (entropy 0: keep everything)
    w[12] = 3.0 * w[12]                                        # unnormalised
    return w


@pytest.mark.parametrize("min_active", [1, 3, 70])
@pytest.mark.parametrize("L", [1, 2, 5, 33, 64])
def test_curriculum_mask_kernel_edges(L, min_active):
    w = _mask_rows(L)
    u = torch.from_numpy(philox.mask_uniforms(5, 2, 11, w.shape[0], L))
    ref = oracle.curriculum_mask(w, u, base_mask_prob=0.9, min_active=min_active)
    m, e, r = ops.curriculum_mask(w.to(DEV), 1, base_mask_prob=0.9, min_active=min_active, seed=5, offset=2, row0=11)
    assert_close("masked", m.cpu(), ref["masked"], FP32_TOL, atol=1e-7)
    assert_close("entropy", e.cpu(), ref["entropy"], FP32_TOL, atol=1e-6)
    assert_close("mask_rate", r.cpu(), ref["mask_rate"], 0.0, atol=0.0)
    for mode in (2, 3):                                        # entropy only (eval / compute_entropy)
        m2, e2, r2 = ops.curriculum_mask(w.to(DEV), mode, want_masked=mode == 2)
        assert_close(f"mode {mode} entropy", e2.cpu(), oracle.shannon_entropy(w), FP32_TOL, atol=1e-6)
        assert float(r2.abs().max()) == 0.0
        if mode == 2:
            assert_close("mode 2 weights", m2.cpu(), w, 0.0, atol=0.0)


@pytest.mark.parametrize("min_active", [1, 3, 70])
@pytest.mark.parametrize("L", [1, 2, 5, 33, 64])
def test_curriculum_mask_backward_edges(L, min_active):
    """The training-mode backward against autograd through the oracle.  Left out are the rows whose kept weights are all
    exactly zero (an all-zero row, or a mask that keeps only zero / non-finite entries): autograd of the oracle's where()
    differentiates the branch it did not take too and gets 0 / 0 there, which says nothing about the kernel.  Degenerate
    rows of tiny non-zero weights, ties and non-finite entries are in."""
    w = _mask_rows(L)
    rows = w.shape[0]
    u = torch.from_numpy(philox.mask_uniforms(5, 2, 11, rows, L))
    g = torch.from_numpy(philox.normal(41, (rows, L))).float()
    compared = torch.ones(rows, dtype=torch.bool)
    if L > 1:
        wr = w.clone().requires_grad_(True)
        ref = oracle.curriculum_mask(wr, u, base_mask_prob=0.9, min_active=min_active)
        (ref["masked"] * g).sum().backward()
        want = wr.grad
        total = torch.where(torch.isfinite(w), w, torch.zeros(())).sum(-1)
        compared = (total != 0) & ((ref["renormalised"] * ref["mask"]).sum(-1) != 0).detach()
        assert not bool(compared[5])
    else:
        want = g                                               # a single token passes through
    got = ops.curriculum_mask_bwd(w.to(DEV), g.to(DEV), base_mask_prob=0.9, min_active=min_active, seed=5, offset=2, row0=11)
    per_row = torch.where(torch.isfinite(want), want, torch.zeros(())).abs().amax(1, keepdim=True).clamp(min=1.0)
    assert_close("d weights / row scale", (got.cpu() / per_row)[compared], (want / per_row)[compared], 1e-4, atol=1e-4)


def test_entropy_loss_over_several_passes_with_non_finite_entries():
    """n > 8192: every thread of the one-block kernel loads several entries; NaN and +-inf are scrubbed as the reference does."""
    for n in (8193, 100003):
        e = torch.from_numpy(philox.normal(50, (n,))).float().abs() * 0.7
        e[7], e[9], e[11], e[n - 1] = float("nan"), float("inf"), float("-inf"), float("nan")
        got = ops.entropy_loss_fwd(e.to(DEV), 0.7 * math.log(2))
        assert_close(f"entropy_loss n={n}", got.cpu(), oracle.entropy_loss(e.double(), 2, 0.7), 1e-5)
        assert torch.isfinite(got).all()


# every JMAX instantiation of the projection-free attention: NC = D / (16 bytes) <= 32 * JMAX
SDPA_SHAPES = [(torch.float32, 128), (torch.float32, 256), (torch.float32, 520), (torch.float32, 1024),
               (torch.bfloat16, 256), (torch.bfloat16, 512), (torch.bfloat16, 1024), (torch.bfloat16, 2048)]


@pytest.mark.parametrize("dtype,D", SDPA_SHAPES, ids=lambda v: str(v).replace("torch.", ""))
def test_sdpa_every_jmax(dtype, D):
    """fp64 reference, T in the hundreds, and a row of large-magnitude logits (the online softmax's rescaling)."""
    B, S, T = 2, 3, 300
    q = torch.from_numpy(philox.normal(60, (B, S, D))).to(dtype)
    k = torch.from_numpy(philox.normal(61, (B, T, D))).to(dtype)
    v = torch.from_numpy(philox.normal(62, (B, T, D))).to(dtype)
    q[1, 2] = (k[1, 150].float() * 8).to(dtype)                # logits of order 8 * sqrt(D): one token dominates
    q[0, 1] = (-q[0, 1].float() * 30).to(dtype)
    g = torch.from_numpy(philox.normal(63, (B, S, D))).to(dtype)
    qd, kd, vd = (t.double().requires_grad_(True) for t in (q, k, v))
    want = oracle.sdpa_single_head(qd, kd, vd)
    (want * g.double()).sum().backward()
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    out = ops.sdpa_fwd(q.to(DEV), k.to(DEV), v.to(DEV))
    assert_close("sdpa out", out.float().cpu(), want.detach(), tol)
    dq, dk, dv = ops.sdpa_bwd(q.to(DEV), k.to(DEV), v.to(DEV), g.to(DEV))
    # d_q and d_k go through p (s - delta) with logits up to ~100 here: the fp32 exp argument alone carries |s| 2^-24, which
    # the softmax backward turns into ~1e-3 of the gradient's scale.  A softmax without the running-max rescale would
    # overflow to inf / NaN instead, which the comparator rejects at any tolerance.
    tol_qk = 2e-3 if dtype == torch.float32 else 5 * BF16_TOL
    for name, a, b in (("d_q", dq, qd.grad), ("d_k", dk, kd.grad), ("d_v", dv, vd.grad)):
        assert_close(name, a.float().cpu(), b, tol_qk if name != "d_v" else tol)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_colsum_many_rows_strided_and_bf16_out(dtype):
    rows = 70001
    full = torch.from_numpy(philox.normal(70, (rows, 136))).to(dtype)
    on_dev = full.to(DEV)
    for cols in (96, 128):                                         # ld = 136 > cols
        x = on_dev[:, :cols]
        assert x.stride(0) == 136
        want = full[:, :cols].double().sum(0)
        assert_close("colsum", ops.colsum(x, torch.float32).cpu(), want, 1e-5, atol=1e-5 * math.sqrt(rows))
        assert_close("colsum bf16 out", ops.colsum(x, torch.bfloat16).float().cpu(), want, 1e-2, atol=1e-5 * math.sqrt(rows))
