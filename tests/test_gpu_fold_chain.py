"""The backward of the folded key projection through its stand-alone entry points, chained by hand as INTEGRATION.md
describes it: ``aecf_pool_bwd_folded`` (with ``d_bias_kv``: per-CTA batch-sum partials and their finalize) -> ``aecf_gemm``
for ``[dWv ; R] = d_vs^T X`` in fp32 -> ``aecf_fold_finish``.  The whole-step backward (``aecf_fusion_bwd``) calls neither
the first nor the last of them, so this is where they run.  Inputs are the oracle's forward results; the gradients are
compared with the oracle's in the folded association at the fp32 tolerance of test_gpu_parity.py.
"""
import ctypes as C
import math

import pytest
import torch

from aecf_b200 import _lib, ops
from tests.golden.cases import CASES_BY_NAME, PHILOX_SEED, build_inputs
from tests.helpers import assert_close, finite_scale, run_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FP32_TOL = 1e-5


def test_standalone_folded_backward_chain_matches_oracle():
    case = CASES_BY_NAME["d64_h8_m3_dropout"]           # one shared query, dropout, gradient on the pooled weights
    B, M, D, H = case.B, case.M, case.D, case.H
    hd = D // H
    dev = torch.device(DEV)
    inp = build_inputs(case)
    ref, ref_grads = run_oracle(case, inp, fold_key=True)
    hs, hsp = ops.fold_score_cols(torch.float32, H)

    # what the folded forward leaves for the backward: q_proj [D] fp32, the values, the scores x . Qk[h] (no key bias)
    in_w = inp["in_proj_weight"]
    q_proj = ref.saved["qp"][0, 0]
    qk = torch.einsum("he,hed->hd", q_proj.view(H, hd), in_w[D:2 * D].view(H, hd, D)) * math.sqrt(1.0 / hd)
    x = inp["x"].reshape(B * M, D)
    scores = torch.zeros(B * M, hs)
    scores[:, :H] = x @ qk.t()
    d_ctx = inp["grad_out"].reshape(B, D) @ inp["out_proj.weight"]
    on_dev = lambda t: t.to(DEV).contiguous()           # noqa: E731
    in_w, q_proj, x, scores, d_ctx = map(on_dev, (in_w, q_proj, x, scores, d_ctx))
    v = on_dev(ref.saved["v"].reshape(B * M, D))
    d_pooled = on_dev(inp["grad_pooled"].reshape(B, M))

    desc = ops.make_pool_desc(dev, torch.float32, batch=B, num_tokens=M, embed_dim=D, num_heads=H, training=True,
                              masking=1, min_active=case.min_active, q_is_shared=True, base_mask_prob=case.base_mask_prob,
                              entropy_target=case.entropy_target, dropout_p=case.dropout, seed=PHILOX_SEED,
                              offset=case.offset, row0=case.row0, fold_key=True)
    lib = _lib.load()
    stream = ops._stream(dev)
    d_vs = torch.empty(B * M, D + hsp, device=dev)
    d_bias_kv = torch.empty(2 * D, device=dev)
    ws = torch.empty(max(lib.aecf_pool_bwd_workspace_bytes(C.byref(desc)), 16), dtype=torch.uint8, device=dev)
    _lib.check(lib.aecf_pool_bwd_folded(C.byref(desc), q_proj.data_ptr(), scores.data_ptr(), v.data_ptr(), None,
                                        d_ctx.data_ptr(), d_pooled.data_ptr(), None, d_vs.data_ptr(), d_bias_kv.data_ptr(),
                                        ws.data_ptr(), ws.numel(), stream), "aecf_pool_bwd_folded")
    g = ops.matmul_tn(d_vs, x, out_dtype=torch.float32)                         # [dWv ; R], [D + HSP, D]
    d_in_w = torch.zeros(3 * D, D, device=dev)
    d_q_proj = torch.empty(D, device=dev)
    _lib.check(lib.aecf_fold_finish(dev.index or 0, _lib.F32, D, H, g.data_ptr(), q_proj.data_ptr(), in_w.data_ptr(),
                                    d_in_w.data_ptr(), d_q_proj.data_ptr(), stream), "aecf_fold_finish")

    want_bias = ref_grads["in_proj_bias"]                   # [d q_proj | d_bk | d_bv]; the key third is analytically zero
    assert_close("d_in_proj_weight[D:3D]", d_in_w[D:].cpu(), ref_grads["in_proj_weight"][D:], FP32_TOL)
    assert not d_in_w[:D].cpu().any(), "aecf_fold_finish wrote the query rows"
    assert_close("d_q_proj", d_q_proj.cpu(), want_bias[:D], FP32_TOL)
    assert_close("d_bias_kv", d_bias_kv.cpu(), want_bias[D:], FP32_TOL, atol=FP32_TOL * finite_scale(want_bias))
