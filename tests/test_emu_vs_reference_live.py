"""The product path (module API -> C ABI -> the CUDA sources under the host emulation, tests/cuda_emu) on seeded random
shapes and options, including shapes no fixture has (D = 768, H = 3, M = 7 ...).

With AECF_REFERENCE naming a checkout of the reference implementation, the comparison is against that UNMODIFIED
reference imported live, on the same inputs with the shared Philox draws injected into its two RNG call sites
(tests/golden/make_golden.py, SURVEY.md Appendix C).  The reference is not part of this repository; without it the same
cases are compared with the oracle (oracle/aecf_oracle.py), which tests/test_oracle_golden.py pins to the reference's own
outputs on the committed fixtures.
"""
import os
import random
import sys

import numpy as np
import pytest
import torch

import aecf_b200
from tests.emu_support import cuda_emulation  # noqa: F401  (fixture)
from oracle import aecf_oracle as oracle
from tests.golden.cases import PHILOX_SEED, Case, build_inputs, masking_kwargs
from tests.helpers import assert_close, finite_scale, run_oracle

REFERENCE = os.environ.get("AECF_REFERENCE", "")
pytestmark = pytest.mark.usefixtures("cuda_emulation")


def _reference_module():
    """The reference's ``aecf`` package under a private name (this repo ships an alias package called ``aecf`` too)."""
    import importlib.util
    assert os.path.isfile(os.path.join(REFERENCE, "aecf", "AECFLayer.py")), f"AECF_REFERENCE={REFERENCE!r} is not a reference checkout"
    spec = importlib.util.spec_from_file_location("aecf_reference_live", os.path.join(REFERENCE, "aecf", "AECFLayer.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[spec.name] = mod
    spec.loader.exec_module(mod)
    return mod


def _load(pool, inp):
    with torch.no_grad():
        pool.attention.in_proj_weight.copy_(inp["in_proj_weight"])
        pool.attention.in_proj_bias.copy_(inp["in_proj_bias"])
        pool.attention.out_proj.weight.copy_(inp["out_proj.weight"])
        pool.attention.out_proj.bias.copy_(inp["out_proj.bias"])


def _run(mod, pool, cm, case, inp, multi, inject):
    query = torch.nn.Parameter((inp["query"] if multi else inp["query0"]).clone())
    x = inp["x"].clone().requires_grad_(True)
    kpm = inp.get("key_padding_mask")
    with inject:
        out, info = pool(query if multi else query.expand(case.B, -1, -1), x, key_padding_mask=kpm, return_info=True)
    ent_loss = cm.entropy_loss(info["entropy"])
    loss = (out * inp["grad_out"]).sum()
    if case.pooled_grad:
        loss = loss + (info["attention_weights"] * inp["grad_pooled"]).sum()
    if not case.training:
        loss = loss + 0.5 * info["entropy"].sum()
    loss.backward()
    att = pool.attention
    return {"out": out, "info": info, "entropy_loss": ent_loss, "x": x.grad, "query": query.grad, "in_w": att.in_proj_weight.grad,
            "in_b": att.in_proj_bias.grad, "out_w": att.out_proj.weight.grad, "out_b": att.out_proj.bias.grad}


class _NoInjection:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


def _want_from_reference(case, inp, multi):
    from tests.golden.injection import inject_uniforms
    ref_mod = _reference_module()
    ref_cm = ref_mod.CurriculumMasking(**masking_kwargs(case))
    ref_pool = ref_mod.MultimodalAttentionPool(case.D, num_heads=case.H, dropout=case.dropout, curriculum_masking=ref_cm)
    _load(ref_pool, inp)
    ref_pool.train(case.training)
    want = _run(ref_mod, ref_pool, ref_cm, case, inp, multi, inject_uniforms(inp["u_mask"], inp["u_drop"]))
    return want, ref_cm._last_seq_len


def _want_from_oracle(case, inp, multi):
    """The same step through the oracle: forward, closed-form backward of the same loss, the reference's info keys."""
    fwd, grads = run_oracle(case, inp)
    info = {k: v for k, v in fwd.info.items() if k not in ("mask", "keep_prob")}
    last = case.M if (case.training and case.M > 1) else 2          # the reference's _last_seq_len (AECFLayer.py:99, :187)
    want = {"out": fwd.out, "info": info, "entropy_loss": oracle.entropy_loss(info["entropy"], last, case.entropy_target),
            "x": grads["key"], "query": grads["query" if multi else "query0"], "in_w": grads["in_proj_weight"],
            "in_b": grads["in_proj_bias"], "out_w": grads["out_proj.weight"], "out_b": grads["out_proj.bias"]}
    return want, last


@pytest.mark.parametrize("seed", range(6))
def test_random_cases_against_the_live_reference(monkeypatch, seed):
    rng = random.Random(7000 + seed)
    multi = seed % 3 == 2
    hd, heads = rng.choice([16, 32, 64, 128]), rng.choice([1, 2, 3, 4, 6, 8])
    if seed == 0:
        hd, heads = 64, 12                                           # D = 768
    tokens = rng.randint(2, 8)
    case = Case(f"live{seed}", B=rng.choice([3, 8, 17]), S=rng.randint(2, 3) if multi else 1, M=tokens, D=hd * heads, H=heads,
                dropout=rng.choice([0.0, 0.1, 0.3]), base_mask_prob=rng.choice([0.15, 0.6, 1.0]), min_active=rng.choice([1, 2, 3]),
                training=rng.random() < 0.8, kpm=rng.random() < 0.3, pooled_grad=rng.random() < 0.5, offset=rng.randint(0, 99),
                row0=rng.choice([0, 11]), data_seed=rng.randint(1000, 10 ** 6), peak=rng.choice([0.5, 1.0, 2.0]))
    inp = build_inputs(case)
    want, want_last_seq_len = (_want_from_reference if REFERENCE else _want_from_oracle)(case, inp, multi)

    cm = aecf_b200.CurriculumMasking(**masking_kwargs(case))
    pool = aecf_b200.MultimodalAttentionPool(case.D, num_heads=case.H, dropout=case.dropout, curriculum_masking=cm)
    _load(pool, inp)
    pool.train(case.training)
    pool.row_offset = case.row0
    aecf_b200.set_rng_state(PHILOX_SEED, case.offset)
    try:
        got = _run(aecf_b200, pool, cm, case, inp, multi, _NoInjection())
    finally:
        aecf_b200.set_rng_state(None)

    tol = 3e-5            # two fp32 implementations with different summation orders
    assert set(got["info"]) == set(want["info"])
    assert_close("out", got["out"], want["out"], tol)
    assert_close("attention_weights", got["info"]["attention_weights"], want["info"]["attention_weights"], tol, atol=tol)
    assert_close("entropy", got["info"]["entropy"], want["info"]["entropy"], tol, atol=tol)
    assert np.array_equal(got["info"]["mask_rate"].detach().numpy(), want["info"]["mask_rate"].detach().numpy()), "mask_rate differs"
    live = want["info"]["attention_weights"].detach() > 0
    assert torch.equal((got["info"]["masked_attention_weights"] > 0) & live, want["info"]["masked_attention_weights"] > 0), "active sets differ"
    assert_close("masked_attention_weights", got["info"]["masked_attention_weights"], want["info"]["masked_attention_weights"], tol, atol=tol)
    assert_close("entropy_loss", got["entropy_loss"], want["entropy_loss"], tol, atol=tol)
    assert cm._last_seq_len == want_last_seq_len
    for name in ("x", "query", "in_w", "out_w", "out_b"):
        assert_close("grad " + name, got[name], want[name], tol)
    scale = finite_scale(want["in_b"])
    assert_close("grad in_b", got["in_b"], want["in_b"], tol, atol=tol * scale)
