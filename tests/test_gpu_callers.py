"""SURVEY.md section 8f rows 1-2: the documented callers of the pool, run end to end on the CUDA path and on
the oracle with identical parameters and Philox draws (fp32, 1e-5-level agreement of logits, losses
and every parameter gradient over several optimiser steps)."""
import copy

import pytest
import torch
import torch.nn.functional as F

import aecf_b200
from examples.models import VisionLanguageModel, XrayFusionModel
from oracle import philox
from tests import oracle_fusion
from tests.helpers import assert_close, finite_scale

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEED = 0xA11CE


def _twin(model_cls, **kwargs):
    torch.manual_seed(3)
    ours = model_cls(fusion=aecf_b200, **kwargs).to(DEV)
    ref = model_cls(fusion=oracle_fusion, **kwargs)
    ref.load_state_dict({k: v.detach().cpu() for k, v in ours.state_dict().items()})
    for m in (ours, ref):                       # the encoders' nn.Dropout draws from torch's RNG: keep it out of the comparison
        for sub in m.modules():
            if isinstance(sub, torch.nn.Dropout):
                sub.p = 0.0
    return ours, ref


def _compare_step(ours, ref, inputs, loss_fn, step, lr=0.05, tol=2e-5):
    aecf_b200.set_rng_state(SEED, step)
    oracle_fusion.set_rng_state(SEED, step)
    try:
        out_o, info_o = ours(*[t.to(DEV) for t in inputs], return_info=True)
    finally:
        aecf_b200.set_rng_state(None)
    out_r, info_r = ref(*inputs, return_info=True)
    loss_o, loss_r = loss_fn(ours, out_o, info_o, DEV), loss_fn(ref, out_r, info_r, "cpu")
    assert_close(f"step {step} logits", out_o.cpu(), out_r, tol)
    assert_close(f"step {step} loss", loss_o.cpu(), loss_r, tol)
    if "entropy" in info_r:
        assert_close(f"step {step} entropy", info_o["entropy"].cpu(), info_r["entropy"], tol, atol=1e-6)
        assert torch.equal(info_o["mask_rate"].cpu(), info_r["mask_rate"].float()), "mask_rate differs"
    for m in (ours, ref):
        m.zero_grad(set_to_none=True)
    loss_o.backward()
    loss_r.backward()
    ref_params = dict(ref.named_parameters())
    for name, p in ours.named_parameters():
        g_ref = ref_params[name].grad
        if g_ref is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, name
            continue
        assert_close(f"step {step} grad {name}", p.grad.cpu(), g_ref, 5 * tol, atol=5 * tol * finite_scale(g_ref) + 1e-9)
    with torch.no_grad():
        for m in (ours, ref):
            for p in m.parameters():
                if p.grad is not None:
                    p -= lr * p.grad


def test_vision_language_model_training_steps():
    """reference README.md:162-208: 2048/768 -> 512, M = 2, default single head (head_dim 512), 1000 classes."""
    ours, ref = _twin(VisionLanguageModel)
    B = 48
    img = torch.from_numpy(philox.normal(1, (B, 2048))).float()
    txt = torch.from_numpy(philox.normal(2, (B, 768))).float()
    labels = torch.from_numpy(philox.normal(3, (B,))).abs().mul(300).long().clamp(max=999)

    def loss_fn(model, logits, info, dev):
        ent = model.fusion_pool.curriculum_masking.entropy_loss(info["entropy"])
        return F.cross_entropy(logits, labels.to(dev)) + 0.01 * ent

    for step in range(3):
        _compare_step(ours, ref, (img, txt), loss_fn, step)
    assert ours.fusion_pool.curriculum_masking._last_seq_len == 2


def test_xray_fusion_model_missing_modalities_and_curriculum_toggle():
    """reference xrays/train_xrays_example.py:108-237: hidden 256, 4 heads, the pool only on the rows where
    both modalities are present (a ragged subset), single-modality rows bypass it, curriculum switched on
    at run time."""
    ours, ref = _twin(XrayFusionModel)
    B = 64
    img = torch.from_numpy(philox.normal(11, (B, 512))).float()
    txt = torch.from_numpy(philox.normal(12, (B, 512))).float()
    drop = torch.from_numpy(philox.normal(13, (B,)))
    img[drop < -0.6] = 0.0                         # image missing
    txt[drop > 0.7] = 0.0                          # text missing
    target = (torch.from_numpy(philox.normal(14, (B, 80))) > 0.8).float()

    def loss_fn(model, logits, info, dev):
        return F.binary_cross_entropy_with_logits(logits, target.to(dev))

    _compare_step(ours, ref, (img, txt), loss_fn, 0)            # curriculum off: info has attention weights only
    for m in (ours, ref):
        m.toggle_curriculum(True)
    _compare_step(ours, ref, (img, txt), loss_fn, 1)
    _compare_step(ours, ref, (img, txt), loss_fn, 2)
    ours.eval(); ref.eval()                                     # missing-modality evaluation (:252-310)
    with torch.no_grad():
        only_img = ours(img.to(DEV), torch.zeros_like(txt).to(DEV))
        assert_close("eval, text missing", only_img.cpu(), ref(img, torch.zeros_like(txt)), 2e-5)
        both = ours(img.to(DEV), txt.to(DEV))
        assert_close("eval, as given", both.cpu(), ref(img, txt), 2e-5)
