"""Mixed precision without a device: the descriptor rules of the C ABI and what the module hands to it."""
import ctypes as C

import pytest
import torch

import aecf_b200 as aecf
from aecf_b200 import _lib, ops


def _desc(dtype, flag):
    return ops.make_pool_desc(torch.device("cpu"), dtype, batch=4, num_tokens=3, embed_dim=64, num_heads=4, training=True,
                              masking=0, min_active=1, q_is_shared=True, base_mask_prob=0.15, entropy_target=0.7,
                              dropout_p=0.0, seed=0, offset=0, row0=0, param_grads_f32=flag)


@pytest.mark.parametrize("dtype,flag", [(torch.float32, 1), (torch.bfloat16, 2), (torch.bfloat16, -1)])
def test_param_grads_f32_rules(dtype, flag):
    """param_grads_f32 = 1 needs bf16 compute; anything but 0 and 1 is invalid.  The descriptor is checked before any
    device work, so this runs without a GPU."""
    lib = _lib.load()
    desc = _desc(dtype, flag)
    assert lib.aecf_fusion_workspace_bytes(C.byref(desc)) == 0
    t, g = _lib.FusionTensors(), _lib.FusionGrads()
    assert lib.aecf_fusion_fwd(C.byref(desc), C.byref(t), None, 0, None) == _lib.ERR_INVALID
    assert lib.aecf_fusion_bwd(C.byref(desc), C.byref(t), C.byref(g), None, 0, None) == _lib.ERR_INVALID


def test_param_grads_f32_layout():
    assert _lib.PoolDesc.param_grads_f32.offset == _lib.PoolDesc.loss_target.offset + 4
    assert "aecf_param_cast" in _lib.EXPORTS and hasattr(_lib.load(), "aecf_param_cast")
    assert _desc(torch.bfloat16, 1).param_grads_f32 == 1 and _desc(torch.bfloat16, 0).param_grads_f32 == 0


@pytest.mark.parametrize("shared", [True, False], ids=["shared_query", "per_row_query"])
def test_mixed_host_plumbing(monkeypatch, shared):
    """fp32 parameters with bf16 inputs: the forward sets the descriptor flag, rounds the parameters (and the shared query)
    in one cast call and passes those shadows as the parameter pointers; the backward allocates fp32 parameter gradients
    and bf16 input gradients."""
    B, M, D, H = 6, 3, 32, 4
    calls = {}

    def fake_cast(tensors):
        calls.setdefault("cast", []).append([None if t is None else (t.dtype, tuple(t.shape)) for t in tensors])
        views = [None if t is None else t.detach().bfloat16() for t in tensors]
        calls.setdefault("views", []).append(views)
        return None, views

    monkeypatch.setattr(ops, "require_cuda", lambda *t: torch.device("cpu"))
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: False)
    monkeypatch.setattr(ops, "param_cast", fake_cast)
    monkeypatch.setattr(ops, "fusion_workspace", lambda desc, dev: torch.empty(1))
    monkeypatch.setattr(ops, "fusion_fwd", lambda desc, tensors, dev: calls.setdefault("fwd", (desc, tensors)))
    monkeypatch.setattr(ops, "fusion_bwd", lambda desc, tensors, grads, ws, dev: calls.setdefault("bwd", (desc, tensors, grads)))
    q0, pool = aecf.create_fusion_pool(D, M, 0.15, num_heads=H)
    assert pool.attention.in_proj_weight.dtype == torch.float32
    k = torch.randn(B, M, D).bfloat16().requires_grad_(True)
    q = q0.expand(B, -1, -1) if shared else torch.randn(B, 1, D).bfloat16().requires_grad_(True)
    out = pool(q, k)
    assert out.dtype == torch.bfloat16
    desc, tensors = calls["fwd"]
    assert desc.dtype == _lib.BF16 and desc.param_grads_f32 == 1 and desc.q_is_shared == int(shared)
    assert desc.fold_key == int(shared)                               # the fold follows the bf16 compute dtype
    assert len(calls["cast"]) == 1
    cast = calls["cast"][0]
    assert cast[:4] == [(torch.float32, (3 * D, D)), (torch.float32, (3 * D,)), (torch.float32, (D, D)), (torch.float32, (D,))]
    assert cast[4] == ((torch.float32, (D,)) if shared else None)
    views = calls["views"][0]
    assert tensors.in_proj_weight == views[0].data_ptr() and tensors.in_proj_bias == views[1].data_ptr()
    assert tensors.out_proj_weight == views[2].data_ptr() and tensors.out_proj_bias == views[3].data_ptr()
    if shared:
        assert tensors.query == views[4].data_ptr()
    out.float().sum().backward()
    desc_b, tensors_b, grads = calls["bwd"]
    assert desc_b is desc and tensors_b.in_proj_weight == views[0].data_ptr()
    att = pool.attention
    for p in (att.in_proj_weight, att.in_proj_bias, att.out_proj.weight, att.out_proj.bias):
        assert p.grad.dtype == torch.float32 and p.grad.shape == p.shape
    assert k.grad.dtype == torch.bfloat16 and k.grad.shape == k.shape
    if shared:
        assert q0.grad.dtype == torch.float32 and q0.grad.shape == q0.shape
    else:
        assert q.grad.dtype == torch.bfloat16 and q.grad.shape == q.shape
    assert grads.d_in_proj_weight == att.in_proj_weight.grad.data_ptr()
