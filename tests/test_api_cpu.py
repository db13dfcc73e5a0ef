"""CPU-side checks of the drop-in surface and of the C-ABI library (no kernel is launched here)."""
import ctypes
import os
import re

import pytest
import torch

import aecf
import aecf_b200
from aecf_b200 import _lib, ops
from aecf_b200.layers import _PhiloxState

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "aecf_b200.h")).read()
    declared = set(re.findall(r"AECF_API[^;(]*?\b(aecf_\w+)\s*\(", header))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.aecf_abi_version() == _lib.ABI_VERSION == 5
    assert b"sm_100a" in lib.aecf_build_info()
    assert lib.aecf_strerror(-2).decode().startswith("shape or dtype outside")


def test_ctypes_structs_mirror_the_header_layout(tmp_path):
    """Every ctypes mirror in _lib.py against what gcc lays out from include/aecf_b200.h: size and the offset of
    each field, by name."""
    import subprocess
    structs = {"aecf_pool_desc": _lib.PoolDesc, "aecf_gemm_desc": _lib.GemmDesc, "aecf_peer_desc": _lib.PeerDesc,
               "aecf_fusion_tensors": _lib.FusionTensors, "aecf_fusion_grads": _lib.FusionGrads}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "aecf_b200.h"', 'int main(void) {']
    for cname, mirror in structs.items():
        lines.append(f'printf("{cname} size %zu\\n", sizeof({cname}));')
        for field, _ in mirror._fields_:
            lines.append(f'printf("{cname} {field} %zu\\n", offsetof({cname}, {field}));')
    lines += ["return 0; }"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n")
    seen = 0
    for line in filter(None, out):
        cname, field, value = line.split()
        mirror = structs[cname]
        want = ctypes.sizeof(mirror) if field == "size" else getattr(mirror, field).offset
        assert int(value) == want, f"{cname}.{field}: header {value}, ctypes {want}"
        seen += 1
    assert seen == sum(len(m._fields_) + 1 for m in structs.values())


def test_descriptor_validation_needs_no_gpu():
    lib = _lib.load()
    d = _lib.PoolDesc(device=0, dtype=_lib.BF16, batch=4, num_tokens=9, embed_dim=64, num_heads=8)
    assert lib.aecf_pool_fwd(ctypes.byref(d), 16, 16, None, 16, 16, None, None, None, None, None) == _lib.ERR_UNSUPPORTED
    d.num_tokens, d.num_heads = 3, 7                                    # 7 does not divide 64
    assert lib.aecf_pool_fwd(ctypes.byref(d), 16, 16, None, 16, 16, None, None, None, None, None) == _lib.ERR_INVALID
    d.num_heads = 8
    assert lib.aecf_pool_fwd(ctypes.byref(d), 8, 16, None, 16, 16, None, None, None, None, None) == _lib.ERR_ALIGNMENT
    assert lib.aecf_pool_bwd_workspace_bytes(ctypes.byref(d)) == 2048 * 3 * 64 * 4
    g = _lib.GemmDesc(device=0, m=4, n=4, k=4, lda=2, ldb=4, ldc=4)     # lda < k
    assert lib.aecf_gemm(ctypes.byref(g), 16, 16, None, 16, None, 0, None) == _lib.ERR_INVALID


def test_alias_package_exposes_the_reference_names():
    for name in ("CurriculumMasking", "MultimodalAttentionPool", "multimodal_attention_pool", "create_fusion_pool"):
        assert getattr(aecf, name) is getattr(aecf_b200, name)
    assert sorted(aecf.__all__) == sorted(["CurriculumMasking", "MultimodalAttentionPool",
                                           "multimodal_attention_pool", "create_fusion_pool"])
    assert aecf.__version__ == "0.1.0"


def test_constructor_validation_matches_reference_messages():
    with pytest.raises(ValueError, match=r"base_mask_prob must be in \(0, 1\], got 0.0"):
        aecf.CurriculumMasking(base_mask_prob=0.0)
    with pytest.raises(ValueError, match=r"entropy_target must be in \(0, 1\], got 1.5"):
        aecf.CurriculumMasking(entropy_target=1.5)
    with pytest.raises(ValueError, match="min_active must be >= 1, got 0"):
        aecf.CurriculumMasking(min_active=0)
    with pytest.raises(ValueError, match="embed_dim must be positive, got 0"):
        aecf.MultimodalAttentionPool(0)
    with pytest.raises(ValueError, match="num_heads must be positive, got 0"):
        aecf.MultimodalAttentionPool(8, num_heads=0)
    with pytest.raises(ValueError, match=r"embed_dim \(10\) must be divisible by num_heads \(3\)"):
        aecf.MultimodalAttentionPool(10, num_heads=3)
    with pytest.raises(ValueError, match=r"dropout must be in \[0, 1\], got 1.5"):
        aecf.MultimodalAttentionPool(8, dropout=1.5)
    with pytest.raises(ValueError, match="embed_dim must be a positive integer, got -1"):
        aecf.create_fusion_pool(-1, 2)
    with pytest.raises(ValueError, match="num_modalities must be a positive integer, got 0"):
        aecf.create_fusion_pool(8, 0)
    with pytest.raises(ValueError, match=r"mask_prob must be in \(0, 1\], got 2"):
        aecf.create_fusion_pool(8, 2, mask_prob=2)


def test_forward_validation_matches_reference():
    pool = aecf.MultimodalAttentionPool(16, num_heads=2)
    q, k = torch.randn(4, 1, 16), torch.randn(4, 3, 16)
    with pytest.raises(TypeError, match="Expected query to be torch.Tensor"):
        pool([1, 2], k)
    with pytest.raises(TypeError, match="Expected key to be torch.Tensor"):
        pool(q, None)
    with pytest.raises(TypeError, match="Expected value to be torch.Tensor or None"):
        pool(q, k, 3)
    with pytest.raises(ValueError, match="Expected 3D query tensor with batch_first=True, got 2D"):
        pool(q[0], k)
    with pytest.raises(ValueError, match="Key sequence length cannot be zero"):
        pool(q, k[:, :0])
    with pytest.raises(RuntimeError, match="incompatible with query shape"):
        pool(q, torch.randn(5, 3, 16))
    with pytest.raises(RuntimeError, match="Value shape .* incompatible with key shape"):
        pool(q, k, torch.randn(4, 2, 16))
    seq = aecf.MultimodalAttentionPool(16, num_heads=2, batch_first=False)
    with pytest.raises(ValueError, match="Expected 3D key tensor with batch_first=False, got 2D"):
        seq(q, k[0])
    with pytest.raises(RuntimeError, match="Shape mismatch"):
        seq(torch.randn(1, 4, 16), torch.randn(3, 5, 16))
    # valid shapes on CPU tensors: the fusion path has no CPU implementation and says so
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        pool(q, k)
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        aecf.CurriculumMasking()(torch.softmax(torch.randn(4, 3), -1))
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        aecf.multimodal_attention_pool(q, k)


def test_state_dict_round_trips_with_torch_multihead_attention():
    torch.manual_seed(7)
    ours = aecf.MultimodalAttentionPool(32, num_heads=4, curriculum_masking=aecf.CurriculumMasking())
    torch.manual_seed(7)
    mha = torch.nn.MultiheadAttention(32, 4, batch_first=True)           # what the reference wraps (:399-407)
    want = {f"attention.{k}": v for k, v in mha.state_dict().items()}
    want["curriculum_masking._eps"] = torch.tensor(1e-8)
    got = ours.state_dict()
    assert list(got) == ["curriculum_masking._eps", "attention.in_proj_weight", "attention.in_proj_bias",
                         "attention.out_proj.weight", "attention.out_proj.bias"]
    for k in want:                                                       # same names, shapes AND default init
        assert torch.equal(got[k], want[k]), k
    other = aecf.MultimodalAttentionPool(32, num_heads=4, curriculum_masking=aecf.CurriculumMasking())
    missing, unexpected = other.load_state_dict(want, strict=True)
    assert not missing and not unexpected
    assert torch.equal(other.attention.in_proj_weight, mha.in_proj_weight)
    nobias = aecf.MultimodalAttentionPool(32, num_heads=4, bias=False)
    assert list(nobias.state_dict()) == ["attention.in_proj_weight", "attention.out_proj.weight"]


def test_factory_and_repr():
    torch.manual_seed(0)
    q, pool = aecf.create_fusion_pool(embed_dim=64, num_modalities=3, mask_prob=0.25, num_heads=8)
    torch.manual_seed(0)
    ref_q = torch.empty(1, 1, 64).normal_(0.0, (2.0 / 64) ** 0.5)
    assert isinstance(q, torch.nn.Parameter) and q.shape == (1, 1, 64) and torch.equal(q.detach(), ref_q)
    assert pool.num_heads == 8 and pool.embed_dim == 64 and pool.batch_first
    assert pool.curriculum_masking.base_mask_prob == 0.25 and pool.curriculum_masking._last_seq_len == 2
    assert "embed_dim=64, num_heads=8, batch_first=True, curriculum_masking=True" in repr(pool)
    assert "base_mask_prob=0.25, entropy_target=0.7, min_active=1" in repr(pool.curriculum_masking)
    _, default = aecf.create_fusion_pool(64, 2)
    assert default.num_heads == 1                                         # reference default (quirk D11)
    pool.curriculum_masking.base_mask_prob = 0.05                         # runtime mutation is allowed (README.md:341-350)
    pool.curriculum_masking = None                                        # and so is removing the stage (xrays:179-187)
    assert "curriculum_masking=False" in repr(pool)


def test_philox_call_counter():
    st = _PhiloxState()
    torch.manual_seed(123)
    assert [st.next() for _ in range(3)] == [(123, 0), (123, 1), (123, 2)]
    torch.manual_seed(5)                                                  # a new seed restarts the offsets
    assert st.next() == (5, 0)
    aecf_b200.set_rng_state(99, 7)
    try:
        assert aecf_b200.get_rng_state() == (99, 7)
    finally:
        aecf_b200.set_rng_state(None)


def test_folded_entry_points_validate_without_a_gpu():
    """Descriptor / argument checks of the folded-key-projection entry points run before any CUDA call."""
    lib = _lib.load()
    assert lib.aecf_fold_score_cols(_lib.BF16, 8) == 8 and lib.aecf_fold_score_cols(_lib.BF16, 12) == 16
    assert lib.aecf_fold_score_cols(_lib.F32, 1) == 4 and lib.aecf_fold_score_cols(_lib.F32, 8) == 8
    assert ops.fold_score_cols(torch.bfloat16, 8) == (8, 8) and ops.fold_score_cols(torch.float32, 6) == (8, 8)
    d = _lib.PoolDesc(device=0, dtype=_lib.BF16, batch=4, num_tokens=3, embed_dim=64, num_heads=8, q_is_shared=0)
    # the fold needs ONE query for all rows
    assert lib.aecf_pool_fwd_folded(ctypes.byref(d), 16, 16, None, 16, 16, None, None, None, None, None) == _lib.ERR_UNSUPPORTED
    d.q_is_shared = 1
    assert lib.aecf_pool_fwd_folded(ctypes.byref(d), None, 16, None, 16, 16, None, None, None, None, None) == _lib.ERR_INVALID
    assert lib.aecf_pool_fwd_folded(ctypes.byref(d), 16, 8, None, 16, 16, None, None, None, None, None) == _lib.ERR_ALIGNMENT
    d.kv_stride_b, d.kv_stride_m = 1, -2                                 # row strides must be positive
    assert lib.aecf_pool_fwd_folded(ctypes.byref(d), 16, 16, None, 16, 16, None, None, None, None, None) == _lib.ERR_INVALID
    d.kv_stride_b, d.kv_stride_m = 0, 0
    assert lib.aecf_pool_bwd_folded(ctypes.byref(d), 16, 16, 16, None, 16, None, None, 16, None, 16, 0, None) == _lib.ERR_WORKSPACE
    g = _lib.GemmDesc(device=0, dtype_a=_lib.BF16, dtype_b=_lib.BF16, dtype_c=_lib.BF16, m=256, n=128, k=64,
                      lda=64, ldb=64, ldc=128)
    for cols, ld in ((0, 8), (33, 36), (8, 4)):                          # no side columns / too many / aux_ld too small
        assert lib.aecf_gemm_aux(ctypes.byref(g), 16, 16, None, 16, 16, cols, ld, None, 0, None) == _lib.ERR_INVALID
    assert lib.aecf_fold_prepare(0, 7, 64, 8, 16, 16, 16, None) == _lib.ERR_INVALID       # unknown dtype
    assert lib.aecf_fold_prepare(0, _lib.BF16, 64, 7, 16, 16, 16, None) == _lib.ERR_INVALID   # 7 does not divide 64
    assert lib.aecf_fold_finish(0, _lib.F32, 64, 8, None, 16, 16, None, None, None) == _lib.ERR_INVALID
    # whole-step entry point: a folded descriptor with per-row queries is refused before anything is enqueued
    d.fold_key, d.q_is_shared = 1, 0
    t = _lib.FusionTensors()
    assert lib.aecf_fusion_fwd(ctypes.byref(d), ctypes.byref(t), 16, 1 << 30, None) == _lib.ERR_UNSUPPORTED


def test_graph_helper_needs_a_gpu_and_says_so():
    from aecf_b200 import graphs
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(RuntimeError, match="no CPU path"):
        graphs.GraphedStep(lambda: None)


def test_pool_exposes_the_fold_switch():
    pool = aecf.MultimodalAttentionPool(16, num_heads=2)
    assert pool.fold_key_projection is None                              # automatic: on for bf16 with a shared query
    pool.fold_key_projection = False
    assert "fold" not in repr(pool)                                      # extra_repr stays the reference's


def test_multi_query_descriptors_validate_without_a_gpu():
    """Several queries per sample (desc.tgt_len > 1): per-row queries only, no folded key projection, sane strides."""
    lib = _lib.load()
    d = _lib.PoolDesc(device=0, dtype=_lib.F32, batch=4, num_tokens=3, embed_dim=64, num_heads=8, q_is_shared=1, tgt_len=2)
    args = (16, 16, None, 16, 16, None, None, None, None, None)
    assert lib.aecf_pool_fwd(ctypes.byref(d), *args) == _lib.ERR_UNSUPPORTED        # one shared query and S > 1
    d.q_is_shared = 0
    d.q_stride_b, d.q_stride_s = -1, 1
    assert lib.aecf_pool_fwd(ctypes.byref(d), *args) == _lib.ERR_INVALID
    d.q_stride_b, d.q_stride_s = 0, 0
    assert lib.aecf_pool_fwd(ctypes.byref(d), 8, 16, None, 16, 16, None, None, None, None, None) == _lib.ERR_ALIGNMENT
    assert lib.aecf_pool_fwd_folded(ctypes.byref(d), *args) == _lib.ERR_UNSUPPORTED
    t = _lib.FusionTensors()
    d.q_is_shared = 1
    assert lib.aecf_fusion_fwd(ctypes.byref(d), ctypes.byref(t), 16, 1 << 30, None) == _lib.ERR_UNSUPPORTED
    one = _lib.PoolDesc(device=0, dtype=_lib.F32, batch=4, num_tokens=3, embed_dim=64, num_heads=8, q_is_shared=0)
    two = _lib.PoolDesc(device=0, dtype=_lib.F32, batch=4, num_tokens=3, embed_dim=64, num_heads=8, q_is_shared=0, tgt_len=4)
    assert lib.aecf_fusion_workspace_bytes(ctypes.byref(two)) >= lib.aecf_fusion_workspace_bytes(ctypes.byref(one)) > 0


@pytest.mark.parametrize("batch_first", [True, False])
def test_multi_query_host_plumbing(monkeypatch, batch_first):
    """What the module hands to the C ABI for a [B, S, D] query, with the native calls recorded instead of run: the
    descriptor (tgt_len, query row strides, bias strides), buffer shapes, the shapes that come back, and the gate."""
    B, S, M, D, H = 6, 3, 4, 32, 4
    calls = {}
    monkeypatch.setattr(ops, "require_cuda", lambda *t: torch.device("cpu"))
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: False)
    monkeypatch.setattr(ops, "fusion_workspace", lambda desc, dev: torch.empty(1))
    monkeypatch.setattr(ops, "fusion_fwd", lambda desc, tensors, dev: calls.setdefault("fwd", (desc, tensors)))
    monkeypatch.setattr(ops, "fusion_bwd", lambda desc, tensors, grads, ws, dev: calls.setdefault("bwd", []).append((desc, grads)))
    pool = aecf.MultimodalAttentionPool(D, num_heads=H, curriculum_masking=aecf.CurriculumMasking(), batch_first=batch_first)
    q = torch.randn(B, S, D, requires_grad=True) if batch_first else torch.randn(S, B, D, requires_grad=True)
    k = torch.randn(B, M, D, requires_grad=True) if batch_first else torch.randn(M, B, D, requires_grad=True)
    kpm = torch.zeros(B, M, dtype=torch.bool)
    am = torch.zeros(S, M)
    out, info = pool(q, k, key_padding_mask=kpm, attn_mask=am, return_info=True)
    desc, tensors = calls["fwd"]
    assert (desc.batch, desc.tgt_len, desc.num_tokens, desc.q_is_shared, desc.fold_key) == (B, S, M, 0, 0)
    assert (desc.q_stride_b, desc.q_stride_s) == ((0, 0) if batch_first else (1, B))
    assert (desc.bias_stride_b, desc.bias_stride_h, desc.bias_stride_s) == (S * M, 0, M)   # [B, 1, S, M] merged bias
    assert (desc.kv_stride_b, desc.kv_stride_m) == ((0, 0) if batch_first else (2 * D, B * 2 * D))
    assert out.shape == ((B, S, D) if batch_first else (S, B, D))
    assert info["attention_weights"].shape == (B, S, M) and info["masked_attention_weights"].shape == (B, S, M)
    assert info["entropy"].shape == info["mask_rate"].shape == info["target_entropy"].shape == (B, S)
    (out.sum() + info["attention_weights"].sum()).backward()
    assert len(calls["bwd"]) == 1                        # the whole backward in one call
    desc_b, grads = calls["bwd"][0]
    assert desc_b is desc and grads.d_q_rows and grads.d_pooled and grads.d_query
    assert q.grad.shape == q.shape and k.grad.shape == k.shape
    assert pool.attention.in_proj_weight.grad.shape == (3 * D, D)
    with pytest.raises(RuntimeError, match=r"2D attn_mask is \(1, 4\), but should be \(3, 4\)"):
        pool(q, k, attn_mask=torch.zeros(1, M))
