"""Heads that are not a power-of-two number of 16-byte chunks (head_dim 24, 48, 80, 96, 384, 768 ...): the padded lane map
of the pool kernels (csrc/pool_core.cuh, PAD instantiations), through the public module API, against the oracle.

The oracle is generic in shape and pinned to the reference by the golden fixtures of tests/test_gpu_parity.py; the bodies
of the parity tests are reused here on the new geometries.  Geometry per case (G = head_dim / V chunks, padded to the next
power of two GP; J chunk columns per lane, R columns per head, WPS warps per sample) is listed next to it.
"""
import pytest
import torch

import aecf_b200
from aecf_b200 import _lib
from tests import test_gpu_multi_query as MQ
from tests import test_gpu_parity as P
from tests.golden.cases import Case

pytestmark = pytest.mark.gpu

#                                                                                  bf16: G -> GP, J, R, WPS  fp32: G -> GP, J, R, WPS
HEAD_DIM_CASES = [
    Case("hd48_d192_h4_m4_kpm", B=24, M=4, D=192, H=4, kpm=True, min_active=2, base_mask_prob=0.8,   # 6->8, 1, 1, 1    12->16, 2, 1, 1
         data_seed=401),
    Case("hd24_d240_h10_m3", B=20, M=3, D=240, H=10, data_seed=402),                                # 3->4, 2, 1, 1    6->8, 2, 1, 2
    Case("hd80_d320_h4_m5_eval", B=16, M=5, D=320, H=4, training=False, pooled_grad=True,           # 10->16, 2, 1, 1  20->32, 2, 1, 2
         data_seed=403),
    Case("hd48_d384_h8_m3_dropout", B=24, M=3, D=384, H=8, dropout=0.1, pooled_grad=True, offset=3,  # 6->8, 2, 1, 1    12->16, 2, 1, 2
         data_seed=404),
    Case("hd384_d384_h1_m3", B=16, M=3, D=384, H=1, data_seed=405),                                 # 48->64, 2, 2, 1  96->128, 4, 4, 1
    Case("hd96_d768_h8_m3", B=12, M=3, D=768, H=8, dropout=0.1, row0=77, data_seed=406),            # 12->16, 2, 1, 2  24->32, 2, 1, 4
    Case("hd96_d1536_h16_m2", B=8, M=2, D=1536, H=16, base_mask_prob=0.5, data_seed=407),           # 12->16, 2, 1, 4  24->32, 2, 1, 8
]
# fp32 D = 768 with one head is 192 chunks per head (GP = 256 > 128): bf16 only
BF16_ONLY_CASES = [
    Case("hd768_d768_h1_m3", B=12, M=3, D=768, H=1, pooled_grad=True, data_seed=408),              # 96->128, 4, 4, 1
]


@pytest.mark.parametrize("case", HEAD_DIM_CASES, ids=lambda c: c.name)
def test_fp32_matches_oracle(case):
    P.test_fp32_matches_oracle(case)
    P.test_fp32_folded_key_projection_matches_oracle(case)


@pytest.mark.parametrize("fold", [True, False], ids=["folded", "unfolded"])
@pytest.mark.parametrize("case", HEAD_DIM_CASES + BF16_ONLY_CASES, ids=lambda c: c.name)
def test_bf16_masks_exact_against_stage_rounded_oracle(case, fold):
    P.test_bf16_masks_exact_against_stage_rounded_oracle(case, fold)


def test_full_size_d768_h8_bf16_folded_against_oracle():
    """The headline test's body at head_dim 96: B = 16 384 puts every product on the tcgen05 GEMMs, peaked inputs; mask bits
    and mask_rate exact, every row of the output and of the input gradient inside the bf16 budget of its own scale."""
    P.test_full_size_bf16_folded_against_oracle(
        Case("full_b16384_d768_h8_m3", B=16384, M=3, D=768, H=8, data_seed=409, offset=1))


MULTI_QUERY_CASES = [
    Case("s2_hd96_d192_h2_m3_dropout", B=12, S=2, M=3, D=192, H=2, dropout=0.1, pooled_grad=True, offset=5,   # 12->16  24->32
         data_seed=410),
    Case("s2_hd96_d384_h4_m4_kpm_eval", B=10, S=2, M=4, D=384, H=4, kpm=True, training=False, pooled_grad=True,
         data_seed=411),
]


@pytest.mark.parametrize("case", MULTI_QUERY_CASES, ids=lambda c: c.name)
def test_multi_query_fp32_and_bf16(case):
    MQ.test_fp32_matches_oracle(case, True)
    MQ.test_bf16_masks_exact_against_stage_rounded_oracle(case)


@pytest.mark.parametrize("dtype,fold", [(torch.float32, False), (torch.float32, True), (torch.bfloat16, True), (torch.bfloat16, False)],
                         ids=["fp32_unfolded", "fp32_folded", "bf16_folded", "bf16_unfolded"])
def test_sample_index_pools_the_listed_rows_in_place(monkeypatch, dtype, fold):
    """The in-place row-index body of the parity tests on a head_dim-96 case: bit-identical to pooling x[idx]."""
    case = Case("hd96_d384_h4_m3_dropout", B=40, M=3, D=384, H=4, dropout=0.1, pooled_grad=True, offset=3, data_seed=412)
    monkeypatch.setitem(P.CASES_BY_NAME, "d64_h8_m3_dropout", case)      # the case the body pools
    P.test_sample_index_pools_the_listed_rows_in_place(dtype, fold)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_graph_replay_matches_eager(dtype):
    """One captured step at head_dim 96 (D = 384, H = 4): the replay is bit-identical to the eager step."""
    torch.manual_seed(4)
    B, M, D, H = 1024, 3, 384, 4
    q, pool = aecf_b200.create_fusion_pool(D, M, 0.4, num_heads=H, dropout=0.1, device=P.DEV, dtype=dtype)
    pool._want_mask_bits = True
    cm = pool.curriculum_masking
    x = torch.randn(B, M, D, device=P.DEV, dtype=dtype).requires_grad_(True)
    params = [q, x, pool.attention.in_proj_weight, pool.attention.in_proj_bias, pool.attention.out_proj.weight,
              pool.attention.out_proj.bias]

    def clear():
        for p in params:
            p.grad = None

    def step():
        out, info = pool(q.expand(B, -1, -1), x, return_info=True)
        loss = out.float().pow(2).mean() + 0.01 * cm.entropy_loss(info["entropy"])
        loss.backward()
        return out, info["mask_bits"], info["attention_weights"], loss

    def snapshot(res):
        return [t.detach().clone() for t in res] + [p.grad.detach().clone() for p in params]

    aecf_b200.set_rng_state(555, 5)
    graphed = aecf_b200.graphs.GraphedStep(step, reset=clear, warmup=2, device=torch.device(P.DEV))
    replay = snapshot(graphed())
    torch.cuda.synchronize()
    aecf_b200.set_rng_state(555, 7)        # warm-up took offsets 5 and 6, prepare() took 7
    clear()
    eager = snapshot(step())
    aecf_b200.set_rng_state(None)
    for j, (a, b) in enumerate(zip(replay, eager)):
        assert torch.equal(a, b), f"tensor {j} of the replay differs from the eager step"


@pytest.mark.parametrize("D,H,dtype", [(768, 1, torch.float32), (144, 4, torch.bfloat16)],
                         ids=["fp32_hd768_gp256", "bf16_hd36_72_bytes"])
def test_shapes_outside_the_map_still_fail_loudly(D, H, dtype):
    """192 chunks per head pad to 256 > 128; 36 bf16 elements are 72 bytes, not a whole number of 16-byte chunks."""
    pool = aecf_b200.MultimodalAttentionPool(D, num_heads=H, device=P.DEV, dtype=dtype)
    with pytest.raises(_lib.UnsupportedShapeError):
        pool(torch.randn(4, 1, D, device=P.DEV, dtype=dtype), torch.randn(4, 3, D, device=P.DEV, dtype=dtype))
