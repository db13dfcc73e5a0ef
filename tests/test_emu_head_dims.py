"""The padded lane map (head_dim not a power-of-two number of 16-byte chunks) on the host emulation: the bodies of
tests/test_gpu_head_dims.py on CPU tensors -- oracle parity in both dtypes, folded and unfolded, several queries per sample,
and in-place row-index pooling.  Small batches, and no D = 1536 case: a block's threads are fibers here, and the
emulated SIMT weight-gradient GEMMs of that width alone take a minute.
"""
import dataclasses

import pytest
import torch

from tests import test_gpu_head_dims as HD
from tests.emu_support import cuda_emulation  # noqa: F401  (fixture)
from tests.test_emu_parity import _cpu_stands_in_for_the_device  # noqa: F401  (autouse fixture: the device patch)

pytestmark = pytest.mark.usefixtures("cuda_emulation")


def small(case, B):
    return dataclasses.replace(case, B=B)


CASES = {c.name: c for c in HD.HEAD_DIM_CASES + HD.BF16_ONLY_CASES}


@pytest.mark.parametrize("name,B", [("hd48_d192_h4_m4_kpm", 6), ("hd80_d320_h4_m5_eval", 5), ("hd384_d384_h1_m3", 4),
                                    ("hd96_d768_h8_m3", 3)])
def test_fp32_matches_oracle(name, B):
    HD.test_fp32_matches_oracle(small(CASES[name], B))


@pytest.mark.parametrize("fold", [True, False], ids=["folded", "unfolded"])
@pytest.mark.parametrize("name,B", [("hd24_d240_h10_m3", 5), ("hd48_d384_h8_m3_dropout", 6), ("hd768_d768_h1_m3", 3)])
def test_bf16_masks_exact_against_stage_rounded_oracle(name, B, fold):
    HD.test_bf16_masks_exact_against_stage_rounded_oracle(small(CASES[name], B), fold)


@pytest.fixture
def multi_query():
    return True


def test_multi_query_fp32_and_bf16(multi_query):
    HD.test_multi_query_fp32_and_bf16(small(HD.MULTI_QUERY_CASES[0], 4))


@pytest.mark.parametrize("dtype,fold", [(torch.float32, True), (torch.bfloat16, False)], ids=["fp32_folded", "bf16_unfolded"])
def test_sample_index_pools_the_listed_rows_in_place(monkeypatch, dtype, fold):
    HD.test_sample_index_pools_the_listed_rows_in_place(monkeypatch, dtype, fold)
