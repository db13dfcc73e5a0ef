"""The tcgen05 / TMEM / TMA projection GEMM on the CPU: gemm_tcgen05.cu compiled for the host emulation, with the
functional model of tests/cuda_emu/tcgen05_emu.h behind its inline-PTX wrappers (mbarriers, tiled TMA with the 128-byte
swizzle, cluster multicast, tensor memory, tcgen05.mma through the shared-memory / instruction descriptors,
cta_group::2).  The model's layouts are validated by the kernels measured on hardware computing correct products under
it.  It sees what a functional model can see -- barrier counts and phases (a wrong count deadlocks the emulation), tile /
box / column indexing, staging layout, a staging box refilled before the wait that protects it -- not missing fences, and
not speed.  (Round 1 used it to pre-check five kernel variants before their first hardware run; round 2 measured them,
kept the pipelined epilogue and deleted the rest -- profiles/r2_gemm_where_the_time_goes.md.)
"""
import os
import subprocess
import sys

import pytest
import torch

from aecf_b200 import _lib
from tests import test_gpu_gemm_tcgen05 as G
from tests import test_gpu_parity as P
from tests.emu_support import cuda_emulation  # noqa: F401  (fixture)
from tests.golden.cases import Case

pytestmark = pytest.mark.usefixtures("cuda_emulation")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# one tile; BN = 256; a cluster of two with multicast; ragged everywhere (zero fill, clipped stores); three 256-wide column
# tiles and three tiles per CTA (both accumulators re-used); cta_group::2 (10 k-blocks); split-K with a ragged k tail
# several row-block groups per CTA pair with two column tiles each (the resident-A-panel kernel's slot hand-over)
SHAPES = [(128, 128, 64), (256, 256, 64), (384, 256, 128), (200, 136, 72), (392, 520, 200), (512, 256, 640), (300, 512, 4100),
          (1024, 512, 128), (512, 512, 520)]         # ... and nine k-blocks, the last one ragged: the dX contraction
LAYOUTS = [(_lib.K_MAJOR, _lib.K_MAJOR), (_lib.K_MAJOR, _lib.MN_MAJOR), (_lib.MN_MAJOR, _lib.MN_MAJOR), (_lib.MN_MAJOR, _lib.K_MAJOR)]


@pytest.fixture(autouse=True)
def _cpu_stands_in_for_the_device(monkeypatch):
    monkeypatch.setattr(G, "DEV", "cpu")
    monkeypatch.setattr(P, "DEV", "cpu")
    plain_to = torch.Tensor.to
    monkeypatch.setattr(torch.Tensor, "to", lambda self, *a, **k: (lambda r: r.clone() if r is self else r)(plain_to(self, *a, **k)))


@pytest.mark.parametrize("layouts", LAYOUTS, ids=["aK_bK", "aK_bMN", "aMN_bMN", "aMN_bK"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_kernels(shape, layouts):
    G.test_tcgen05_gemm(shape, *layouts)


def test_cta_pair_kernels_with_an_odd_number_of_row_blocks():
    """TMA stores of the emulation read their staging box at the latest moment the kernel allows.  Five row blocks on CTA
    pairs leave a filler tile; every epilogue round commits one (possibly empty) bulk group, so `wait_group.read 1` keeps
    protecting the buffer of the previous tile's last store.  (The round-1 instantiation without that commit failed here.)"""
    G.test_tcgen05_gemm((640, 256, 640), _lib.K_MAJOR, _lib.K_MAJOR)


def test_strided_operands_and_kernel_choice():
    G.test_tcgen05_strided_output_and_operand_views()
    G.test_tcgen05_is_what_auto_picks_for_the_projection_shapes()


@pytest.mark.parametrize("shape", [(640, 512, 512, 8), (300, 256, 128, 4)], ids=lambda s: "x".join(map(str, s)))
def test_side_output(shape):
    P.test_gemm_with_side_output(shape, torch.bfloat16)


def test_whole_step_on_the_tensor_core_gemms():
    """B*M = 480 rows: the folded forward (192-wide tiles, fp32 score side output), the K = D + 8 contraction of dX and the
    split-K weight gradients all take the tcgen05 kernels, against the stage-rounded oracle with bit-exact masks."""
    case = Case("emu_d256_h8_m3_b160", B=160, M=3, D=256, H=8, dropout=0.1, pooled_grad=True, data_seed=77, offset=4)
    P.test_bf16_masks_exact_against_stage_rounded_oracle(case, True)
    P.test_bf16_masks_exact_against_stage_rounded_oracle(case, False)


def test_reported_kernel():
    """aecf_gemm_last_kernel() names what ran (bench.py records it per launch site)."""
    from aecf_b200 import ops
    bf = torch.bfloat16
    a, b = torch.randn(512, 128, dtype=bf), torch.randn(256, 128, dtype=bf)
    ops.gemm(a, b, m=512, n=256, k=128, a_layout=_lib.K_MAJOR, b_layout=_lib.K_MAJOR, lda=128, ldb=128)           # 2 k-blocks
    assert _lib.gemm_last_kernel() == "tcgen05 1sm bn256 cluster2 splits1"
    a, b = torch.randn(512, 640, dtype=bf), torch.randn(256, 640, dtype=bf)
    ops.gemm(a, b, m=512, n=256, k=640, a_layout=_lib.K_MAJOR, b_layout=_lib.K_MAJOR, lda=640, ldb=640)           # 10 k-blocks
    assert _lib.gemm_last_kernel() == "tcgen05 2sm bn256 splits1"
    a, b = torch.randn(640, 512, dtype=bf), torch.randn(520, 512, dtype=bf)
    ops.gemm_aux(a, b, m=640, n=512, k=512, aux_cols=8)
    assert _lib.gemm_last_kernel() == "tcgen05 1sm bn192 cluster2 splits1"
    ops.gemm(a[:64].float(), b[:64].float(), m=64, n=64, k=512, a_layout=_lib.K_MAJOR, b_layout=_lib.K_MAJOR, lda=512, ldb=512)
    assert _lib.gemm_last_kernel() == "simt"
