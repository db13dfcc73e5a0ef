"""The bodies of tests/test_gpu_nonfinite.py on the host emulation (tests/cuda_emu), on CPU tensors: fully padded samples,
NaN gradients of the eval-mode entropy, the small kernels at their edges."""
import pytest
import torch

from tests import test_gpu_multi_query as MQ
from tests import test_gpu_nonfinite as N
from tests import test_gpu_parity as P
from tests.emu_support import cuda_emulation  # noqa: F401  (fixture)

pytestmark = pytest.mark.usefixtures("cuda_emulation")


@pytest.fixture(autouse=True)
def _cpu_stands_in_for_the_device(monkeypatch):
    """As in tests/test_emu_parity.py: ``t.to("cpu")`` of a CPU tensor is the tensor itself; make it a copy, so that no
    test's inputs collect the gradients of its runs."""
    for module in (P, MQ, N):
        monkeypatch.setattr(module, "DEV", "cpu")
    plain_to = torch.Tensor.to

    def to_copy(self, *args, **kwargs):
        moved = plain_to(self, *args, **kwargs)
        return moved.clone() if moved is self else moved

    monkeypatch.setattr(torch.Tensor, "to", to_copy)


@pytest.mark.parametrize("mode", list(N.MODES))
@pytest.mark.parametrize("pad", list(N.PADDINGS))
@pytest.mark.parametrize("fold", [False, True], ids=["unfolded", "folded"])
def test_fp32_fully_padded_samples(pad, mode, fold):
    N.test_fp32_fully_padded_samples(pad, mode, fold)


@pytest.mark.parametrize("mode", list(N.MODES))
@pytest.mark.parametrize("fold", [False, True], ids=["unfolded", "folded"])
def test_bf16_fully_padded_samples(mode, fold):
    N.test_bf16_fully_padded_samples("chunk_edges", mode, fold)


def test_fully_padded_sample_leaves_the_others_key_gradients_alone():
    N.test_fully_padded_sample_leaves_the_others_key_gradients_alone()


@pytest.mark.parametrize("batch_first", [True, False], ids=["batch_first", "seq_first"])
@pytest.mark.parametrize("case", N.MQ_PADDED, ids=lambda c: c.name)
def test_multi_query_fully_padded_samples(case, batch_first):
    N.test_multi_query_fully_padded_samples(case, batch_first)


@pytest.mark.parametrize("case", N.MQ_PADDED, ids=lambda c: c.name)
def test_multi_query_bf16_fully_padded_samples(case):
    N.test_multi_query_bf16_fully_padded_samples(case)


@pytest.mark.parametrize("dtype,fold", [(torch.float32, False), (torch.float32, True), (torch.bfloat16, True)],
                         ids=["fp32_unfolded", "fp32_folded", "bf16_folded"])
def test_sample_index_with_non_finite_samples(dtype, fold):
    N.test_sample_index_with_non_finite_samples(dtype, fold)


@pytest.mark.parametrize("fold", [False, True], ids=["unfolded", "folded"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_eval_entropy_gradient_at_padded_tokens(dtype, fold):
    N.test_eval_entropy_gradient_at_padded_tokens(dtype, fold)


def test_standalone_entropy_gradient_at_zero_weights():
    N.test_standalone_entropy_gradient_at_zero_weights()


@pytest.mark.parametrize("min_active", [1, 3, 70])
@pytest.mark.parametrize("L", [1, 2, 5, 33, 64])
def test_curriculum_mask_kernel_edges(L, min_active):
    N.test_curriculum_mask_kernel_edges(L, min_active)


@pytest.mark.parametrize("min_active", [1, 3, 70])
@pytest.mark.parametrize("L", [1, 2, 5, 33, 64])
def test_curriculum_mask_backward_edges(L, min_active):
    N.test_curriculum_mask_backward_edges(L, min_active)


def test_entropy_loss_over_several_passes_with_non_finite_entries():
    N.test_entropy_loss_over_several_passes_with_non_finite_entries()


@pytest.mark.parametrize("dtype,D", [(torch.float32, 128), (torch.float32, 1024), (torch.bfloat16, 512), (torch.bfloat16, 2048)],
                         ids=["fp32_128", "fp32_1024", "bf16_512", "bf16_2048"])
def test_sdpa_jmax(dtype, D):
    N.test_sdpa_every_jmax(dtype, D)


def test_colsum_many_rows_strided_and_bf16_out():
    N.test_colsum_many_rows_strided_and_bf16_out(torch.float32)
