"""The mixed-precision bodies of tests/test_gpu_mixed_precision.py on CPU tensors, through the host emulation of the CUDA
sources (tests/cuda_emu), at small sizes.  The CUDA-graph, data-parallel and headline-size bodies need the device."""
import pytest

from tests import test_gpu_mixed_precision as G
from tests.emu_support import cuda_emulation  # noqa: F401  (fixture)

pytestmark = pytest.mark.usefixtures("cuda_emulation")


@pytest.fixture(autouse=True)
def _small(monkeypatch):
    monkeypatch.setattr(G, "DEV", "cpu")
    monkeypatch.setattr(G, "B", 24)
    monkeypatch.setattr(G, "D", 64)
    monkeypatch.setattr(G, "H", 4)
    monkeypatch.setattr(G, "D_PAD", 96)
    monkeypatch.setattr(G, "H_PAD", 1)


@pytest.mark.parametrize("case", list(G.CASES))
def test_mixed_matches_bf16_twin(case):
    G.test_mixed_matches_bf16_twin(case)


def test_param_cast_rounds_like_tensor_bfloat16():
    G.test_param_cast_rounds_like_tensor_bfloat16()


def test_mixed_gradients_closer_to_oracle_than_bf16():
    G.test_mixed_gradients_closer_to_oracle_than_bf16()


def test_mixed_projections_match_bf16_twin():
    G.test_mixed_projections_match_bf16_twin()


def test_mixed_rejections_stay():
    G.test_mixed_rejections_stay()
