"""The stand-alone folded backward chain of tests/test_gpu_fold_chain.py on CPU tensors, through the host emulation of
the CUDA sources (tests/cuda_emu)."""
import pytest

from tests import test_gpu_fold_chain as F
from tests.emu_support import cuda_emulation  # noqa: F401  (fixture)

pytestmark = pytest.mark.usefixtures("cuda_emulation")


def test_standalone_folded_backward_chain_matches_oracle(monkeypatch):
    monkeypatch.setattr(F, "DEV", "cpu")
    F.test_standalone_folded_backward_chain_matches_oracle()
