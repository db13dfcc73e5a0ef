"""tests/helpers.py::assert_close sees non-finite values: NaN and infinities must sit exactly where the reference has them,
and the finite elements are compared on the scale of the finite reference elements."""
import math

import pytest
import torch

from tests.helpers import assert_close, finite_scale

NAN, INF = float("nan"), float("inf")


@pytest.mark.parametrize("got,want", [
    ([NAN, 1.0], [1.0, 1.0]),             # NaN from the kernel where the reference is finite
    ([5.0, -7.0], [NAN, 1.0]),            # a NaN in the reference must not switch the check off for the rest
    ([1.0, 1.0], [NAN, 1.0]),             # ... nor accept a finite value where the reference is NaN
    ([1e30, 1.0], [INF, 1.0]),            # an infinity in the reference accepts no finite value
    ([-INF, 1.0], [INF, 1.0]),            # infinities of the other sign
    ([NAN, 1.0], [INF, 1.0]),
    ([INF, 1.0], [NAN, 1.0]),
    ([INF, 1.0], [1.0, 1.0]),
], ids=["nan_got", "nan_want_finite_elsewhere_wrong", "finite_where_nan", "finite_where_inf", "inf_sign",
        "nan_where_inf", "inf_where_nan", "inf_got"])
def test_non_finite_mismatches_fail(got, want):
    with pytest.raises(AssertionError):
        assert_close("x", got, want, 1e-6)


def test_same_pattern_and_close_finite_values_pass():
    want = torch.tensor([NAN, INF, -INF, 1.0, -2.0, 0.0])
    assert_close("x", want + torch.tensor([0, 0, 0, 1e-7, -1e-7, 1e-7]), want, 1e-6)
    assert_close("x", want.float(), want.double(), 1e-6)


def test_scale_comes_from_the_finite_elements():
    """The default atol is rtol times the largest finite |want|: an infinity does not widen it to everything, and the
    explicit form reads the same scale."""
    want = torch.tensor([INF, 1.0, 0.0])
    assert_close("x", [INF, 1.0, 5e-7], want, 1e-6)
    with pytest.raises(AssertionError):
        assert_close("x", [INF, 1.0, 5e-6], want, 1e-6)
    assert finite_scale(torch.tensor([NAN, -3.0, INF, 2.0])) == 3.0
    assert finite_scale(torch.tensor([NAN, INF])) == 0.0


def test_a_non_finite_explicit_atol_is_refused():
    with pytest.raises(AssertionError, match="atol"):
        assert_close("x", [1.0, 100.0], [1.0, 1.0], 1e-6, atol=math.nan)
