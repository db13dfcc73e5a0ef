"""Shared helpers for the parity tests (CPU and GPU)."""
from __future__ import annotations

import json
import math
import os
from typing import Dict, Optional

import numpy as np
import torch

from oracle import aecf_oracle as oracle
from tests.golden.cases import Case, build_inputs, masking_kwargs

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(case: Case) -> Dict[str, np.ndarray]:
    with np.load(os.path.join(GOLDEN_DIR, case.name + ".npz")) as z:
        g = {k: z[k] for k in z.files}
    more = os.path.join(GOLDEN_DIR, case.name + ".more.npz")      # what did not fit in one file of at most 1 MB
    if os.path.exists(more):
        with np.load(more) as z:
            g.update({k: z[k] for k in z.files})
    assert json.loads(str(g["meta"])) == case.meta(), "fixture is stale: rerun tests/golden/make_golden.py"
    return g


def score_bias_from_kpm(kpm: Optional[torch.Tensor], dtype) -> Optional[torch.Tensor]:
    """torch turns a boolean key_padding_mask into an additive -inf mask (functional.py:6608-6620)."""
    if kpm is None:
        return None
    B, M = kpm.shape
    return torch.zeros(B, 1, 1, M, dtype=dtype).masked_fill(kpm.view(B, 1, 1, M), float("-inf"))


def run_oracle(case: Case, inp: Optional[dict] = None, dtype: Optional[torch.dtype] = None,
               storage: Optional[torch.dtype] = None, fold_key: bool = False):
    """Oracle forward + closed-form backward on a golden case; returns (forward result, grads)."""
    inp = inp if inp is not None else build_inputs(case, dtype)
    B, D, S = case.B, case.D, case.S
    q = inp["query"] if S > 1 else inp["query0"].expand(B, 1, D)       # S > 1: a query vector per (b, s)
    value = inp.get("value")
    fwd = oracle.pool_forward(
        q, inp["x"], value, inp["in_proj_weight"], inp["in_proj_bias"],
        inp["out_proj.weight"], inp["out_proj.bias"], case.H,
        dropout_p=case.dropout, training=case.training, u_drop=inp["u_drop"], u_mask=inp["u_mask"],
        score_bias=score_bias_from_kpm(inp.get("key_padding_mask"), inp["x"].dtype),
        masking=masking_kwargs(case), storage=storage, fold_key=fold_key, per_row_query_storage=S > 1)
    grads = oracle.pool_backward(
        q, inp["x"], value, inp["in_proj_weight"], inp["out_proj.weight"], case.H, fwd.saved,
        inp["grad_out"], grad_pooled=inp["grad_pooled"] if case.pooled_grad else None,
        grad_entropy=None if case.training else torch.full((B, S), 0.5, dtype=inp["x"].dtype),
        dropout_p=case.dropout, training=case.training, storage=storage, fold_key=fold_key,
        per_row_query_storage=S > 1)
    if S == 1:
        grads["query0"] = grads.pop("query").sum(0, keepdim=True)
    return fwd, grads


def finite_scale(t) -> float:
    """The largest magnitude among the finite elements of t (0 when there are none)."""
    t = torch.as_tensor(t).detach().double()
    t = t[torch.isfinite(t)]
    return float(t.abs().max()) if t.numel() else 0.0


def assert_close(name, got, want, rtol, atol=None):
    """got matches want: NaN exactly where want has NaN, +inf and -inf exactly where want has them, and the finite
    elements within atol + rtol |want|.  The default atol is rtol times the largest finite |want|.  A test that allows
    no non-finite value at all says so with torch.isfinite(...).all()."""
    got = torch.as_tensor(got).double().reshape(-1)
    want = torch.as_tensor(want).double().reshape(-1)
    assert got.shape == want.shape, f"{name}: shape {got.shape} vs {want.shape}"
    finite = torch.isfinite(want)
    same = torch.where(finite, torch.isfinite(got), torch.isnan(want) & torch.isnan(got) | (got == want))
    assert bool(same.all()), (
        f"{name}: non-finite pattern differs at {int((~same).sum())}/{got.numel()} elements, first at "
        f"{int((~same).nonzero()[0])} (got {int((~torch.isfinite(got)).sum())} non-finite, want {int((~finite).sum())})")
    if atol is None:                       # relative to the tensor's own scale
        atol = rtol * max(finite_scale(want), 1e-30)
    assert math.isfinite(atol), f"{name}: atol {atol} is not finite"
    got, want = got[finite], want[finite]
    err = (got - want).abs()
    bound = atol + rtol * want.abs()
    bad = err > bound
    assert not bool(bad.any()), (
        f"{name}: {int(bad.sum())}/{got.numel()} beyond rtol={rtol} atol={atol:.3e}; "
        f"max abs err {float(err.max()):.3e} (scale {finite_scale(want):.3e})")
