"""Generate tests/golden/*.npz by running the UNMODIFIED reference on the shared cases.

Needs a checkout of the reference implementation, named by AECF_REFERENCE.  The reference's two random
draws are replaced by the shared Philox uniforms exactly as SURVEY.md Appendix C
describes -- both call sites resolve the function at call time:

  * curriculum mask:  ``torch.bernoulli(p)``             (reference aecf/AECFLayer.py:204)
  * attention dropout ``torch.nn.functional.dropout``    (torch/nn/functional.py:6645)

    AECF_REFERENCE=<reference checkout> python tests/golden/make_golden.py      # rewrites every fixture
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
MAX_FILE_BYTES = 1_000_000          # no committed fixture file is larger
sys.path.insert(0, ROOT)
REFERENCE = os.environ.get("AECF_REFERENCE", "")
if not os.path.isfile(os.path.join(REFERENCE, "aecf", "AECFLayer.py")):     # not this repository's alias package
    sys.exit("set AECF_REFERENCE to a checkout of the reference implementation")
sys.path.insert(0, REFERENCE)

import aecf as ref  # noqa: E402  (the reference package)

from tests.golden.cases import CASES, MULTI_QUERY_CASES, Case, build_inputs, masking_kwargs  # noqa: E402


from tests.golden.injection import inject_uniforms  # noqa: E402,F401


def run_reference(case: Case):
    dt = getattr(torch, case.dtype)
    inp = build_inputs(case)
    cm = ref.CurriculumMasking(**masking_kwargs(case))
    pool = ref.MultimodalAttentionPool(case.D, num_heads=case.H, dropout=case.dropout,
                                       curriculum_masking=cm, dtype=dt)
    with torch.no_grad():
        pool.attention.in_proj_weight.copy_(inp["in_proj_weight"])
        pool.attention.in_proj_bias.copy_(inp["in_proj_bias"])
        pool.attention.out_proj.weight.copy_(inp["out_proj.weight"])
        pool.attention.out_proj.bias.copy_(inp["out_proj.bias"])
    pool.train(case.training)
    multi = case.S > 1
    query0 = torch.nn.Parameter((inp["query"] if multi else inp["query0"]).clone())
    x = inp["x"].clone().requires_grad_(True)
    value = inp["value"].clone().requires_grad_(True) if case.separate_value else None
    kpm = inp.get("key_padding_mask")

    with inject_uniforms(inp["u_mask"], inp["u_drop"]):
        out, info = pool(query0 if multi else query0.expand(case.B, -1, -1), x, value, key_padding_mask=kpm,
                         return_info=True)
    ent_loss = cm.entropy_loss(info["entropy"])
    loss = (out * inp["grad_out"]).sum()
    if case.pooled_grad:
        loss = loss + (info["attention_weights"] * inp["grad_pooled"]).sum()
    if not case.training:
        loss = loss + 0.5 * info["entropy"].sum()          # eval: entropy carries gradient (:151-156)
    loss.backward()

    rec = {
        "out": out, "attention_weights": info["attention_weights"],
        "entropy": info["entropy"], "mask_rate": info["mask_rate"],
        "masked_attention_weights": info["masked_attention_weights"],
        "entropy_loss": ent_loss, "last_seq_len": torch.tensor(cm._last_seq_len),
        "grad_x": x.grad, ("grad_query" if multi else "grad_query0"): query0.grad,
        "grad_in_proj_bias": pool.attention.in_proj_bias.grad,
        "grad_out_proj_bias": pool.attention.out_proj.bias.grad,
    }
    if "target_entropy" in info:
        rec["target_entropy"] = info["target_entropy"]
    if value is not None:
        rec["grad_value"] = value.grad
    gwi, gwo = pool.attention.in_proj_weight.grad, pool.attention.out_proj.weight.grad
    if case.full_grads:
        rec["grad_in_proj_weight"], rec["grad_out_proj_weight"] = gwi, gwo
    else:   # large D: keep the fixture small -- row/column sums and a strided sample
        for name, g in (("in_proj_weight", gwi), ("out_proj_weight", gwo)):
            rec[f"grad_{name}_rowsum"] = g.sum(1)
            rec[f"grad_{name}_colsum"] = g.sum(0)
            rec[f"grad_{name}_strided"] = g.flatten()[::97]
    arrays = {k: v.detach().cpu().numpy() for k, v in rec.items()}
    arrays["info_keys"] = np.array(json.dumps(sorted(info.keys())))
    arrays["meta"] = np.array(json.dumps(case.meta()))
    arrays["torch_version"] = np.array(torch.__version__)
    return arrays


def main():
    torch.set_num_threads(1)
    for case in CASES + MULTI_QUERY_CASES:
        arrays = run_reference(case)
        path, more = os.path.join(HERE, case.name + ".npz"), os.path.join(HERE, case.name + ".more.npz")
        if os.path.exists(more):                      # tests/helpers.py load_golden would merge a stale one
            os.remove(more)
        np.savez_compressed(path, **arrays)
        if os.path.getsize(path) > MAX_FILE_BYTES:    # the out-projection weight gradient goes to a second file
            np.savez_compressed(more, grad_out_proj_weight=arrays.pop("grad_out_proj_weight"))
            np.savez_compressed(path, **arrays)
        ent = arrays["entropy"].reshape(-1)
        norm = ent / np.log(case.M) if case.M > 1 else ent
        q = np.quantile(norm, [0.1, 0.5, 0.9]) if ent.size else [0, 0, 0]
        print(f"{case.name:32s} {os.path.getsize(path) / 1024:8.1f} KiB  "
              f"norm-entropy q10/q50/q90 = {q[0]:.3f}/{q[1]:.3f}/{q[2]:.3f}  "
              f"mask_rate mean = {arrays['mask_rate'].mean():.4f}")


if __name__ == "__main__":
    main()
