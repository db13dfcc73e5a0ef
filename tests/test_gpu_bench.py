"""bench.py --dump-outputs on the GPU: the last timed step's outputs as float32 .npy files within 64 MB, checked against
the oracle on bench.py's own seeded inputs, for the graph-replayed and for the eager step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import aecf_b200
from oracle import aecf_oracle as oracle
from tests.helpers import assert_close

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, M, D, H = 65536, 3, 512, 8          # bench.py's default workload: one input batch, larger than the L2


def _bench_dump(out_dir, graph):
    args = ["--steps", "3", "--warmup", "2", "--graph", graph, "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 3 and line["value"] > 0 and line["cuda_graph"] == (graph == "on")
    return {p[:-4]: np.load(os.path.join(out_dir, p)) for p in sorted(os.listdir(out_dir))}


def _oracle_step():
    """bench.py's seeded parameters, input batch and upstream gradient through the oracle in fp32.  Without dropout
    the output, the pooled weights and the gradients of out.backward(d_out) do not depend on the curriculum-mask draws."""
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    query, pool = aecf_b200.create_fusion_pool(D, M, 0.15, num_heads=H, device=dev, dtype=torch.bfloat16)
    torch.manual_seed(1234)
    x = torch.randn(B, M, D, device=dev, dtype=torch.bfloat16)
    d_out = torch.randn(B, 1, D, device=dev, dtype=torch.bfloat16)
    att = pool.attention
    with torch.no_grad():
        q, wi, wo = query.float().expand(B, 1, D), att.in_proj_weight.float(), att.out_proj.weight.float()
        fwd = oracle.pool_forward(q, x.float(), None, wi, att.in_proj_bias.float(), wo, att.out_proj.bias.float(), H)
        grads = oracle.pool_backward(q, x.float(), None, wi, wo, H, fwd.saved, d_out.float())
    return {"out": fwd.out.cpu(), "attention_weights": fwd.pooled.cpu(), "grad_x": grads["key"].cpu(),
            "grad_query": grads["query"].sum(0, keepdim=True).cpu(), "grad_attention.in_proj_weight": grads["in_proj_weight"].cpu(),
            "grad_attention.out_proj.weight": grads["out_proj.weight"].cpu()}


@pytest.mark.parametrize("graph", ["on", "off"])
def test_dump_outputs_of_the_last_timed_step(tmp_path, graph):
    got = _bench_dump(tmp_path, graph)
    assert {"out", "attention_weights", "masked_attention_weights", "entropy", "mask_rate", "entropy_loss", "grad_x", "grad_query",
            "grad_attention.in_proj_weight", "grad_attention.out_proj.weight"} <= set(got)
    assert sum(v.nbytes for v in got.values()) <= 64 << 20
    for name, v in got.items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), name
    assert got["grad_attention.in_proj_weight"].shape == (3 * D, D) and got["grad_x"].shape[1:] == (M, D)

    want = _oracle_step()
    assert got["attention_weights"].shape == (B, 1, M) and got["out"].shape[1:] == (1, D)
    for name, w in want.items():
        g = got[name]
        if g.shape[0] < w.shape[0]:                      # a per-row array bench.py cut to its seeded sample of rows
            w = w[torch.from_numpy(np.sort(np.random.default_rng(0).permutation(w.shape[0])[:g.shape[0]]))]
        assert_close(name, g, w, 2e-2)
