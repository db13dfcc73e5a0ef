"""Batch-sharded data parallelism end to end on CPU: world_size 2 over gloo, every rank running the PRODUCT path --
MultimodalAttentionPool -> C ABI -> the CUDA sources under the host emulation (tests/cuda_emu) -- with
``GradientSync`` attached, against the same step on one rank.  tests/test_dp_gloo.py checks dp.py's host logic with
the oracle as the compute; here the fused backward itself writes its gradients into the bucket.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.golden.cases import CASES_BY_NAME, PHILOX_SEED, build_inputs, masking_kwargs

WORLD = 2
CASE = CASES_BY_NAME["d64_h8_m3_dropout"]
PARAMS = ("in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias")


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _step(dtype, fold, rank, world):
    """One training step of this rank's shard of CASE through the module API; returns arrays to compare."""
    import aecf_b200
    from aecf_b200.dp import GradientSync
    inp = build_inputs(CASE)
    cm = aecf_b200.CurriculumMasking(**masking_kwargs(CASE))
    pool = aecf_b200.MultimodalAttentionPool(CASE.D, num_heads=CASE.H, dropout=CASE.dropout, curriculum_masking=cm, dtype=dtype)
    with torch.no_grad():
        for name in PARAMS:
            obj = pool.attention
            for part in name.split(".")[:-1]:
                obj = getattr(obj, part)
            getattr(obj, name.split(".")[-1]).copy_(inp[name])
    pool.fold_key_projection = fold
    pool._want_mask_bits = True
    query = torch.nn.Parameter(inp["query0"].to(dtype).clone())
    sync = GradientSync(pool, query, average=False).attach()
    row0, rows = sync.set_shard(CASE.B)
    sl = slice(row0, row0 + rows)
    x = inp["x"][sl].to(dtype).clone().requires_grad_(True)
    aecf_b200.set_rng_state(PHILOX_SEED, CASE.offset)
    out, info = pool(query.expand(rows, -1, -1), x, return_info=True)
    loss = (out.float() * inp["grad_out"][sl]).sum() + (info["attention_weights"] * inp["grad_pooled"][sl]).sum()
    loss.backward()
    sync.finish()
    got = {"row0": row0, "rows": rows, "out": out.detach().float().numpy(), "bits": info["mask_bits"].numpy(),
           "g_x": x.grad.float().numpy(), "g_query": query.grad.float().numpy()}
    for name in PARAMS:
        obj = pool.attention
        for part in name.split("."):
            obj = getattr(obj, part)
        got["g_" + name] = obj.grad.float().numpy()
        assert world == 1 or obj.grad.data_ptr() == sync.views[name].data_ptr()       # written in place into the bucket
    return got


def _worker(rank, port, out_dir, dtype, fold):
    from tests.emu_support import enable_in_this_process
    enable_in_this_process()
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=WORLD)
    try:
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **_step(dtype, fold, rank, WORLD))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("dtype,fold", [(torch.float32, True), (torch.bfloat16, None)], ids=["fp32_folded", "bf16_default"])
def test_two_emulated_ranks_reproduce_one(tmp_path, dtype, fold):
    from tests.emu_support import enable_in_this_process, load_emulation
    load_emulation()                                     # build once, before the workers race for it
    mp.spawn(_worker, args=(_free_port(), str(tmp_path), dtype, fold), nprocs=WORLD, join=True)
    shards = [np.load(tmp_path / f"rank{r}.npz") for r in range(WORLD)]
    assert sum(int(s["rows"]) for s in shards) == CASE.B and int(shards[1]["row0"]) == int(shards[0]["rows"])

    import aecf_b200
    from aecf_b200 import _lib, ops
    saved = (_lib._lib, ops.require_cuda, ops._stream, torch.cuda.is_current_stream_capturing, torch.cuda.synchronize)
    try:
        enable_in_this_process()
        full = _step(dtype, fold, 0, 1)
    finally:
        _lib._lib, ops.require_cuda, ops._stream, torch.cuda.is_current_stream_capturing, torch.cuda.synchronize = saved
        aecf_b200.set_rng_state(None)
    # per-sample results of the shards are the full batch's bit for bit: Philox is keyed on the GLOBAL row
    for key in ("out", "bits", "g_x"):
        assert np.array_equal(np.concatenate([s[key] for s in shards]), full[key]), key
    # every rank ends with the same summed parameter gradients, equal to the one-rank gradients up to summation order
    tol = 1e-5 if dtype == torch.float32 else 2e-2
    for name in PARAMS + ("query",):
        a, b = shards[0]["g_" + name], shards[1]["g_" + name]
        assert np.array_equal(a, b), name
        want = full["g_" + name].reshape(a.shape)
        assert float(np.abs(a - want).max()) <= tol * max(float(np.abs(want).max()), 1e-12) + 1e-7, name
