"""Host-side logic of the data-parallel layer on CPU: world_size 2 over gloo.

The compute inside each rank is the CPU oracle (the CUDA path needs a GPU); what is tested here is
what ``aecf_b200/dp.py`` adds -- row sharding, Philox offsets keyed on the global row, the flat fp32
gradient bucket and its one all-reduce -- i.e. that an N-rank run reproduces the 1-rank run.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from aecf_b200.dp import PARAM_ORDER, GradientSync, shard_rows
from oracle import aecf_oracle as oracle
from oracle import philox

WORLD = 2
B, M, D, H = 48, 3, 64, 8
SEED, OFFSET = 0x5EED, 11
MASKING = dict(base_mask_prob=0.6, entropy_target=0.7, min_active=1)


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _inputs():
    f = lambda seed, shape, scale=1.0: torch.from_numpy(philox.normal(seed, shape) * scale).float()
    return dict(Wi=f(1, (3 * D, D), 0.1), bi=f(2, (3 * D,), 0.05), Wo=f(3, (D, D), 0.1), bo=f(4, (D,), 0.05),
                q0=f(5, (1, 1, D), 0.2), x=f(6, (B, M, D)), g=f(7, (B, 1, D)))


def _step(t, row0, rows):
    """Oracle forward/backward on global rows [row0, row0 + rows) with the global-row Philox draws."""
    sl = slice(row0, row0 + rows)
    u_mask = torch.from_numpy(philox.mask_uniforms(SEED, OFFSET, row0, rows, M))
    u_drop = torch.from_numpy(philox.dropout_uniforms(SEED, OFFSET, row0, rows, H, M))
    q = t["q0"].expand(rows, 1, D)
    fwd = oracle.pool_forward(q, t["x"][sl], None, t["Wi"], t["bi"], t["Wo"], t["bo"], H, dropout_p=0.1, training=True,
                              u_drop=u_drop, u_mask=u_mask, masking=MASKING)
    grads = oracle.pool_backward(q, t["x"][sl], None, t["Wi"], t["Wo"], H, fwd.saved, t["g"][sl], dropout_p=0.1,
                                 training=True)
    grads["query"] = grads["query"].sum(0, keepdim=True)
    return fwd, grads


class _Params(torch.nn.Module):
    """Stand-in with the attribute layout GradientSync expects from MultimodalAttentionPool."""

    def __init__(self, t):
        super().__init__()
        self.attention = torch.nn.Module()
        self.attention.in_proj_weight = torch.nn.Parameter(t["Wi"].clone())
        self.attention.in_proj_bias = torch.nn.Parameter(t["bi"].clone())
        self.attention.out_proj = torch.nn.Module()
        self.attention.out_proj.weight = torch.nn.Parameter(t["Wo"].clone())
        self.attention.out_proj.bias = torch.nn.Parameter(t["bo"].clone())
        self.row_offset = 0
        self._grad_ready = None
        self._grad_buffers = None


def _worker(rank, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=WORLD)
    try:
        t = _inputs()
        pool = _Params(t)
        query = torch.nn.Parameter(t["q0"].clone())
        sync = GradientSync(pool, query, average=False).attach()
        row0, rows = sync.set_shard(B)
        assert pool.row_offset == row0 and pool._grad_ready is not None and set(pool._grad_buffers) == set(PARAM_ORDER)
        fwd, grads = _step(t, row0, rows)
        # report in the order the fused backward produces them: out_proj first, in_proj and query last
        for name in PARAM_ORDER:
            if name == "query":
                sync._query_hook(grads[name])
            elif name == "in_proj_weight":                # what the fused backward does: write in place
                pool._grad_buffers[name].copy_(grads[name])
                pool._grad_ready(name, pool._grad_buffers[name])
            else:                                         # a gradient produced elsewhere is copied in
                pool._grad_ready(name, grads[name])
            # nothing is reduced yet: the whole bucket is reduced once, in finish()
            assert not sync.bucket_is_reduced and name in sync.reported
            assert torch.equal(sync.views[name], grads[name].reshape(sync.views[name].shape))
        sync.finish()
        assert sync.bucket_is_reduced and not sync.reported
        assert pool.attention.in_proj_weight.grad.data_ptr() == pool._grad_buffers["in_proj_weight"].data_ptr()
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), row0=row0, rows=rows,
                 mask=fwd.info["mask"].numpy(), out=fwd.out.numpy(),
                 **{f"g_{n}": p.grad.numpy() for n, p in sync.params.items()})
    finally:
        dist.destroy_process_group()


def test_two_ranks_reproduce_one_rank(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(port, str(tmp_path)), nprocs=WORLD, join=True)
    t = _inputs()
    full_fwd, full_grads = _step(t, 0, B)
    shards = [np.load(tmp_path / f"rank{r}.npz") for r in range(WORLD)]
    assert [int(s["row0"]) for s in shards] == [0, B // 2] and sum(int(s["rows"]) for s in shards) == B
    # masks and outputs of the shards are the full batch's, bit for bit (Philox keyed on the global row)
    assert np.array_equal(np.concatenate([s["mask"] for s in shards]), full_fwd.info["mask"].numpy())
    assert np.array_equal(np.concatenate([s["out"] for s in shards]), full_fwd.out.numpy())
    # every rank ends with the same summed gradients, equal to the 1-rank gradients
    for name in PARAM_ORDER:
        a, b = shards[0][f"g_{name}"], shards[1][f"g_{name}"]
        assert np.array_equal(a, b), name
        want = full_grads[name].numpy().reshape(a.shape)
        scale = max(float(np.abs(want).max()), 1e-12)
        assert float(np.abs(a - want).max()) <= 1e-5 * scale + 1e-7, name


def test_shard_rows_cover_the_batch_exactly():
    for batch in (1, 7, 64, 65536, 1000003):
        for world in (1, 2, 3, 4, 8):
            pieces = [shard_rows(batch, r, world) for r in range(world)]
            assert pieces[0][0] == 0 and sum(n for _, n in pieces) == batch
            for (s0, n0), (s1, _) in zip(pieces, pieces[1:]):
                assert s0 + n0 == s1
            assert max(n for _, n in pieces) - min(n for _, n in pieces) <= 1


def test_single_process_sync_leaves_gradients_alone():
    t = _inputs()
    pool = _Params(t)
    query = torch.nn.Parameter(t["q0"].clone())
    sync = GradientSync(pool, query).attach()
    g = torch.randn_like(pool.attention.out_proj.weight)
    pool.attention.out_proj.weight.grad = g.clone()
    pool._grad_ready("out_proj.weight", g * 3)          # ignored: there is nobody to reduce with
    sync.finish()
    assert torch.equal(pool.attention.out_proj.weight.grad, g) and not sync.reported


# ---- gradient accumulation (ADVICE r1, high): param.grad lives in the bucket after finish() ------------------------------
def _backward_like_the_fused_pool(pool, sync, grads):
    """What FusedPoolFunction.backward + autograd's AccumulateGrad do with the sync's buffers: ask for a place to write
    each gradient, report it, then either install it as .grad or add it to .grad in place."""
    for name in ("out_proj.bias", "out_proj.weight", "in_proj_weight", "in_proj_bias"):
        param = sync.params[name]
        buf = pool._grad_buffers.get(name)
        new = grads[name].clone() if buf is None else buf.copy_(grads[name])
        pool._grad_ready(name, new)
        if param.grad is None:
            param.grad = new
        else:
            param.grad += new


def _accumulate_worker(rank, port, out_dir, mode):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=WORLD)
    try:
        t = _inputs()
        pool = _Params(t)
        sync = GradientSync(pool, None, average=(mode == "mean_every_microbatch")).attach()
        g1 = {n: torch.full_like(p, 1.0 + rank) for n, p in sync.params.items()}
        g2 = {n: torch.full_like(p, 10.0 * (1 + rank)) for n, p in sync.params.items()}
        if mode == "no_sync_then_sync":                      # DDP's no_sync pattern: reduce once, after the last micro-batch
            sync.enabled = False
            _backward_like_the_fused_pool(pool, sync, g1); sync.finish()
            sync.enabled = True
            _backward_like_the_fused_pool(pool, sync, g2); sync.finish()
            want = (1.0 + 2.0) + (10.0 + 20.0)               # sum over ranks of g1 + g2
        elif mode == "mean_every_microbatch":                # every micro-batch averaged over the ranks, then accumulated
            _backward_like_the_fused_pool(pool, sync, g1); sync.finish()
            _backward_like_the_fused_pool(pool, sync, g2); sync.finish()
            want = 1.5 + 15.0
        elif mode == "zero_grad_in_place":                   # zero_grad(set_to_none=False): .grad stays in the bucket, zeroed
            _backward_like_the_fused_pool(pool, sync, g1); sync.finish()
            for p in sync.params.values():
                p.grad.zero_()
            _backward_like_the_fused_pool(pool, sync, g2); sync.finish()
            want = 10.0 + 20.0
        elif mode == "sum_every_microbatch":                 # only the new gradient is summed, not the summed one again
            _backward_like_the_fused_pool(pool, sync, g1); sync.finish()
            _backward_like_the_fused_pool(pool, sync, g2); sync.finish()
            want = (1.0 + 2.0) + (10.0 + 20.0)
        else:                                                # zero in place, then the no_sync pattern
            _backward_like_the_fused_pool(pool, sync, g1); sync.finish()
            for p in sync.params.values():
                p.grad.zero_()
            sync.enabled = False
            _backward_like_the_fused_pool(pool, sync, g1); sync.finish()
            sync.enabled = True
            _backward_like_the_fused_pool(pool, sync, g2); sync.finish()
            want = (1.0 + 2.0) + (10.0 + 20.0)
        ok = all(bool((p.grad == want).all()) for p in sync.params.values())
        with open(os.path.join(out_dir, f"rank{rank}.txt"), "w") as f:
            f.write("ok" if ok else f"got {float(sync.params['out_proj.bias'].grad[0])} want {want}")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["no_sync_then_sync", "mean_every_microbatch", "zero_grad_in_place", "sum_every_microbatch", "zero_in_place_then_no_sync"])
def test_gradient_accumulation_with_the_bucket_attached(tmp_path, mode):
    mp.spawn(_accumulate_worker, args=(_free_port(), str(tmp_path), mode), nprocs=WORLD, join=True)
    for r in range(WORLD):
        assert open(tmp_path / f"rank{r}.txt").read() == "ok"


def test_a_grad_tensor_of_its_own_is_refused():
    t = _inputs()
    pool = _Params(t)
    GradientSync(pool, None).attach()
    pool.attention.out_proj.weight.grad = torch.zeros_like(pool.attention.out_proj.weight)
    with pytest.raises(RuntimeError, match="set_to_none=True"):
        pool._grad_buffers.get("out_proj.weight")
