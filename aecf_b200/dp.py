"""Batch-sharded data parallelism for the fusion pool: one process per GPU, NVLink between them.

The reference has no distributed code (SURVEY.md section 2.2); this layer is the north_star's item (3).
Samples are independent in the forward and in every activation gradient, so ranks only meet in one sum of the
fusion parameter gradients per step (1 051 136 parameters at D = 512).

  * rank r owns global rows [r*B/N, (r+1)*B/N); ``pool.row_offset`` keys the Philox counters on the
    GLOBAL row, so any N reproduces the 1-GPU masks and dropout bit for bit
  * ``collective="fused"`` (the default on CUDA with the folded key projection): the sum happens INSIDE the backward.
    The backward's gradient tail (csrc/grad_tail.cu) leaves the raw fp32 sums -- [dWv ; R], dWo, colsum(d_out), the pool
    kernel's bias sums, half as many numbers as there are parameters -- in a buffer every rank has mapped (CUDA IPC); one
    kernel per rank then sums them over the ranks through NVLink peer loads (flag barrier, rank r sums slice r in rank
    order and stores it to every rank, flag barrier) and only then are they converted to the parameter dtype.  The whole
    tail runs on a side stream next to the dX product, so nothing of it is on the critical path, and the gradients are
    summed in fp32 whatever the parameter dtype: an N-rank run rounds once, like a 1-rank run.  ``finish()`` is a no-op.
  * ``collective="nccl"`` / ``"peer"``: the backward writes its parameter gradients into one flat bucket (no copies) and
    ``finish()`` reduces it with ONE all-reduce after the backward -- ``torch.distributed`` (NCCL on the GPUs, gloo in the
    CPU tests of the host logic) or ``PeerAllReduce`` (csrc/peer_allreduce.cu).  This is also what runs wherever the
    fused tail does not apply (unfolded key projection, per-row queries).
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Tuple

import torch
import torch.distributed as dist

PARAM_ORDER = ("out_proj.bias", "out_proj.weight", "in_proj_weight", "in_proj_bias", "query")


def shard_rows(global_batch: int, rank: int, world_size: int) -> Tuple[int, int]:
    """(first global row, row count) of ``rank``: contiguous, sizes differ by at most one."""
    base, extra = divmod(global_batch, world_size)
    start = rank * base + min(rank, extra)
    return start, base + (1 if rank < extra else 0)


_imported: Dict[bytes, int] = {}          # IPC handle bytes -> base address in this process (a handle is opened once)


def _map_peer_tensors(tensors: List[torch.Tensor], group=None) -> List[List[int]]:
    """Collective: every rank exports ``tensors`` (CUDA, kept alive by the caller) through CUDA IPC -- 64-byte handle of the
    allocation each one lies in plus its offset, gathered with ``all_gather_object`` -- and opens every other rank's in the
    context of ITS OWN device (``aecf_peer_import``), so that kernels of this rank can address them.  Returns, per tensor,
    the W device ADDRESSES of its instances as seen from this process (own rank: ``tensor.data_ptr()``)."""
    import ctypes as C

    from . import _lib
    lib = _lib.load()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = tensors[0].device
    torch.cuda.synchronize(dev)
    exported = []
    for t in tensors:
        handle, offset = (C.c_char * 64)(), C.c_int64(0)
        _lib.check(lib.aecf_peer_export(dev.index or 0, t.data_ptr(), handle, C.byref(offset)), "aecf_peer_export")
        exported.append((bytes(handle), int(offset.value)))
    gathered = [None] * world
    dist.all_gather_object(gathered, (exported, dev.index or 0), group=group)
    out: List[List[int]] = [[] for _ in tensors]
    for r, (handles, peer_dev) in enumerate(gathered):
        if r == rank:
            for i, t in enumerate(tensors):
                out[i].append(t.data_ptr())
            continue
        _lib.check(lib.aecf_peer_enable_access(dev.index or 0, peer_dev), f"peer access {dev.index} -> {peer_dev}")
        for i, (handle, offset) in enumerate(handles):
            base = _imported.get(handle)
            if base is None:
                ptr = C.c_void_p()
                _lib.check(lib.aecf_peer_import(dev.index or 0, handle, C.byref(ptr)), f"aecf_peer_import (rank {r})")
                base = _imported[handle] = int(ptr.value)
            out[i].append(base + offset)
    dist.barrier(group=group)                            # everybody has mapped everything before anybody signals
    return out


def compute_dtype_of(pool) -> torch.dtype:
    """The dtype the folded backward of ``pool`` runs in by default: its parameter dtype -- except for fp32 parameters
    whose key projection is not forced to fold, where the folded backward only runs in mixed precision, on bf16 inputs."""
    dtype = pool.attention.in_proj_weight.dtype
    if dtype == torch.float32 and getattr(pool, "fold_key_projection", None) is not True:
        return torch.bfloat16
    return dtype


class FusedGradSum:
    """The cross-rank gradient sum of the folded backward (``aecf_dp_desc``): raw-sum and reduced-sum buffers of every
    rank mapped into this process, plus the flag blocks of the kernel's two barriers.  Construction is collective.
    The pool's backward passes ``pointer()`` to ``aecf_fusion_bwd`` whenever ``usable(desc)``."""

    def __init__(self, pool, group=None, average: bool = True, *, local_ranks: Optional[Tuple[int, int, list, list]] = None,
                 compute_dtype: Optional[torch.dtype] = None):
        """``local_ranks = (rank, world, buffers, flag blocks)``: W ranks EMULATED on one device (tests): the W buffers
        (``None`` entries are allocated) and flag blocks are plain local tensors shared by the W instances, no IPC.
        ``compute_dtype``: the dtype the backward runs in, which sets the layout of the raw sums (``compute_dtype_of``)."""
        import ctypes as C

        from . import _lib, ops
        att = pool.attention
        dev = att.in_proj_weight.device
        dtype = compute_dtype or compute_dtype_of(pool)
        if local_ranks is not None:
            self.rank, self.world = local_ranks[0], local_ranks[1]
        else:
            self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > 8:
            raise ValueError("the fused gradient sum covers the (at most 8) GPUs of one NVLink node")
        probe = ops.make_pool_desc(dev, dtype, batch=1, num_tokens=2, embed_dim=pool.embed_dim, num_heads=pool.num_heads,
                                   training=True, masking=0, min_active=1, q_is_shared=True, base_mask_prob=0.15,
                                   entropy_target=0.7, dropout_p=0.0, seed=0, offset=0, row0=0, fold_key=True)
        self.floats = ops.fusion_grad_sums_floats(probe)
        if self.floats == 0:
            raise ValueError("this pool has no fused gradient tail (the folded key projection does not apply)")
        self.embed_dim, self.num_heads, self.dtype = pool.embed_dim, pool.num_heads, dtype
        if local_ranks is not None:
            buffers, flags = local_ranks[2], local_ranks[3]
            for r in range(self.world):
                if buffers[r] is None:
                    buffers[r] = torch.zeros(2 * self.floats, dtype=torch.float32, device=dev)
                    flags[r] = ops.peer_flag_block(dev)
            self.buffer, self.flags = buffers[self.rank], flags[self.rank]
            self._keep = (buffers, flags)
            buffer_ptrs, flag_ptrs = [b.data_ptr() for b in buffers], [f.data_ptr() for f in flags]
        else:
            self.buffer = torch.zeros(2 * self.floats, dtype=torch.float32, device=dev)      # [raw sums | reduced sums]
            self.flags = ops.peer_flag_block(dev)
            buffer_ptrs, flag_ptrs = _map_peer_tensors([self.buffer, self.flags], group)
        n = self.floats * 4
        self._sums = (C.c_void_p * self.world)(*buffer_ptrs)
        self._reduced = (C.c_void_p * self.world)(*[b + n for b in buffer_ptrs])
        self._flags = (C.c_void_p * self.world)(*flag_ptrs)
        self._desc = _lib.DpDesc(world=self.world, rank=self.rank, average=int(average), reserved0=0,
                                 sums=self._sums, reduced=self._reduced, flags=self._flags)
        self._ptr = C.pointer(self._desc)
        self.ran = False                                 # set by the backward that used it (GradientSync.finish looks)

    def usable(self, desc) -> bool:
        """Whether the backward of ``desc`` can sum through these buffers: its raw sums must have the layout they were sized
        for (embed_dim, num_heads and the compute dtype, whose 16-byte rounding of the heads sets the columns of R)."""
        from . import ops
        return (self.world > 1 and desc.fold_key == 1 and desc.embed_dim == self.embed_dim and desc.num_heads == self.num_heads
                and desc.dtype == ops.dtype_code(self.dtype))

    def pointer(self):
        return self._ptr


class PeerAllReduce:
    """In-place all-reduce of one CUDA tensor across the ranks of ONE node over NVLink peer memory, without NCCL:
    ``csrc/peer_allreduce.cu`` (barrier, every rank reduces its slice from all buckets in rank order and stores it
    into all buckets, barrier; bit-identical results on every rank, graph-capturable).

    Construction is collective (``_map_peer_tensors``).  The bucket must stay alive, and must not be reallocated, for the
    lifetime of this object.  ``GradientSync(collective="peer")`` uses it for the gradient bucket where the backward's
    own fused sum does not apply.
    """

    def __init__(self, bucket: torch.Tensor, group=None, average: bool = True):
        from . import ops
        if not bucket.is_cuda or not bucket.is_contiguous():
            raise ValueError("PeerAllReduce needs a contiguous CUDA tensor")
        self.bucket, self.group, self.average = bucket, group, average
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        if self.world > 8:
            raise ValueError("PeerAllReduce covers the (at most 8) GPUs of one NVLink node")
        self.flags = ops.peer_flag_block(bucket.device)
        self.buckets, self.flag_blocks = [bucket.data_ptr()], [self.flags.data_ptr()]     # device addresses, rank order
        if self.world > 1:
            self.buckets, self.flag_blocks = _map_peer_tensors([bucket, self.flags], group)
        self._ops = ops

    def __call__(self) -> None:
        """Enqueue the all-reduce on the current stream of the bucket's device."""
        if self.world == 1:
            return
        with torch.cuda.device(self.bucket.device):
            self._ops.peer_allreduce(self.buckets, self.flag_blocks, self.rank, average=self.average, mine=self.bucket)


class _BucketViews:
    """What the backward asks for a place to write a parameter gradient (``pool._grad_buffers``): the parameter's slice
    of the all-reduce bucket -- unless ``param.grad`` already LIVES there (a second micro-batch before the optimizer step,
    or ``zero_grad(set_to_none=False)``): writing the new gradient over the old one and letting autograd add the tensor
    to itself would double it, so the backward then gets no buffer, allocates its own, and autograd accumulates into the
    bucket slice in place."""

    def __init__(self, sync: "GradientSync"):
        self.sync = sync

    def get(self, name: str):
        view = self.sync.views.get(name)
        if view is None:
            return None
        grad = self.sync.params[name].grad
        if grad is None:
            self.sync.bucket_is_reduced = False          # a fresh step overwrites the slice
            return view
        if grad.data_ptr() == view.data_ptr():
            return None                                   # accumulate: see the class comment
        raise RuntimeError(
            f"GradientSync: {name}.grad is a tensor of its own; the synchronised gradients live in the sync's bucket. "
            "Clear gradients with set_to_none=True (or keep the .grad tensors finish() assigned) when GradientSync is attached.")

    def keys(self):
        return self.sync.views.keys()

    def __iter__(self):
        return iter(self.sync.views)

    def __getitem__(self, name):
        return self.sync.views[name]


class GradientSync:
    """Sum (mean by default) of the fusion parameter gradients of one pool + its query over the ranks.

    ``attach()`` hooks the pool.  With ``collective="fused"`` the pool's backward then sums across the ranks itself (see
    the module docstring) and ``finish()`` has nothing left to do; otherwise the backward writes gradients into
    ``self.bucket`` and ``finish()`` -- call it after ``loss.backward()`` either way -- reduces the bucket and points every
    ``param.grad`` at its slice.  Gradient accumulation over micro-batches: set ``enabled = False`` for all but the last
    micro-batch (like DDP's ``no_sync``) in bucket mode; in fused mode every backward is already summed over the ranks.
    """

    def __init__(self, pool, query: Optional[torch.nn.Parameter] = None, process_group=None,
                 average: bool = True, collective: Optional[str] = None):
        self.pool, self.query, self.group, self.average = pool, query, process_group, average
        att = pool.attention
        device, dtype = att.in_proj_weight.device, att.in_proj_weight.dtype
        self.cuda = device.type == "cuda"
        if collective is None:
            collective = os.environ.get("AECF_DP_COLLECTIVE") or ("fused" if self.cuda else "nccl")
        if collective not in ("fused", "nccl", "peer"):
            raise ValueError(f"collective must be 'fused', 'nccl' or 'peer', got {collective!r}")
        self.collective = collective
        self.overlap = False                             # read by bench.py: the bucket is always reduced in one piece
        self.params: Dict[str, torch.nn.Parameter] = {}
        for name, p in (("out_proj.bias", att.out_proj.bias), ("out_proj.weight", att.out_proj.weight),
                        ("in_proj_weight", att.in_proj_weight), ("in_proj_bias", att.in_proj_bias), ("query", query)):
            if p is not None:
                self.params[name] = p
        if any(p.dtype != dtype for p in self.params.values()):
            raise ValueError("GradientSync needs the fusion query and the pool parameters in one dtype")
        self.slices: Dict[str, slice] = {}
        n = 0
        for name in PARAM_ORDER:
            if name in self.params:
                k = self.params[name].numel()
                self.slices[name] = slice(n, n + k)
                n += (k + 7) // 8 * 8                       # keep every slice 16-byte aligned
        self.bucket = torch.zeros(n, dtype=dtype, device=device)
        self.views = {name: self.bucket[sl].view(self.params[name].shape) for name, sl in self.slices.items()}
        self.reported: set = set()
        self.bucket_is_reduced = False                   # the bucket holds a cross-rank result (a finished step)
        self.enabled = True                              # False: gradients stay local (gradient accumulation, measurements)
        self.peer = None
        self.fused = None
        multi = dist.is_initialized() and dist.get_world_size(process_group) > 1
        if self.cuda and multi and collective == "fused":
            try:
                self.fused = FusedGradSum(pool, process_group, average)
            except ValueError:
                self.fused = None                        # no fused tail for this pool: bucket + NCCL
        if self.cuda and multi and collective == "peer":
            self.peer = PeerAllReduce(self.bucket, process_group, average)     # one kernel for the whole bucket

    # -- wiring -----------------------------------------------------------------------------
    def attach(self) -> "GradientSync":
        self.pool._grad_ready = self.on_ready
        self.pool._grad_buffers = _BucketViews(self)     # the fused backward writes its gradients here
        self.pool._dp = self.fused
        if self.query is not None:
            self.query.register_hook(self._query_hook)
        return self

    def select(self, mode: str) -> None:
        """Switch what the next backward does with the gradients (measurements): 'fused' (the in-backward sum, where it was
        set up), 'bucket' (one all-reduce of the bucket in finish()), 'local' (no cross-rank sum at all)."""
        if mode not in ("fused", "bucket", "local"):
            raise ValueError(mode)
        if mode == "fused" and self.fused is None:
            raise ValueError("the fused gradient sum was not set up for this pool")
        self.pool._dp = self.fused if mode == "fused" else None
        self.enabled = mode != "local"

    def _fused_ran(self) -> bool:
        return self.fused is not None and self.fused.ran

    def _query_hook(self, grad: torch.Tensor) -> torch.Tensor:
        if self._fused_ran() or not self.enabled or self.world_size == 1:
            return grad                                  # already summed over the ranks inside the backward / nothing to do
        view = self.views["query"]
        accumulating = self.query.grad is not None and self.query.grad.data_ptr() == view.data_ptr()
        if grad.data_ptr() != view.data_ptr() and not accumulating:   # the shared-query bypass did not apply: copy in
            view.copy_(grad.reshape(view.shape))
        self.on_ready("query", grad if accumulating else view)
        return grad

    @property
    def world_size(self) -> int:
        return dist.get_world_size(self.group) if dist.is_initialized() else 1

    def set_shard(self, global_batch: int) -> Tuple[int, int]:
        """Point the pool's Philox row offset at this rank's shard; returns (row0, rows)."""
        rank = dist.get_rank(self.group) if dist.is_initialized() else 0
        row0, rows = shard_rows(global_batch, rank, self.world_size)
        self.pool.row_offset = row0
        return row0, rows

    # -- called from the backward (autograd worker thread) -----------------------------------
    def on_ready(self, name: str, grad: torch.Tensor) -> None:
        if name not in self.slices or self.world_size == 1:
            return                                                     # single process: autograd's .grad is final
        view = self.views[name]
        param_grad = self.params[name].grad
        accumulating = (param_grad is not None and param_grad.data_ptr() == view.data_ptr()
                        and grad.data_ptr() != view.data_ptr())
        if not self.enabled:
            if accumulating:
                self.bucket_is_reduced = False           # local gradients are being added to the slice: reduce it whole later
            return
        if name in self.reported:
            return
        if accumulating:
            # param.grad lives in the bucket and autograd adds `grad` to it AFTER this backward returns.
            if self.bucket_is_reduced:
                # ... onto numbers that are already a cross-rank result (or zeros): only the NEW gradient is reduced,
                # here and now, before autograd adds it (rare path: one small collective per parameter)
                self._reduce_now(grad)
                return
            # ... onto local, unreduced gradients (enabled=False micro-batches): the bucket is reduced whole in finish()
        elif grad.data_ptr() != view.data_ptr():                       # produced elsewhere: copy into the bucket
            view.copy_(grad.reshape(view.shape))
        self.reported.add(name)

    def _reduce_now(self, tensor: torch.Tensor) -> None:
        avg = self.average and dist.get_backend(self.group) == "nccl"
        dist.all_reduce(tensor, op=dist.ReduceOp.AVG if avg else dist.ReduceOp.SUM, group=self.group)
        if self.average and not avg:
            tensor.mul_(1.0 / self.world_size)

    # -- called by the training loop after loss.backward() -----------------------------------
    def finish(self) -> None:
        """Reduce the bucket (one all-reduce) and point every reported ``param.grad`` at its slice."""
        if self._fused_ran():
            self.fused.ran = False                       # the backward summed over the ranks itself: .grad is final
            self.reported.clear()
            return
        if not self.reported:
            return
        if self.peer is not None:
            self.peer()                                  # in place, on the compute stream, complete when it returns on-stream
        else:
            self._reduce_now(self.bucket)
        for name in self.reported:
            self.params[name].grad = self.views[name]
        self.bucket_is_reduced = True
        self.reported.clear()
