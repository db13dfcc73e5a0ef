#!/usr/bin/env python
"""BASELINE.json configs[2]: the README VisionLanguageModel training step (2048/768 -> 512, M = 2,
1000-class head), batch-sharded over N GPUs of one box.

    python examples/train_vlm.py --steps 30
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 examples/train_vlm.py --steps 30
    python examples/train_vlm.py --dtype mixed     # fp32 master parameters, bf16 features and compute

The fusion parameters go through aecf_b200.dp.GradientSync (summed over the ranks inside the pool's backward); the two
encoder projections and the classifier are the model's nn.Linear PARAMETERS driven by the library's GEMMs
(aecf_b200.project_tokens / linear: the encoders write straight into the [B, 2, 512] token buffer, no torch.stack, no
cuBLAS), and their gradients are all-reduced in one flat NCCL call.  Prints one JSON line with samples/s (synthetic
features, random-init weights).  --launch-list prints the kernels of one step by name (torch profiler) to show that.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch
import torch.distributed as dist
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from aecf_b200.dp import GradientSync  # noqa: E402
from examples.models import VisionLanguageModel  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=16384, help="rows per GPU")
    ap.add_argument("--heads", type=int, default=1, help="the README model uses the default single head")
    ap.add_argument("--dtype", choices=["bf16", "fp32", "mixed"], default="bf16",
                    help="mixed: fp32 parameters and optimizer, bf16 features; every GEMM and the pool run in bf16")
    ap.add_argument("--launch-list", action="store_true", help="rank 0: kernel names of one step (torch profiler)")
    args = ap.parse_args()

    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=dev)
    dtype = torch.float32 if args.dtype == "fp32" else torch.bfloat16          # of the features
    param_dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32

    torch.manual_seed(0)                                       # same init on every rank
    model = VisionLanguageModel(num_heads=args.heads).to(dev, param_dtype)
    sync = GradientSync(model.fusion_pool, model.fusion_query).attach()
    sync.set_shard(args.batch * world)
    fusion_ids = {id(p) for p in sync.params.values()}
    others = [p for p in model.parameters() if id(p) not in fusion_ids]
    opt = torch.optim.SGD(model.parameters(), lr=1e-3)

    torch.manual_seed(100 + rank)
    img = torch.randn(args.batch, 2048, device=dev, dtype=dtype)
    txt = torch.randn(args.batch, 768, device=dev, dtype=dtype)
    labels = torch.randint(0, 1000, (args.batch,), device=dev)

    def step():
        logits, info = model(img, txt, return_info=True)
        loss = F.cross_entropy(logits.float(), labels) + 0.01 * model.fusion_pool.curriculum_masking.entropy_loss(info["entropy"])
        opt.zero_grad(set_to_none=True)
        loss.backward()
        if world > 1:
            flat = torch.cat([p.grad.reshape(-1) for p in others])
            dist.all_reduce(flat, op=dist.ReduceOp.AVG)
            off = 0
            for p in others:
                p.grad.copy_(flat[off:off + p.numel()].view_as(p))
                off += p.numel()
        sync.finish()
        opt.step()
        return loss

    for _ in range(args.warmup):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        loss = step()
    t1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([t0.elapsed_time(t1) / args.steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    kernels = None
    if args.launch_list and rank == 0 and world == 1:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.synchronize()
        names = {}
        for e in prof.events():
            if e.device_type is not None and "cuda" in str(e.device_type).lower():
                names[e.name] = names.get(e.name, 0) + 1
        kernels = {"kernels_of_one_step": names,
                   "cublas_or_cutlass_kernels": sorted(n for n in names if any(t in n.lower() for t in ("cublas", "cutlass", "gemm_", "sm90", "sm100", "xmma", "nvjet")) and "aecf" not in n and "tc::" not in n)}
    if rank == 0:
        if kernels is not None:
            print(json.dumps(kernels))
        print(json.dumps({"workload": "VisionLanguageModel training step (README.md:162-208 of the reference)",
                          "value": args.batch * world / (float(ms) * 1e-3), "unit": "samples/s", "n_gpus": world,
                          "ms_per_step": float(ms), "batch_per_gpu": args.batch, "dtype": args.dtype,
                          "heads": args.heads, "loss": float(loss), "data": "synthetic", "scaling": "weak"}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
