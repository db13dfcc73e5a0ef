#!/usr/bin/env python
"""Benchmark of the AECF fusion hot path (BASELINE.json metric):

    fused-pool fwd+bwd samples/sec at B=64K, M=3, D=512, H=8; HBM GB/s as % of peak

    python bench.py [--gpus N --steps K --warmup W]          this repo's sm_100a path
    python bench.py --impl reference [...]                    the reference's CPU path (oracle port)
    python bench.py [...] --dump-outputs DIR                  also write the last timed step's outputs as DIR/*.npy

One step = MultimodalAttentionPool forward(return_info=True) + CurriculumMasking.entropy_loss +
backward from an upstream gradient d_out (SURVEY.md section 8d), through the public module API.
`value`  : whole-job samples/s with the batch already resident in HBM.
`e2e`    : the same, with the batch starting in pinned host memory every step (H2D inside the timed
           region, double-buffered on a copy stream) and the entropy-loss scalar read back each step.
`roofline`: the fused pool backward kernel (the largest HBM-bound kernel), algorithmic bytes per launch
           divided by its CUDA-event duration inside the timed steps, against MEASURED_PEAKS.json.
`kernels`: per-launch-site CUDA-event averages from the same timed steps (pool forward roofline and
           tensor-pipe utilisation of the projection GEMMs are derived from these).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "fused-pool fwd+bwd samples/sec at B=64K,M=3,D=512,H=8; HBM GB/s as % of peak"
UNIT = "samples/s"
FALLBACK_HBM_GBS = 6650.0          # /opt/skills/guides/B200_PROFILING.md
FALLBACK_BF16_TFLOPS = 1590.0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--batch", type=int, default=65536, help="rows per GPU (weak scaling)")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="strong scaling: this many rows in total, sharded over the ranks (overrides --batch); the timed "
                         "steps rotate over enough input buffers to exceed the L2 when one shard fits in it")
    ap.add_argument("--tokens", type=int, default=3)
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--heads", type=int, default=8)
    ap.add_argument("--dtype", choices=["bf16", "fp32"], default="bf16")
    ap.add_argument("--dropout", type=float, default=0.0)
    ap.add_argument("--cpu-sample", type=int, default=0, help="rows of the CPU-baseline sample (0: the full batch, halved only if 4 steps would take > 40 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dp-study", action="store_true",
                    help="N > 1: also time the step with the other all-reduce mode and with no all-reduce at all "
                         "(separates collective cost from rank-to-rank variance); per-rank times are reported either way")
    ap.add_argument("--graph", choices=["on", "off"], default="on",
                    help="replay the step as one CUDA graph (aecf_b200.graphs) instead of enqueueing ~25 kernels from Python")
    ap.add_argument("--fold", choices=["auto", "on", "off"], default="auto",
                    help="folded key projection (auto: the module's choice, on for bf16)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one returned (pool output, info tensors, entropy loss, "
                         "gradients of x, the fusion query and the parameters) as DIR/<name>.npy in float32, at most 64 MB "
                         "in all; rank 0 only.  The inputs depend only on the arguments, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the sm_100a path: it needs --impl b200")
    return args


def ncu_traffic(kernel: str, args):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture of this exact workload
    (profiles/ncu_traffic.json), or None when the workload differs from the captured one."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)
        key = f"B={args.batch},M={args.tokens},D={args.dim},H={args.heads},{args.dtype},dropout={args.dropout}"
        if getattr(args, "folded", False):
            key += ",fold"
        return t.get(key, {}).get(kernel)
    except Exception:
        return None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"hbm_gbs": FALLBACK_HBM_GBS, "bf16_tflops": FALLBACK_BF16_TFLOPS, "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every ~2 ms DURING the timed region
    (nvidia-smi takes longer per query than a whole timed region lasts)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        self.index, self.samples, self.stop_flag, self.thread = index, [], threading.Event(), None
        self.max_mhz, self.handle, self.nvml = None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _run(self):
        nv = self.nvml
        while not self.stop_flag.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                self.samples.append((float(mhz), int(reasons)))
            except Exception:
                pass
            self.stop_flag.wait(0.002)

    def __enter__(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        return self

    def __exit__(self, *exc):
        self.stop_flag.set()
        if self.thread is not None:
            self.thread.join(timeout=10)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        sm = sorted(s[0] for s in self.samples)
        bits = 0
        for _, r in self.samples:
            bits |= r
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.max_mhz,
                "reasons": [name for bit, name in self.REASONS.items() if bits & bit], "samples": len(self.samples),
                "source": "NVML, sampled every 2 ms inside the timed region"}


# ------------------------------------------------------------------------------------------------
# The reference arm and the CPU baseline: the UNMODIFIED reference from baseline/_ref (installed there with
# `pip install --no-index --no-deps --target baseline/_ref`, DESIGN.md section 5), stock autograd, all host threads;
# the oracle port only where baseline/_ref is absent (kind says which).
# ------------------------------------------------------------------------------------------------
def load_reference():
    """The reference package as installed under baseline/_ref, imported under a private name (the repo's own drop-in
    alias package is also called `aecf`).  None when it is not there."""
    init = os.path.join(ROOT, "baseline", "_ref", "aecf", "__init__.py")
    if not os.path.exists(init):
        return None
    if "aecf_reference_unmodified" in sys.modules:
        return sys.modules["aecf_reference_unmodified"]
    import importlib.util
    spec = importlib.util.spec_from_file_location("aecf_reference_unmodified", init,
                                                  submodule_search_locations=[os.path.dirname(init)])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["aecf_reference_unmodified"] = mod
    spec.loader.exec_module(mod)
    return mod


def reference_step_fn(ref, args, rows, device, dtype):
    """BASELINE.md section 5: create_fusion_pool(D, M, 0.15, num_heads=H) default init, x = randn(rows, M, D), one step =
    forward(return_info=True) + entropy_loss + autograd backward of out.pow(2).mean() + 0.01 * entropy_loss."""
    import torch
    torch.manual_seed(0)
    M, D, H = args.tokens, args.dim, args.heads
    query, pool = ref.create_fusion_pool(D, M, 0.15, num_heads=H, dropout=args.dropout)
    pool = pool.to(device=device, dtype=dtype)
    query = torch.nn.Parameter(query.detach().to(device=device, dtype=dtype))
    x = torch.randn(rows, M, D).to(device=device, dtype=dtype).requires_grad_(True)
    params = [query, x] + list(pool.parameters())

    def step():
        out, info = pool(query.expand(rows, -1, -1), x, return_info=True)
        loss = out.float().pow(2).mean() + 0.01 * pool.curriculum_masking.entropy_loss(info["entropy"])
        loss.backward()
        for t in params:
            t.grad = None
        return loss
    return step


def port_step_fn(args, rows):
    """Fallback when baseline/_ref is absent: the oracle port (closed-form backward, no autograd)."""
    import torch
    from oracle import aecf_oracle as oracle
    from oracle import philox

    torch.manual_seed(0)
    M, D, H = args.tokens, args.dim, args.heads
    mha = torch.nn.MultiheadAttention(D, H, batch_first=True)          # default init of the reference's module
    params = {"in_proj_weight": mha.in_proj_weight.detach(), "in_proj_bias": mha.in_proj_bias.detach(),
              "out_proj.weight": mha.out_proj.weight.detach(), "out_proj.bias": mha.out_proj.bias.detach()}
    q0 = torch.randn(1, 1, D) * (2.0 / D) ** 0.5
    x = torch.randn(rows, M, D)
    u_mask = torch.from_numpy(philox.mask_uniforms(0x5EED, 0, 0, rows, M))
    d_out = torch.randn(rows, 1, D)
    masking = dict(base_mask_prob=0.15, entropy_target=0.7, min_active=1)

    def step():
        with torch.no_grad():
            q = q0.expand(rows, 1, D)
            fwd = oracle.pool_forward(q, x, None, params["in_proj_weight"], params["in_proj_bias"],
                                      params["out_proj.weight"], params["out_proj.bias"], H, training=True,
                                      u_mask=u_mask, masking=masking)
            loss = oracle.entropy_loss(fwd.info["entropy"], M)
            grads = oracle.pool_backward(q, x, None, params["in_proj_weight"], params["out_proj.weight"], H,
                                         fwd.saved, d_out)
            return loss, grads
    return step


def time_cpu(args, rows, steps, warmup, budget_s=240.0):
    """(samples/s, ms per step, threads, kind, rows timed).  The full batch unless (warmup + steps) steps of it would not
    finish inside `budget_s` on this host, in which case the rows are halved until they do (and the line says so)."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = load_reference()
    kind = "reference" if ref is not None else "port"
    make = (lambda r: reference_step_fn(ref, args, r, "cpu", torch.float32)) if ref is not None else (lambda r: port_step_fn(args, r))
    step = make(rows)
    t0 = time.perf_counter()
    step()                                              # first warm-up step doubles as the probe
    probe = time.perf_counter() - t0
    while probe * (warmup + steps) > budget_s and rows > 1024:
        rows //= 2
        step = make(rows)
        t0 = time.perf_counter()
        step()
        probe = time.perf_counter() - t0
    for _ in range(max(0, warmup - 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return rows / dt, dt * 1e3, cores, kind, rows


def time_reference_gpu_eager(args, dev, steps=10, warmup=3):
    """BASELINE.md section 5.6: the unmodified reference on THIS B200 (stock PyTorch eager: cuBLAS + ~35 ATen ops and >= 5
    host syncs per forward), same rows and dtype as the measured arm, CUDA events.  None without baseline/_ref."""
    import torch
    ref = load_reference()
    if ref is None:
        return None
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    try:
        step = reference_step_fn(ref, args, args.batch, dev, dtype)
        for _ in range(warmup):
            step()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            step()
        b.record()
        torch.cuda.synchronize(dev)
        ms = a.elapsed_time(b) / steps
        del step
        torch.cuda.empty_cache()
        return {"value": args.batch / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "warmup": warmup,
                "dtype": args.dtype, "rows": args.batch,
                "kind": "reference (baseline/_ref, unmodified) in stock PyTorch eager on this GPU, autograd backward"}
    except Exception as e:                              # a baseline for context must never take the measurement down
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def cublas_yardstick(args, dev, folded):
    """torch.matmul (cuBLAS) on the six projection shapes of this workload, CUDA events, us per call, operand sets rotated
    so that no call finds its operands in L2 -- a yardstick for `gemm_tensor_pipe`, not a path of this library: at K = 512
    with 400 MB of traffic per product nobody reaches the 8192^3 rate the `peak` of that object quotes (profiles/
    r2_gemm_where_the_time_goes.md)."""
    import torch
    if args.dtype != "bf16":
        return None
    try:
        B, M, D = args.batch, args.tokens, args.dim
        rows, kf = B * M, (D + 8 if folded else 2 * D)
        bf = torch.bfloat16
        rnd = lambda *shape: (torch.randn(*shape, device=dev) * 0.1).to(bf)

        def timed(make, sets):
            ops_ = [make() for _ in range(sets)]
            for i in range(3):
                ops_[i % sets]()
            torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(10):
                ops_[i % sets]()
            b.record()
            torch.cuda.synchronize(dev)
            return a.elapsed_time(b) * 100.0          # ms / 10 calls -> us per call

        def prod(a_shape, b_shape, ta=False, tb=False):
            def make():
                a, b = rnd(*a_shape), rnd(*b_shape)
                return lambda: torch.matmul(a.t() if ta else a, b.t() if tb else b)
            return make
        out = {"kv_proj": timed(prod((rows, D), (kf if folded else 2 * D, D), tb=True), 2),
               "out_proj": timed(prod((B, D), (D, D), tb=True), 4), "d_ctx": timed(prod((B, D), (D, D)), 4),
               "d_out_weight": timed(prod((B, D), (B, D), ta=True), 4),
               "d_x": timed(prod((rows, kf), (kf, D)), 2), "d_kv_weight": timed(prod((rows, kf), (rows, D), ta=True), 2)}
        torch.cuda.empty_cache()
        out["note"] = ("torch.matmul, bf16, same shapes" + (" (kv_proj with the 8 score rows as ordinary output columns)" if folded else "")
                       + "; not a path of this library")
        return out
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"[:200]}


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


L2_BYTES = 126 * 1024 * 1024


def input_buffers_needed(x_bytes: int) -> int:
    """How many distinct input batches the timed steps must rotate over so that a step never finds its input in
    the 126 MB L2: 1 when one batch is larger than the L2 (the default workload), else enough to exceed twice the L2."""
    return 1 if x_bytes > L2_BYTES else min(32, -(-2 * L2_BYTES // max(x_bytes, 1)))


def workload_config(args, n_gpus):
    es = 2 if args.dtype == "bf16" else 4
    x_mb = args.batch * args.tokens * args.dim * es / 1e6
    strong = getattr(args, "global_batch", 0) > 0
    rot = input_buffers_needed(int(x_mb * 1e6))
    if rot == 1:
        l2 = f"inputs larger than L2 (x {x_mb:.0f} MB, values {x_mb:.0f} MB per step vs 126 MB L2); no flush needed"
    elif rot * x_mb * 1e6 > L2_BYTES:
        l2 = (f"one shard's input ({x_mb:.0f} MB) fits in the 126 MB L2: the timed steps rotate over {rot} input batches "
              f"({rot * x_mb:.0f} MB), so no step finds its input in L2")
    else:
        l2 = (f"L2-RESIDENT: {rot} input batches of {x_mb:.2f} MB are smaller than the 126 MB L2 together; "
              "not a bandwidth measurement")
    return {"workload": f"MultimodalAttentionPool D={args.dim} H={args.heads} M={args.tokens} with CurriculumMasking, "
                        + (f"B={args.global_batch} in total over {n_gpus} GPUs" if strong else f"B={args.batch} per GPU")
                        + " (BASELINE.json configs[1]; arithmetic type in `dtype`)",
            "global_batch": args.global_batch if strong else args.batch * n_gpus,
            "tokens": args.tokens, "embed_dim": args.dim, "heads": args.heads,
            "dropout": args.dropout, "parallelism": f"dp{n_gpus}",
            "l2": l2,
            "step": "forward(return_info) + entropy_loss + backward, public module API"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores -- the unmodified
    package from baseline/_ref through its public API with autograd (the oracle port only if that install is absent),
    all host threads, the arm's own workload (B rows, fp32 as BASELINE.md section 5 prescribes), --steps / --warmup honoured."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    value, ms, cores, kind, rows = time_cpu(args, args.batch, max(1, args.steps), max(1, args.warmup))
    cfg = workload_config(args, args.gpus)
    sample = (f"{rows} rows per step" + ("" if rows == args.batch else f" (halved from {args.batch} to fit the time budget)")
              + f", fp32, {'unmodified reference from baseline/_ref, autograd' if kind == 'reference' else 'oracle port, closed-form backward'}"
              + f", {cores} threads ({cpu_model()})")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": max(1, args.steps), "warmup": max(1, args.warmup), "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "same_config": rows == args.batch,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# the sm_100a path
# ------------------------------------------------------------------------------------------------
def kernel_averages(sites, steps):
    """aecf_timing_collect() totals -> {launch site: {ms per launch, launches per step}}."""
    return {name: {"ms": total / count, "calls_per_step": count / steps} for name, (total, count) in sites.items()}


DUMP_BYTES = 64 << 20


def sample_outputs(outputs, budget=DUMP_BYTES):
    """{name: float32 device copy} of the tensors one step returned.  An array larger than its equal share of `budget`
    keeps a fixed sample of its leading-dimension rows (the first rows of numpy's default_rng(0) permutation, in
    order), so two builds run with the same arguments dump the same elements."""
    import numpy as np
    import torch
    tensors = {k: v.detach() for k, v in outputs.items() if isinstance(v, torch.Tensor)}
    share = budget // max(1, len(tensors))
    kept = {}
    for name, t in tensors.items():
        if t.dim() and t.numel() * 4 > share:
            rows = max(1, share // (4 * max(1, t[0].numel())))
            idx = np.sort(np.random.default_rng(0).permutation(t.shape[0])[:rows])
            t = t.index_select(0, torch.from_numpy(idx).to(t.device))
        kept[name] = t.float().clone()
    return kept


def write_outputs(directory, kept):
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in kept.items():
        np.save(os.path.join(directory, name + ".npy"), t.cpu().numpy())


def finish_process(world, nccl_in_graphs=True):
    """With the step captured into CUDA graphs that hold NCCL kernels, destroy_process_group() blocked for minutes on the
    8-GPU box (r1 run 16: the communicator waits for work it believes outstanding); in that case every rank has passed
    the last barrier and rank 0 has printed its line, so leave directly.  With the gradient sum inside the backward
    (the default) no NCCL kernel is ever captured and the group is torn down normally."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        if nccl_in_graphs:
            os._exit(0)
        import torch.distributed as dist
        dist.destroy_process_group()


def run_b200(args):
    import torch
    import torch.distributed as dist

    import aecf_b200
    from aecf_b200 import _lib
    from aecf_b200.dp import GradientSync

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: aecf_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"            # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
        # a multi-rank run that wedges (a lost peer, a collective that never completes) must not sit on N GPUs
        # until somebody's outer timeout: hard stop after 10 minutes
        guard = threading.Timer(600.0, lambda: os._exit(3))
        guard.daemon = True
        guard.start()
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    es = 2 if dtype == torch.bfloat16 else 4
    strong = args.global_batch > 0
    if strong:                                         # strong scaling: a fixed global batch, sharded over the ranks
        from aecf_b200.dp import shard_rows
        args.batch = shard_rows(args.global_batch, rank, world)[1]
        if args.batch == 0:
            raise SystemExit(f"--global-batch {args.global_batch} leaves rank {rank} of {world} without rows")
    B, M, D, H = args.batch, args.tokens, args.dim, args.heads
    total_rows = args.global_batch if strong else B * world

    torch.manual_seed(0)
    query, pool = aecf_b200.create_fusion_pool(D, M, 0.15, num_heads=H, dropout=args.dropout, device=dev, dtype=dtype)
    cm = pool.curriculum_masking
    pool.fold_key_projection = {"auto": None, "on": True, "off": False}[args.fold]
    args.folded = (dtype == torch.bfloat16 and os.environ.get("AECF_FOLD", "1") != "0") if args.fold == "auto" else args.fold == "on"
    sync = GradientSync(pool, query).attach()
    sync.set_shard(total_rows)                                    # Philox keyed on the global row
    torch.manual_seed(1234 + rank)
    # one input batch when it is larger than the L2 (the default workload); otherwise the timed steps rotate over
    # enough batches that none is found in L2 (input_buffers_needed)
    rot = input_buffers_needed(B * M * D * es)
    xs = [torch.randn(B, M, D, device=dev, dtype=dtype).requires_grad_(True) for _ in range(rot)]
    x = xs[0]
    d_out = torch.randn(B, 1, D, device=dev, dtype=dtype)

    def step(xin, outputs=False):
        """One step; returns the loss, or with `outputs` every tensor its caller receives (static tensors when the step
        is a graph replay) for --dump-outputs."""
        out, info = pool(query.expand(B, -1, -1), xin, return_info=True)
        loss = cm.entropy_loss(info["entropy"])
        out.backward(d_out)
        sync.finish()
        if not outputs:
            return loss
        grads = {"grad_x": xin.grad, "grad_query": query.grad}
        grads.update({"grad_" + name: p.grad for name, p in pool.named_parameters()})
        # detached: a kept result must not hold the autograd graph of its step alive
        return {k: v.detach() for k, v in {"out": out, **info, "entropy_loss": loss, **grads}.items() if v is not None}

    def clear():
        for xi in xs:
            xi.grad = None
        query.grad = None
        pool.zero_grad(set_to_none=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing -----------------------------------------------------------
    # Region A (the reported value): K steps, no per-kernel events -- kernels chain by programmatic dependent
    # launch; with --graph on (default) the step was captured once (warm-up steps run eagerly first) and each
    # timed step is one graph replay.  Region B: K more EAGER steps with a CUDA event pair around every launch
    # of the library (on the launching stream) for the per-kernel durations behind `roofline`, `kernels` and
    # `gemm_tensor_pipe`.
    use_graph = args.graph == "on"
    for _ in range(args.warmup):
        step(x); clear()
    barrier()
    launches0 = _lib.launch_count()
    turn = [0]
    dump = bool(args.dump_outputs) and rank == 0
    last = [None]                                                        # what the last timed step returned (dump only)
    if use_graph:
        graphs = []                                                      # one graph per input batch
        for xi in xs:
            graphs.append(aecf_b200.graphs.GraphedStep(lambda xi=xi: step(xi, dump), reset=clear, warmup=0, device=dev))
            if len(graphs) == 1:
                launches_per_step = _lib.launch_count() - launches0      # counted while capturing one step
        for i in range(max(args.warmup, rot)):
            graphs[i % rot]()

        def run_step():
            graphs[turn[0] % rot]()
            turn[0] += 1
    else:
        def run_step():
            final = dump and turn[0] == args.steps - 1                  # only the last step's outputs are kept
            result = step(xs[turn[0] % rot], final); clear()
            if final:
                last[0] = result
            turn[0] += 1
    barrier()
    launches0 = _lib.launch_count()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        if world > 1:
            # device-side rendezvous right before the clock starts: the host barrier above lets the ranks go tens of
            # microseconds apart, which a 12 ms timed region would count as step time (VERDICT r1, scaling item iii)
            dist.all_reduce(torch.zeros(1, device=dev))
        start.record()
        t_issue = time.perf_counter()
        for _ in range(args.steps):
            run_step()
        end.record()
        issue_ms = (time.perf_counter() - t_issue) * 1e3 / args.steps   # host time to enqueue one step
        barrier()
        ms = start.elapsed_time(end) / args.steps
        launches = launches_per_step * args.steps if use_graph else (_lib.launch_count() - launches0)
        # copied on the device now: the parameter gradients live in the GradientSync bucket, which region B rewrites
        if dump and use_graph:
            last[0] = graphs[(args.steps - 1) % rot].result                # the static outputs of the last replay
        dumped = sample_outputs(last[0]) if dump else None
        clear()
        # region B measures each kernel ON ITS OWN: the gradient tail, which the timed step runs on a side stream next to the
        # [dWv;R] and dX products, is serialised onto the compute stream here (next to a product its kernels take several
        # times longer and the product a little longer -- durations that describe the overlap, not the kernels)
        side_was = os.environ.get("AECF_SIDE_STREAM")
        os.environ["AECF_SIDE_STREAM"] = "0"
        _lib.timing_enable(True)
        start_b, end_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start_b.record()
        for i in range(args.steps):
            step(xs[i % rot]); clear()
        end_b.record()
        barrier()
        if side_was is None:
            os.environ.pop("AECF_SIDE_STREAM", None)
        else:
            os.environ["AECF_SIDE_STREAM"] = side_was
    ms_with_events = start_b.elapsed_time(end_b) / args.steps
    kernels = kernel_averages(_lib.timing_collect(), args.steps)
    _lib.timing_enable(False)

    def time_region(run):
        """W warm-up + K timed calls of `run`, CUDA events, this rank's ms per step."""
        for _ in range(args.warmup):
            run()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.steps):
            run()
        b.record()
        barrier()
        return a.elapsed_time(b) / args.steps

    def gather_ms(local_ms):
        t = torch.zeros(world, device=dev, dtype=torch.float64)
        t[rank] = local_ms
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    dp_info = None
    if world > 1:
        per_rank = gather_ms(ms)
        ms = max(per_rank)
        dp_info = {"gradient_sum": ("inside the backward: fp32 raw sums over NVLink peer memory, one kernel per rank on the side stream "
                                    "(csrc/grad_tail.cu, peer_allreduce.cu)") if sync.fused is not None else
                                   ("bucket, overlapped NCCL all-reduce in two groups" if sync.overlap else "bucket, one NCCL all-reduce after the backward"),
                   "collective": sync.collective, "per_rank_ms": per_rank, "rank_spread": (max(per_rank) - min(per_rank)) / max(per_rank),
                   "in_graph": use_graph}
        if args.dp_study:
            def variant(mode):
                sync.select(mode); clear()
                if use_graph:
                    g = aecf_b200.graphs.GraphedStep(lambda: step(x), reset=clear, warmup=1, device=dev)
                    t_ms = time_region(g)
                    del g
                else:
                    t_ms = time_region(lambda: (step(x), clear()))
                clear()
                return gather_ms(t_ms)

            for mode in ("bucket", "local"):               # one NCCL all-reduce after the backward / no cross-rank sum at all
                t = variant(mode)
                dp_info[mode] = {"per_rank_ms": t, "ms_per_step": max(t), "value": total_rows / (max(t) * 1e-3)}
            sync.select("fused" if sync.fused is not None else "bucket")
    value = total_rows / (ms * 1e-3)

    # ---- end to end: batch starts in pinned host memory every step -----------------------------
    e2e = None
    if not args.no_e2e:
        host = torch.randn(B, M, D, dtype=dtype).pin_memory()
        host_loss = torch.zeros(1, dtype=torch.float32).pin_memory()
        bufs = [torch.empty(B, M, D, device=dev, dtype=dtype).requires_grad_(True) for _ in range(2)]
        copy_stream = torch.cuda.Stream(device=dev)
        copied = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]

        def upload(i):
            slot = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[slot])
                bufs[slot].detach().copy_(host, non_blocking=True)
                copied[slot].record(copy_stream)

        def clear_all():
            for b in bufs:
                b.grad = None
            query.grad = None
            pool.zero_grad(set_to_none=True)

        if use_graph:                                   # one graph per input slot (each replays on its own buffer)
            clear_all()
            slot_steps = [aecf_b200.graphs.GraphedStep(lambda b=b: step(b), reset=clear_all, warmup=1, device=dev)
                          for b in bufs]
        else:
            def eager_slot(b):
                def run():
                    loss = step(b)
                    return loss
                return run
            slot_steps = [eager_slot(b) for b in bufs]

        def e2e_loop(n):
            for c in consumed:
                c.record()
            upload(0)
            for i in range(n):
                slot = i % 2
                if i + 1 < n:
                    upload(i + 1)
                torch.cuda.current_stream().wait_event(copied[slot])
                loss = slot_steps[slot]()
                host_loss.copy_(loss.reshape(1), non_blocking=True)
                consumed[slot].record()
                if not use_graph:
                    clear_all()
            torch.cuda.synchronize()

        e2e_loop(max(2, args.warmup))
        barrier()
        t0 = time.perf_counter()
        e2e_loop(args.steps)
        barrier()
        e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
        if world > 1:
            t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_ms = float(t.item())
        e2e = {"value": total_rows / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": total_rows * M * D * es, "d2h_bytes_per_step": 4 * world,
               "note": "host batch -> double-buffered H2D on a copy stream -> step -> loss scalar D2H"}

    nccl_captured = use_graph and world > 1 and (sync.fused is None or args.dp_study)
    if rank != 0:
        barrier()                                        # rank 0 is past its last collective too
        finish_process(world, nccl_captured)
        return

    # ---- roofline of the fused pool kernels and tensor-pipe use of the GEMMs ----------------------
    peaks = measured_peaks()
    # algorithmic bytes per launch of the kernels AS LAUNCHED.  Unfolded (SURVEY.md section 8d): fwd reads K and V,
    # bwd re-reads them and writes dK and dV.  Folded key projection: K does not exist -- fwd reads V and the fp32
    # scores, bwd reads V, scores, d_ctx and writes [dV | ds] (DESIGN.md section 4.1).
    hs, hsp = (H + 3) // 4 * 4, (H + (16 // es) - 1) // (16 // es) * (16 // es)
    if args.folded:
        fwd_bytes = B * (es * (M * D + D) + 4 * M * hs + 4 * (2 * M + 2))
        bwd_bytes = B * (es * (M * D + D + M * (D + hsp)) + 4 * M * hs)
    else:
        fwd_bytes = B * (es * (2 * M * D + D) + 4 * (2 * M + 2))
        bwd_bytes = B * (es * (2 * M * D + D + 2 * M * D))

    survey_bytes = {"pool_fwd": B * (es * (2 * M * D + D) + 4 * (2 * M + 2)), "pool_bwd": B * (es * (2 * M * D + D + 2 * M * D))}

    def hbm(name, nbytes):
        if name not in kernels:
            return None
        gbs = nbytes / (kernels[name]["ms"] * 1e-3) / 1e9
        r = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
             "frac": gbs / peaks["hbm_gbs"], "frac_of_nominal_8TBs": gbs / 8000.0, "traffic": ncu_traffic(name, args),
             "ms": kernels[name]["ms"], "algorithmic_bytes": nbytes, "peak_source": peaks["source"]}
        if args.folded:
            # SURVEY.md section 8d counts the bytes of the reference's data flow (K and V read, dK and dV written).
            # The folded kernels do not move K or dK at all, so `achieved` above uses THEIR bytes; this is the
            # bandwidth an unfolded kernel would need to finish the same rows in the same time.
            r["survey_8d_bytes"] = survey_bytes[name]
            r["equivalent_gbs_at_survey_8d_bytes"] = survey_bytes[name] / (kernels[name]["ms"] * 1e-3) / 1e9
        return r

    kvw = (D + hsp) if args.folded else 2 * D       # projected columns per token: [V | scores] or [K | V]
    gemm_flops = {"kv_proj": 2 * B * M * D * kvw, "out_proj": 2 * B * D * D, "d_ctx": 2 * B * D * D,
                  "d_out_weight": 2 * B * D * D, "d_x": 2 * B * M * kvw * D, "d_kv_weight": 2 * B * M * kvw * D}
    gemms = {}
    for name, fl in gemm_flops.items():
        if name in kernels:
            tf = fl / (kernels[name]["ms"] * 1e-3) / 1e12
            gemms[name] = {"ms": kernels[name]["ms"], "tflops": tf, "frac_of_peak": tf / peaks["bf16_tflops"]}
    roof = hbm("pool_bwd", bwd_bytes)
    pool_ms = sum(kernels[k]["ms"] for k in ("pool_fwd", "pool_bwd") if k in kernels)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "bf16" if dtype == torch.bfloat16 else "f32", "data": "synthetic",
            "config": workload_config(args, world), "impl": "b200",
            "implementation": {"fold_key_projection": bool(args.folded),
                               "cuda_graph": "step captured once with aecf_b200.graphs.GraphedStep and replayed" if use_graph else "eager",
                               "gradient_tail": ("on a side stream next to the [dWv;R] and dX products" if os.environ.get("AECF_SIDE_STREAM", "1") != "0"
                                                 else "on the compute stream"),
                               "entropy_loss": "fused into the pool forward kernel" if os.environ.get("AECF_FUSED_LOSS", "1") != "0" else "stand-alone kernel",
                               "pool_backward": ("no batch sums in the kernel (the tail forms the in-projection bias gradient from colsum(d_out)); "
                                                 + ("persistent grid" if os.environ.get("AECF_POOL_BWD_CHUNK") == "0" else
                                                    f"{os.environ.get('AECF_POOL_BWD_CHUNK', '16')} consecutive samples per CTA, handed out by the block scheduler"))
                                                if args.folded and args.dropout == 0.0 else "see DESIGN.md section 4.1",
                               "kernels_note": "`kernels`, `roofline*` and `gemm_tensor_pipe` are per-kernel durations with the gradient tail "
                                               "serialised (each kernel on its own); `ms_per_step` / `value` is the overlapped, graph-replayed step"},
            "roofline": roof, "roofline_pool_fwd": hbm("pool_fwd", fwd_bytes),
            "pool_kernels_only": {"value": B / (pool_ms * 1e-3) if pool_ms else None, "unit": UNIT, "ms": pool_ms,
                                  "bytes_per_sample": (fwd_bytes + bwd_bytes) // B,
                                  "note": "fused pool fwd+bwd kernels alone, per GPU (the 273 M samples/s target)"},
            "gemm_tensor_pipe": gemms, "kernels": kernels, "host_issue_ms_per_step": issue_ms,
            "ms_per_step_with_kernel_events": ms_with_events,
            "kernel_ms_sum": sum(k["ms"] * k["calls_per_step"] for k in kernels.values()),
            "e2e": e2e, "gpu_launches": launches, "cuda_graph": use_graph, "clocks": clocks.summary(),
            "library": _lib.build_info(),
            # opt-in kernel variants in effect and the GEMM kernel each launch site used: A/B runs are self-describing
            "switches": {k: v for k, v in sorted(os.environ.items()) if k.startswith("AECF_")},
            "gemm_kernels": _lib.site_gemm_kernels()}
    if dp_info is not None:
        line["data_parallel"] = dp_info

    if world == 1 and not args.no_cpu_baseline:
        line["gemm_yardstick_cublas_us"] = cublas_yardstick(args, dev, bool(args.folded))
        line["reference_gpu_eager"] = time_reference_gpu_eager(args, dev)
        cpu_value, cpu_ms, cores, kind, rows = time_cpu(args, args.cpu_sample or B, 3, 1, budget_s=40.0)
        line["cpu_baseline"] = {"value": cpu_value, "unit": UNIT, "cores": cores, "kind": kind,
                                "sample": f"{rows} rows of the same workload per step, 1 warm-up + 3 timed steps, fp32, "
                                          + ("unmodified reference (baseline/_ref), autograd" if kind == "reference"
                                             else "oracle port, closed-form backward")
                                          + f" ({cpu_model()})", "ms_per_step": cpu_ms}
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    print(json.dumps(line))
    barrier()
    finish_process(world, nccl_captured)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
