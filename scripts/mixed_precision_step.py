#!/usr/bin/env python
"""Mixed precision against bf16 on the config-2 training step of the fusion pool.

    python scripts/mixed_precision_step.py [--steps 200] [--runs 2] [--out DIR] [--no-vlm]

B = 65 536, M = 3, D = 512, H = 8, the folded key projection (the bf16 default), CurriculumMasking, one CUDA-graph
replay per step.  The bf16 module (bf16 parameters) and the mixed module (fp32 parameters, bf16 tokens, fp32 parameter
gradients) are timed alternately, `--runs` runs each, in one process.  Prints the card name and power limit, ms per
step of every run, and the time of the parameter-shadow launch (``AECF_SITE_PARAM_CAST``, CUDA events around it over
eager steps).  Then runs ``examples/train_vlm.py --dtype bf16`` and ``--dtype mixed`` on one GPU and prints their
samples/s.  Everything is printed as one JSON line (and written to DIR/mixed_precision_step.json with --out).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import aecf_b200  # noqa: E402
from aecf_b200 import _lib, graphs  # noqa: E402

B, M, D, H = 65536, 3, 512, 8


def card() -> dict:
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()
        out["nvidia_smi"] = q[0] if q else ""
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = f"unavailable: {e}"
    return out


def make(param_dtype: torch.dtype, dev: torch.device):
    torch.manual_seed(0)
    q, pool = aecf_b200.create_fusion_pool(D, M, 0.15, num_heads=H, device=dev, dtype=param_dtype)
    gen = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(B, M, D, device=dev, generator=gen).bfloat16()
    g = torch.randn(B, 1, D, device=dev, generator=gen).bfloat16()
    params = list(pool.parameters()) + [q]

    def step():
        out, info = pool(q.expand(B, -1, -1), x, return_info=True)
        loss = (out.float() * g.float()).sum() + 0.01 * pool.curriculum_masking.entropy_loss(info["entropy"])
        loss.backward()
        return loss

    def reset():
        for p in params:
            p.grad = None

    return step, reset


def time_replays(graphed, steps: int) -> float:
    for _ in range(10):
        graphed()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        graphed()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def cast_time(step, reset, n: int = 20) -> dict:
    for _ in range(3):
        reset(); step()
    torch.cuda.synchronize()
    _lib.timing_enable(True)
    for _ in range(n):
        reset(); step()
    sites = _lib.timing_collect()
    _lib.timing_enable(False)
    ms, launches = sites.get("param_cast", (0.0, 0))
    return {"param_cast_us_per_step": 1e3 * ms / n, "param_cast_launches_per_step": launches / n}


def vlm(dtype: str) -> dict:
    cmd = [sys.executable, os.path.join(ROOT, "examples", "train_vlm.py"), "--dtype", dtype, "--steps", "30"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    if res.returncode != 0 or not lines:
        return {"error": res.stderr[-2000:]}
    r = json.loads(lines[-1])
    return {"samples_per_s": r["value"], "ms_per_step": r["ms_per_step"], "loss": r["loss"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200, help="graph replays per timed run")
    ap.add_argument("--runs", type=int, default=2, help="timed runs of each module, alternating")
    ap.add_argument("--out", default="", help="also write the JSON line to DIR/mixed_precision_step.json")
    ap.add_argument("--no-vlm", action="store_true", help="skip the examples/train_vlm.py runs")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mixed_precision_step.py measures on a CUDA device; there is none")
    dev = torch.device("cuda", 0)
    result = {"card": card(), "config": {"B": B, "M": M, "D": D, "H": H, "graph": True, "fold": "auto"}}
    steps = {"bf16": make(torch.bfloat16, dev), "mixed": make(torch.float32, dev)}
    result.update({f"{k}_cast": cast_time(*v) for k, v in steps.items()})
    graphed = {k: graphs.GraphedStep(v[0], reset=v[1]) for k, v in steps.items()}
    ms = {"bf16": [], "mixed": []}
    for _ in range(args.runs):
        for k in ("bf16", "mixed"):
            aecf_b200.set_rng_state(5, 0)
            ms[k].append(time_replays(graphed[k], args.steps))
    result["ms_per_step"] = ms
    best = {k: min(v) for k, v in ms.items()}
    result["mixed_over_bf16"] = best["mixed"] / best["bf16"]
    if not args.no_vlm:
        result["train_vlm_1gpu"] = {d: vlm(d) for d in ("bf16", "mixed")}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "mixed_precision_step.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
