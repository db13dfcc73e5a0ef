"""The six projection products of config 2 as stand-alone aecf_gemm calls, CUDA-event timed, one JSON line.

    python scripts/gemm_bench.py [--cublas] [--tag NAME]

The library picks each product's kernel from its shape, as in a training step; the kernel that ran is reported per
product.  Every product rotates over enough operand sets that no call finds its operands in the 126 MB L2.  --cublas also
times torch.matmul on the same shapes (a yardstick, not a product path).
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from aecf_b200 import _lib, ops  # noqa: E402

DEV = torch.device("cuda", 0)
B, M, D, H = 65536, 3, 512, 8
HSP = 8
K, MN = _lib.K_MAJOR, _lib.MN_MAJOR


def time_us(fn, sets, iters=20, warmup=3):
    for i in range(warmup):
        fn(i % sets)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fn(i % sets)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cublas", action="store_true")
    ap.add_argument("--tag", default="")
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    rows = B * M
    bf = torch.bfloat16
    rnd = lambda *s: (torch.randn(*s, device=DEV) * 0.1).to(bf)
    res = {}
    products = ("kv_proj", "out_proj", "d_ctx", "d_out_weight", "d_x", "d_kv_weight")
    only = set(args.only.split(",")) if args.only else set(products)

    def run(name, sets, make):
        if name not in only:
            return
        ops_sets = [make() for _ in range(sets)]
        call = lambda i: ops_sets[i]["call"]()
        us = time_us(call, sets)
        kern = _lib.gemm_last_kernel()
        flops = ops_sets[0]["flops"]
        r = {"us": us, "tflops": flops / us / 1e6, "kernel": kern}
        got, want = ops_sets[0]["call"](), ops_sets[0]["ref"]()
        torch.cuda.synchronize()
        r["rel_err"] = float((got.float() - want.float()).abs().max() / want.float().abs().max())
        if args.cublas:
            r["cublas_us"] = time_us(lambda i: ops_sets[i]["ref"](), sets)
        res[name] = r
        del ops_sets
        torch.cuda.empty_cache()

    def kv_proj():
        x, w = rnd(rows, D), rnd(D + HSP, D)
        w[D + H:] = 0
        # (gemm_aux allocates its outputs per call: torch's caching allocator hands the same blocks back, no cudaMalloc)
        return {"call": lambda: ops.gemm_aux(x, w, m=rows, n=D, k=D, aux_cols=H)[0],
                "ref": lambda: (x @ w[:D].t()), "flops": 2 * rows * (D + HSP) * D}

    run("kv_proj", 2, kv_proj)

    def out_proj():
        a, w = rnd(B, D), rnd(D, D)
        out = torch.empty(B, D, device=DEV, dtype=bf)
        return {"call": lambda: ops.linear(a, w, None, out=out), "ref": lambda: a @ w.t(), "flops": 2 * B * D * D}
    run("out_proj", 4, out_proj)

    def d_ctx():
        g, w = rnd(B, D), rnd(D, D)
        out = torch.empty(B, D, device=DEV, dtype=bf)
        return {"call": lambda: ops.matmul_nn(g, w, out=out), "ref": lambda: g @ w, "flops": 2 * B * D * D}
    run("d_ctx", 4, d_ctx)

    def d_out_weight():
        g, c = rnd(B, D), rnd(B, D)
        out = torch.empty(D, D, device=DEV, dtype=bf)
        return {"call": lambda: ops.matmul_tn(g, c, out=out), "ref": lambda: g.t() @ c, "flops": 2 * B * D * D}
    run("d_out_weight", 4, d_out_weight)

    def d_x():
        dvs, w = rnd(rows, D + HSP), rnd(D + HSP, D)
        out = torch.empty(rows, D, device=DEV, dtype=bf)
        return {"call": lambda: ops.matmul_nn(dvs, w, out=out), "ref": lambda: dvs @ w, "flops": 2 * rows * (D + HSP) * D}
    run("d_x", 2, d_x)

    def d_kv_weight():
        dvs, x = rnd(rows, D + HSP), rnd(rows, D)
        out = torch.empty(D + HSP, D, device=DEV, dtype=torch.float32)
        return {"call": lambda: ops.matmul_tn(dvs, x, out=out), "ref": lambda: dvs.t() @ x, "flops": 2 * rows * (D + HSP) * D}
    run("d_kv_weight", 2, d_kv_weight)

    print(json.dumps({"tag": args.tag, "switches": {k: v for k, v in sorted(os.environ.items()) if k.startswith("AECF_")},
                      "products": res}))


if __name__ == "__main__":
    main()
