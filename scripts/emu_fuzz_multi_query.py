"""Offline fuzz of the emulated product path (tests/cuda_emu) against the oracle, several queries per sample:
    python scripts/emu_fuzz_multi_query.py SEED SECONDS"""
import os, random, sys, time
import torch
sys.path.insert(0, __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__))))
from tests import test_gpu_multi_query as MQ
from tests.golden.cases import Case, build_inputs
from tests.helpers import run_oracle
from tests.emu_support import enable_in_this_process
enable_in_this_process()
MQ.DEV = "cpu"
orig_to = torch.Tensor.to
torch.Tensor.to = lambda self, *a, **k: (lambda r: r.clone() if r is self else r)(orig_to(self, *a, **k))
rng = random.Random(int(sys.argv[1]) if len(sys.argv) > 1 else 0)
budget = float(sys.argv[2]) if len(sys.argv) > 2 else 300
t0 = time.time(); n = 0; fails = 0
while time.time() - t0 < budget:
    hd = rng.choice([8, 16, 24, 32, 48, 64, 80, 96, 128])    # 24 .. 96: heads of a non-power-of-two number of chunks
    H = rng.choice([1, 2, 3, 4, 6, 8, 12])
    D = hd * H
    if D > 512: continue
    case = Case(f"mq{n}", B=rng.choice([1, 2, 5, 8, 9, 17]), S=rng.randint(2, 5), M=rng.randint(1, 8), D=D, H=H,
                dropout=rng.choice([0.0, 0.1, 0.5]), base_mask_prob=rng.choice([0.15, 0.5, 1.0]), min_active=rng.choice([1, 2, 9]),
                training=rng.random() < 0.8, kpm=rng.random() < 0.3, pooled_grad=rng.random() < 0.5,
                offset=rng.randint(0, 1000), row0=rng.choice([0, 7, 123456789012]), data_seed=400 + n, peak=rng.choice([0.5, 1.0, 2.0]))
    if case.kpm and case.M == 1: continue
    n += 1
    inp = build_inputs(case)
    for bf in (True, False):
        try:
            ref, ref_grads = run_oracle(case, inp)
            out, info, ent_loss, grads, cm = MQ.run_cuda(case, inp, torch.float32, batch_first=bf)
            MQ.check_against_oracle(case, out, info, ent_loss, grads, ref, ref_grads, 2e-5)
        except Exception as e:
            fails += 1
            print(f"FAIL fp32 bf={bf} {case}\n   {repr(e)[:400]}", flush=True)
    if hd % 8 == 0:
        try:
            MQ.test_bf16_masks_exact_against_stage_rounded_oracle(case)
        except Exception as e:
            fails += 1
            print(f"FAIL bf16 {case}\n   {repr(e)[:400]}", flush=True)
print(f"{n} cases, {fails} failures, {time.time() - t0:.0f}s")
