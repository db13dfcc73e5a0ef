"""Offline fuzz of the emulated product path (tests/cuda_emu) against the oracle, one query per sample:
    python scripts/emu_fuzz_single_query.py SEED SECONDS"""
import random, sys, time, traceback
import torch
sys.path.insert(0, __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__))))
from tests import test_gpu_parity as P
from tests.golden.cases import Case
from tests.emu_support import enable_in_this_process
enable_in_this_process()
P.DEV = "cpu"
orig_to = torch.Tensor.to
def to_copy(self, *a, **k):
    r = orig_to(self, *a, **k)
    return r.clone() if r is self else r
torch.Tensor.to = to_copy
rng = random.Random(int(sys.argv[1]) if len(sys.argv) > 1 else 0)
budget = float(sys.argv[2]) if len(sys.argv) > 2 else 300
t0 = time.time(); n = 0; fails = 0
while time.time() - t0 < budget:
    hd = rng.choice([8, 16, 24, 32, 48, 64, 80, 96, 128])    # 24 .. 96: heads of a non-power-of-two number of chunks
    H = rng.choice([1, 2, 3, 4, 5, 6, 8, 12, 16])
    D = hd * H
    if D > 768: continue
    M = rng.randint(1, 8)
    B = rng.choice([1, 2, 3, 7, 8, 9, 15, 17, 31, 33, 40])
    case = Case(f"fuzz{n}", B=B, M=M, D=D, H=H, dropout=rng.choice([0.0, 0.0, 0.1, 0.5]),
                base_mask_prob=rng.choice([0.15, 0.5, 0.9, 1.0]), min_active=rng.choice([1, 1, 2, 3, 9]),
                training=rng.random() < 0.8, kpm=rng.random() < 0.3 and M > 1, separate_value=rng.random() < 0.2,
                pooled_grad=rng.random() < 0.5, offset=rng.randint(0, 1000), row0=rng.choice([0, 5, 123456789012]),
                data_seed=100 + n, peak=rng.choice([0.5, 1.0, 2.0, 4.0]))
    n += 1
    tests = [("fp32", lambda: P.test_fp32_matches_oracle(case))]
    if not case.separate_value:
        tests.append(("fold32", lambda: P.test_fp32_folded_key_projection_matches_oracle(case)))
    if hd % 8 == 0:
        tests.append(("bf16f", lambda: P.test_bf16_masks_exact_against_stage_rounded_oracle(case, True)))
        tests.append(("bf16u", lambda: P.test_bf16_masks_exact_against_stage_rounded_oracle(case, False)))
    for tag, fn in tests:
        try:
            fn()
        except Exception as e:
            fails += 1
            print(f"FAIL {tag} {case}\n   {repr(e)[:400]}", flush=True)
print(f"{n} cases, {fails} failures, {time.time() - t0:.0f}s")
