"""Offline check: every tensor torch.empty/zeros/randn hands out ends right before a PROT_NONE page, then the emulated
product path runs a set of cases; an out-of-bounds access past any buffer's end is a segfault (faulthandler prints it)."""
import ctypes, faulthandler, mmap, sys
import torch
faulthandler.enable()
sys.path.insert(0, __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__))))
from tests.emu_support import enable_in_this_process
enable_in_this_process()
libc = ctypes.CDLL(None, use_errno=True)
PAGE = 4096
keep = []
real_empty = torch.empty
def guarded(shape, dtype):
    numel = 1
    for s in shape: numel *= int(s)
    es = torch.empty((), dtype=dtype).element_size() if False else torch.tensor([], dtype=dtype).element_size()
    nbytes = numel * es
    if nbytes == 0: return real_empty(tuple(shape), dtype=dtype)
    n = (nbytes + 15) // 16 * 16
    total = (n + PAGE - 1) // PAGE * PAGE + PAGE
    m = mmap.mmap(-1, total)
    base = ctypes.addressof(ctypes.c_char.from_buffer(m))
    if libc.mprotect(ctypes.c_void_p(base + total - PAGE), PAGE, 0) != 0: raise OSError(ctypes.get_errno())
    start = total - PAGE - n
    buf = (ctypes.c_char * n).from_buffer(m, start)
    keep.append((m, buf))
    return torch.frombuffer(buf, dtype=torch.uint8)[:nbytes].view(dtype).reshape(tuple(shape))
def norm_shape(args):
    if len(args) == 1 and isinstance(args[0], (tuple, list, torch.Size)): return tuple(args[0])
    return tuple(args)
def g_empty(*args, dtype=None, device=None, **kw):
    return guarded(norm_shape(args), dtype or torch.get_default_dtype())
def g_zeros(*args, dtype=None, device=None, **kw):
    return g_empty(*args, dtype=dtype).zero_()
torch.empty, torch.zeros = g_empty, g_zeros
real_empty_like = torch.empty_like
torch.empty_like = lambda t, **kw: g_empty(t.shape, dtype=kw.get("dtype", t.dtype))
orig_to = torch.Tensor.to
def to_guarded(self, *a, **k):
    r = orig_to(self, *a, **k)
    if r.is_floating_point() or r.dtype in (torch.bool, torch.uint8):
        g = guarded(r.shape, r.dtype); g.copy_(r.detach()); 
        return g.requires_grad_(r.requires_grad) if r.requires_grad else g
    return r
torch.Tensor.to = to_guarded
from tests import test_gpu_parity as P
from tests import test_gpu_multi_query as MQ
from tests.golden.cases import Case, MULTI_QUERY_CASES
P.DEV = "cpu"; MQ.DEV = "cpu"
cases = [c for c in P.FP32_CASES if c.D <= 256] + [Case("tail7", B=7, M=3, D=64, H=8, dropout=0.1, data_seed=901), Case("one", B=1, M=8, D=32, H=1, data_seed=902),
         Case("b33", B=33, M=5, D=128, H=4, kpm=True, data_seed=903)]
n = 0
for c in cases:
    P.test_fp32_matches_oracle(c); n += 1
    if not c.separate_value:
        P.test_fp32_folded_key_projection_matches_oracle(c); n += 1
    if (c.D // c.H) % 8 == 0 and c.dtype == "float32":
        P.test_bf16_masks_exact_against_stage_rounded_oracle(c, True); P.test_bf16_masks_exact_against_stage_rounded_oracle(c, False); n += 2
for c in MULTI_QUERY_CASES[:3]:
    MQ.test_fp32_matches_oracle(c, True); MQ.test_fp32_matches_oracle(c, False); n += 2
P.test_bf16_masks_exact_against_stage_rounded_oracle(cases[1], True); n += 1
print("ok:", n, "runs with every buffer ending at a guard page,", len(keep), "guarded buffers")
