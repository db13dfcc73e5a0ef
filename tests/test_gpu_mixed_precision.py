"""Mixed precision: fp32 master parameters, bf16 activations (include/aecf_b200.h, "mixed precision").

A pool whose parameters are fp32, called with bf16 key / value, must compute exactly what a bf16 twin holding
``p.bfloat16()`` computes -- outputs, info tensors, mask bits and input gradients bit for bit -- and return fp32 parameter
gradients whose bf16 rounding is the twin's gradient bit for bit.  tests/test_emu_mixed_precision.py runs the same bodies
on the host emulation at small sizes (``DEV`` and the sizes below are what it changes).
"""
import copy

import pytest
import torch

import aecf_b200
from aecf_b200 import _lib, ops
from aecf_b200.dp import FusedGradSum, shard_rows

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
B, M, D, H = 1024, 3, 256, 4           # twin cases: tcgen05 products (split-K weight gradients) on the device
D_PAD, H_PAD = 384, 4                  # head_dim 96: the padded lane map
PARAMS = ("in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias")

CASES = {
    "folded": {},
    "unfolded": {"fold": False},
    "per_row_query": {"per_row": True},
    "two_queries": {"S": 2},
    "separate_value": {"value": True},
    "key_padding_mask": {"kpm": True},
    "dropout": {"dropout": 0.1},
    "eval_entropy_grad": {"eval": True},
    "sample_index": {"index": True},
    "seq_first": {"batch_first": False},
    "head_dim_96": {"D": "pad"},
}


def _pools(D_, H_, dropout=0.0, batch_first=True, seed=0):
    """(mixed pool, its shared fp32 query), (bf16 twin, the twin's query): same values, the twin's rounded to bf16."""
    torch.manual_seed(seed)
    q, pool = aecf_b200.create_fusion_pool(D_, M, 0.3, num_heads=H_, dropout=dropout, batch_first=batch_first,
                                           device=DEV, dtype=torch.float32)
    with torch.no_grad():
        pool.attention.in_proj_bias.normal_(0, 0.1)
        pool.attention.out_proj.bias.normal_(0, 0.1)
        q.mul_(6.0)
    twin = aecf_b200.MultimodalAttentionPool(D_, num_heads=H_, dropout=dropout, batch_first=batch_first,
                                             curriculum_masking=aecf_b200.CurriculumMasking(0.3), device=DEV,
                                             dtype=torch.bfloat16)
    names = {n for n, _ in pool.named_parameters()}
    twin.load_state_dict({k: (v.bfloat16() if k in names else v) for k, v in pool.state_dict().items()})
    q_twin = torch.nn.Parameter(q.detach().bfloat16())
    for p in (pool, twin):
        p._want_mask_bits = True
    return (pool, q), (twin, q_twin)


def _step(pool, q, x, inputs, c):
    """One forward + backward; returns (out, info, input gradients)."""
    S, bf = c.get("S", 1), c.get("batch_first", True)
    rows = x.shape[0] if bf else x.shape[1]
    xk = x.clone().requires_grad_(True)
    xv = inputs["v"].clone().requires_grad_(True) if c.get("value") else None
    if c.get("per_row") or S > 1:
        query = inputs["q_rows"].clone().requires_grad_(True)
    else:                                               # the shared fusion query, an expand of the [1, 1, D] parameter
        query = q.expand(rows, -1, -1) if bf else q.expand(-1, rows, -1)
    aecf_b200.set_rng_state(1234, 9)
    out, info = pool(query, xk, xv, key_padding_mask=inputs.get("kpm"), return_info=True,
                     sample_index=inputs.get("index"))
    loss = (out.float() * inputs["g"].float()).sum() + (info["attention_weights"] * inputs["w"]).sum()
    if c.get("eval"):
        loss = loss + (info["entropy"] * 0.5).sum()
    loss.backward()
    grads = {"key": xk.grad, "value": None if xv is None else xv.grad}
    if query.is_leaf and query.requires_grad:
        grads["query_rows"] = query.grad
    return out, info, grads


def _inputs(c, D_, rows):
    S, bf = c.get("S", 1), c.get("batch_first", True)
    gen = torch.Generator().manual_seed(5)
    shape = (rows, M, D_) if bf else (M, rows, D_)
    qshape = (rows, S, D_) if bf else (S, rows, D_)
    inp = {"x": (torch.randn(shape, generator=gen) * 2).bfloat16().to(DEV),
           "v": (torch.randn(shape, generator=gen) * 2).bfloat16().to(DEV),
           "q_rows": (torch.randn(qshape, generator=gen) * 3).bfloat16().to(DEV),
           "g": torch.randn(qshape, generator=gen).bfloat16().to(DEV),
           "w": torch.randn((rows, S, M), generator=gen).to(DEV)}
    if c.get("kpm"):
        kpm = torch.rand((rows, M), generator=gen) < 0.3
        kpm[:, 0] = False
        inp["kpm"] = kpm.to(DEV)
    if c.get("index"):
        inp["index"] = torch.randperm(rows, generator=gen)[: rows // 2].sort().values.to(DEV)
        inp["w"] = inp["w"][: rows // 2]
    return inp


def _compare_twin(c, rows, D_, H_):
    (pool, q), (twin, q_twin) = _pools(D_, H_, dropout=c.get("dropout", 0.0), batch_first=c.get("batch_first", True))
    for p in (pool, twin):
        if c.get("fold") is False:
            p.fold_key_projection = False
        if c.get("eval"):
            p.curriculum_masking.eval()
    inp = _inputs(c, D_, rows)
    out_m, info_m, g_m = _step(pool, q, inp["x"], inp, c)
    out_t, info_t, g_t = _step(twin, q_twin, inp["x"], inp, c)
    aecf_b200.set_rng_state(None)
    assert out_m.dtype == torch.bfloat16 and torch.equal(out_m, out_t), "out"
    assert set(info_m) == set(info_t)
    for k in info_m:
        assert info_m[k].dtype == info_t[k].dtype and torch.equal(info_m[k], info_t[k]), f"info[{k!r}]"
    for k, v in g_m.items():
        if v is not None:
            assert v.dtype == torch.bfloat16 and torch.equal(v, g_t[k]), f"{k}.grad"
    att_m, att_t = pool.attention, twin.attention
    for name in PARAMS:
        gm, gt = att_m.get_parameter(name).grad, att_t.get_parameter(name).grad
        assert gm.dtype == torch.float32, f"{name}.grad is {gm.dtype}"
        assert torch.equal(gm.bfloat16(), gt), f"{name}.grad rounded to bf16 differs from the twin's"
    if q.grad is not None or q_twin.grad is not None:
        assert q.grad.dtype == torch.float32 and torch.equal(q.grad.bfloat16(), q_twin.grad), "fusion query .grad"
    return pool, twin


@pytest.mark.parametrize("case", list(CASES))
def test_mixed_matches_bf16_twin(case):
    c = CASES[case]
    D_, H_ = (D_PAD, H_PAD) if c.get("D") == "pad" else (D, H)
    _compare_twin(c, B, D_, H_)


def test_mixed_matches_bf16_twin_at_headline_size():
    """B = 65 536, M = 3, D = 512, H = 8: the 2SM and split-K products and the streaming pool kernels."""
    _compare_twin({}, 65536, 512, 8)


def test_param_cast_rounds_like_tensor_bfloat16():
    gen = torch.Generator().manual_seed(3)
    specials = torch.tensor([0.0, -0.0, float("inf"), float("-inf"), 3.4e38, -3.4e38, 3.3895e38, 1e-40, -1e-40, 1e-45,
                             1.17e-38, 2.0 ** -133, 1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, -(1.0 + 2.0 ** -8),
                             1.0 + 2.0 ** -8 + 2.0 ** -20, 65504.0, 1.0 / 3.0])
    halves = (torch.randint(0, 1 << 16, (4096,), generator=gen, dtype=torch.int32) << 16 | 0x8000).view(torch.float32)
    rnd = torch.randn(100003, generator=gen) * torch.exp(torch.randn(100003, generator=gen) * 20)
    segments = [torch.cat([specials, halves, rnd]), torch.randn(1, generator=gen), torch.randn(13, generator=gen),
                torch.randn(8, generator=gen), torch.randn(0), torch.randn(7, 9, generator=gen),
                torch.randn(257, generator=gen), torch.randn(3, 5, generator=gen)]
    segments = [s.to(DEV) for s in segments]
    seg0 = segments[0]
    seg0[5] = float("nan")
    block, views = ops.param_cast(segments)
    for s, v in zip(segments, views):
        assert v.shape == s.shape and v.dtype == torch.bfloat16
        assert v.data_ptr() % 16 == 0
        want = s.bfloat16()
        nan = torch.isnan(s)
        assert torch.equal(torch.isnan(v), nan)
        assert torch.equal(v[~nan].view(torch.int16), want[~nan].view(torch.int16))
    # an fp32 source that is not 16-byte aligned takes the scalar path
    odd = torch.randn(1000, device=DEV)[1:]
    _, (v,) = ops.param_cast([odd])
    assert torch.equal(v.view(torch.int16), odd.bfloat16().view(torch.int16))
    with pytest.raises(ValueError):
        ops.param_cast([torch.zeros(8, device=DEV)] * 9)


def test_mixed_gradients_closer_to_oracle_than_bf16():
    """The point of the feature: the fp32 gradients keep the bits the bf16 module rounds away.  Against the fp32
    stage-rounded oracle (bf16 storage, the bf16-rounded weights both modules compute with), each parameter gradient's
    max relative error of the mixed module is no larger than the bf16 twin's."""
    from oracle import aecf_oracle as oracle
    (pool, q), (twin, q_twin) = _pools(D, H)
    for p in (pool, twin):
        p.curriculum_masking = None
    inp = _inputs({}, D, B)
    inp["w"] = torch.zeros_like(inp["w"])
    _step(pool, q, inp["x"], inp, {})
    _step(twin, q_twin, inp["x"], inp, {})
    cpu = lambda t: t.detach().float().cpu()
    att = twin.attention
    x, q0 = cpu(inp["x"]), cpu(q_twin).expand(B, 1, D)
    fwd = oracle.pool_forward(q0, x, None, cpu(att.in_proj_weight), cpu(att.in_proj_bias), cpu(att.out_proj.weight),
                              cpu(att.out_proj.bias), H, storage=torch.bfloat16, fold_key=True)
    ref = oracle.pool_backward(q0, x, None, cpu(att.in_proj_weight), cpu(att.out_proj.weight), H, fwd.saved, cpu(inp["g"]),
                               storage=torch.bfloat16, fold_key=True)
    ref["query"] = ref["query"].sum(0, keepdim=True)
    report = {}
    for name in PARAMS + ("query",):
        gm = q.grad if name == "query" else pool.attention.get_parameter(name).grad
        gt = q_twin.grad if name == "query" else twin.attention.get_parameter(name).grad
        r = ref[name].reshape(gm.shape)
        scale = float(r.abs().max())
        em = float((cpu(gm) - r).abs().max()) / scale
        et = float((cpu(gt) - r).abs().max()) / scale
        report[name] = (em, et)
    print("max relative error against the oracle, mixed / bf16:", {k: f"{a:.2e} / {b:.2e}" for k, (a, b) in report.items()})
    for name, (em, et) in report.items():
        assert em <= et, f"{name}: mixed {em:.3e} > bf16 {et:.3e}"


def test_mixed_step_replays_in_a_cuda_graph():
    """A graphed mixed step replays bit-identically to eager steps, and picks up fp32 masters changed in place between
    replays (an optimizer step): the shadow is made inside the graph, on every replay."""
    from aecf_b200 import graphs
    (pool, q), _ = _pools(D, H)
    inp = _inputs({}, D, B)
    x, g = inp["x"], inp["g"]
    params = {n: pool.attention.get_parameter(n) for n in PARAMS} | {"query": q}

    def step():
        out = pool(q.expand(B, -1, -1), x)
        (out.float() * g.float()).sum().backward()
        return {n: p.grad for n, p in params.items()}

    def reset():
        for p in params.values():
            p.grad = None

    def eager():
        reset()
        aecf_b200.set_rng_state(77, 0)
        got = {n: t.clone() for n, t in step().items()}
        torch.cuda.synchronize()
        return got

    graphed = graphs.GraphedStep(step, reset=reset)
    for update in range(2):
        want = eager()
        aecf_b200.set_rng_state(77, 0)
        got = graphed()
        torch.cuda.synchronize()
        for k in want:
            assert got[k].dtype == torch.float32 and torch.equal(got[k], want[k]), f"replay {update} differs from eager in {k}"
        with torch.no_grad():                           # an optimizer step on the fp32 masters
            for p in params.values():
                p.add_(torch.randn_like(p) * 0.05)
    aecf_b200.set_rng_state(None)


@pytest.mark.parametrize("heads", [8, 12])
def test_mixed_fused_data_parallel_sum(heads):
    """The in-backward cross-rank sum with W ranks emulated on one device: fp32 gradients identical on every rank, and
    their bf16 rounding equal to the bf16 module's run of the same ranks.  H = 12: the raw-sum layout of the bf16 compute
    (16 score columns) differs from an fp32 one (12), so the buffers must be sized for the compute dtype."""
    world, rows_total, D_ = 2, 2048, 768
    (pool0, q0), (twin0, qt0) = _pools(D_, heads)
    x = (torch.randn(rows_total, M, D_, generator=torch.Generator().manual_seed(2)) * 2).bfloat16().to(DEV)
    g = torch.randn(rows_total, 1, D_, generator=torch.Generator().manual_seed(4)).bfloat16().to(DEV)

    def run(base, qbase):
        buffers, flags = [None] * world, [None] * world
        ranks = []
        for r in range(world):                          # each rank on its own stream: the sum's flag barrier waits for all
            pool = copy.deepcopy(base)
            q = torch.nn.Parameter(qbase.detach().clone())
            pool._dp = FusedGradSum(pool, average=False, local_ranks=(r, world, buffers, flags))
            ranks.append((pool, q, torch.cuda.Stream(device=DEV)))
        torch.cuda.synchronize()
        for r, (pool, q, stream) in enumerate(ranks):
            row0, rows = shard_rows(rows_total, r, world)
            pool.row_offset = row0
            with torch.cuda.stream(stream):
                aecf_b200.set_rng_state(3, 1)
                out = pool(q.expand(rows, -1, -1), x[row0:row0 + rows])
                (out.float() * g[row0:row0 + rows].float()).sum().backward()
        torch.cuda.synchronize()
        assert all(p._dp.ran for p, _, _ in ranks)
        return [{n: p.attention.get_parameter(n).grad for n in PARAMS} | {"query": q.grad} for p, q, _ in ranks]

    got = run(pool0, q0)
    ref = run(twin0, qt0)
    aecf_b200.set_rng_state(None)
    for r in range(1, world):
        for k in got[0]:
            assert torch.equal(got[r][k], got[0][k]), f"rank {r} differs from rank 0 in {k}"
    for k in got[0]:
        assert got[0][k].dtype == torch.float32 and torch.equal(got[0][k].bfloat16(), ref[0][k]), k


def test_mixed_projections_match_bf16_twin():
    gen = torch.Generator().manual_seed(8)
    lin_a = torch.nn.Linear(48, 64).to(DEV)
    lin_b = torch.nn.Linear(32, 64).to(DEV)
    head = torch.nn.Linear(64, 40).to(DEV)
    twins = [copy.deepcopy(m).bfloat16() for m in (lin_a, lin_b, head)]
    rows = 256
    xa = torch.randn(rows, 48, generator=gen).bfloat16().to(DEV)
    xb = torch.randn(rows, 32, generator=gen).bfloat16().to(DEV)
    g_tok = torch.randn(rows, 2, 64, generator=gen).bfloat16().to(DEV)
    g_head = torch.randn(rows, 40, generator=gen).bfloat16().to(DEV)

    def run(a, b, h):
        xa_ = xa.clone().requires_grad_(True)
        tokens = aecf_b200.project_tokens([(xa_, a), (xb, b)])
        logits = aecf_b200.linear(tokens[:, 0, :].contiguous(), h)
        ((tokens.float() * g_tok.float()).sum() + (logits.float() * g_head.float()).sum()).backward()
        return tokens, logits, xa_.grad

    t_m, l_m, gx_m = run(lin_a, lin_b, head)
    t_t, l_t, gx_t = run(*twins)
    assert t_m.dtype == torch.bfloat16 and torch.equal(t_m, t_t)
    assert l_m.dtype == torch.bfloat16 and torch.equal(l_m, l_t)
    assert torch.equal(gx_m, gx_t)
    for m, t in zip((lin_a, lin_b, head), twins):
        for name in ("weight", "bias"):
            gm, gt = getattr(m, name).grad, getattr(t, name).grad
            assert gm.dtype == torch.float32 and torch.equal(gm.bfloat16(), gt), name


def test_mixed_rejections_stay():
    (pool, q), (twin, q_twin) = _pools(64, 2)
    x32 = torch.randn(4, M, 64, device=DEV)
    with pytest.raises(RuntimeError, match="expected query/key/value of dtype torch.bfloat16"):
        twin(q_twin.float().expand(4, -1, -1), x32)                       # bf16 parameters, fp32 inputs
    with pytest.raises(RuntimeError, match="expected query/key/value of dtype torch.float32"):
        pool(q_twin.expand(4, -1, -1), x32.bfloat16())                    # bf16 shared query on fp32 parameters
    with pytest.raises(RuntimeError, match="expected query/key/value of dtype torch.float32"):
        pool(q.expand(4, -1, -1), x32.bfloat16(), x32)                    # fp32 value next to a bf16 key
    assert _lib.SITE_COUNT == 22
