"""GPU: the native LlamaRMSNorm kernels (csrc/glue.cu) against the stock HF forward and its eager backward, bit for bit.

Every comparison goes through an integer view, so signed zeros, inf and NaN patterns count too."""
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
EPS = 1e-6


def _bits_equal(a, b, what):
    assert a.shape == b.shape and a.dtype == b.dtype, (what, a.shape, b.shape, a.dtype, b.dtype)
    it = {2: torch.int16, 4: torch.int32}[a.element_size()]
    ai, bi = a.contiguous().view(it), b.contiguous().view(it)
    bad = (ai != bi).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.shape[0]} elements differ, first at {bad[0].tolist()}: " \
                             f"{a[tuple(bad[0])].item()} vs {b[tuple(bad[0])].item()}"


def _stock_forward():
    from transformers.models.llama import modeling_llama as ml
    return ml.LlamaRMSNorm.forward


def _norm(H, dt):
    from transformers.models.llama import modeling_llama as ml
    m = ml.LlamaRMSNorm(H, eps=EPS).to(DEV, dt)
    with torch.no_grad():
        m.weight.copy_((1 + 0.5 * torch.randn(H, generator=torch.Generator().manual_seed(H))).to(dt))
    return m


def _both(m, x, dy, train_w=True):
    """(y, dx, dw) of the stock forward and of the native path on the same inputs."""
    from sow_b200.llama_glue import _RMSNorm, rmsnorm_native_ok
    out = []
    m.weight.requires_grad_(train_w)
    for native in (False, True):
        xi = x.clone().requires_grad_(True)
        if native:
            assert rmsnorm_native_ok(xi, m.weight, m.variance_epsilon)
            y = _RMSNorm.apply(xi, m.weight, m.variance_epsilon)
        else:
            y = _stock_forward()(m, xi)
        ins = (xi, m.weight) if train_w else (xi,)
        gs = torch.autograd.grad(y, ins, dy)
        out.append((y, gs[0], gs[1] if train_w else None))
    m.weight.requires_grad_(True)
    return out


def _check(m, x, dy, train_w=True):
    (ys, dxs, dws), (yn, dxn, dwn) = _both(m, x, dy, train_w)
    _bits_equal(yn, ys, "y")
    _bits_equal(dxn, dxs, "dx")
    if train_w:
        _bits_equal(dwn, dws, "dw")


def _mixed(shape, dt, gen):
    """Values over the whole range: normal draws at several scales, subnormals, +-0, +-inf, NaN."""
    n = 1
    for s in shape:
        n *= s
    e = torch.randint(-20, 20, (n,), device=DEV, generator=gen).float()
    v = (torch.randn(n, device=DEV, generator=gen) * torch.exp2(e)).to(dt)
    sel = torch.randint(0, 64, (n,), device=DEV, generator=gen)
    v = torch.where(sel == 0, torch.zeros_like(v), v)
    v = torch.where(sel == 1, -torch.zeros_like(v), v)
    v = torch.where(sel == 2, (torch.rand(n, device=DEV, generator=gen) * torch.finfo(dt).tiny).to(dt), v)
    return v.view(shape)


WIDTHS = [128, 512, 1024, 4096]
ROWS = [1, 15, 16, 17, 2048, 32768]


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("rows", ROWS)
def test_rmsnorm_matches_stock_bit_for_bit(rows, H, dt):
    from sow_b200.llama_glue import rmsnorm_native_ok
    gen = torch.Generator(device=DEV).manual_seed(rows * 7 + H)
    m = _norm(H, dt)
    x = torch.randn(rows, H, device=DEV, generator=gen).to(dt)
    if not rmsnorm_native_ok(x, m.weight, EPS):
        assert rows < 16 and H != 128            # torch's reduction order differs there: the stock path runs
        return
    dy = (torch.randn(x.shape, device=DEV, generator=gen) * 1e-2).to(dt)
    _check(m, x, dy)


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_rmsnorm_matches_stock_at_the_bench_shape_with_saved_rs(dt):
    from sow_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(5)
    m = _norm(1024, dt)
    x = (torch.randn(128, 256, 1024, device=DEV, generator=gen) * 3).to(dt)
    dy = (torch.randn(x.shape, device=DEV, generator=gen) * 1e-3).to(dt)
    _check(m, x, dy)
    xf = x.float()
    rs_stock = torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + EPS)[..., 0]
    _, rs = ops.rmsnorm_fwd(x, m.weight, EPS)
    _bits_equal(rs, rs_stock, "rs")


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("H", [512, 1024])
def test_rmsnorm_edge_values(H, dt):
    """Large dynamic range, zeros, whole-zero rows, subnormals; then rows with +-inf and NaN; then w * hb overflowing."""
    gen = torch.Generator(device=DEV).manual_seed(11)
    m = _norm(H, dt)
    x = _mixed((64, H), dt, gen)
    x[3] = 0.0
    x[4] = -0.0
    x[5] = (torch.rand(H, device=DEV, generator=gen) * torch.finfo(dt).tiny).to(dt)   # a row of subnormals
    dy = _mixed((64, H), dt, gen)
    dy[7] = 0.0
    _check(m, x, dy)
    x2 = x.clone()
    x2[8, 3] = float("inf")
    x2[9, 5] = float("-inf")
    x2[10, 7] = float("nan")
    dy2 = dy.clone()
    dy2[11, 1] = float("inf")
    dy2[12, 2] = float("nan")
    _check(m, x2, dy2)
    # a huge weight: w * hb (and dy * w) overflow, to inf in fp16, as eager's rounding does
    big = torch.finfo(dt).max / 4
    with torch.no_grad():
        m.weight[::7] = big
    _check(m, x, (torch.randn(x.shape, device=DEV, generator=gen) * 1e3).to(dt))


def test_saved_rs_matches_stock_over_every_bf16_magnitude():
    """rs = rsqrtf(mean(x^2) + eps) against torch.rsqrt over a wide range of arguments: row i holds the i-th finite
    bf16 pattern once (and zeros), so mean(x^2) runs from 0 through subnormal, normal and overflowing (inf) values."""
    from sow_b200 import ops
    m = _norm(128, torch.bfloat16)
    pats = torch.arange(0, 32768, device=DEV, dtype=torch.int32).to(torch.int16).view(torch.bfloat16)
    pats = pats[torch.isfinite(pats)]
    x = torch.zeros(pats.numel(), 128, device=DEV, dtype=torch.bfloat16)
    x[:, 0] = pats
    x[:, 77] = pats.flip(0)
    for eps in (EPS, 1e-5, 0.0):
        _, rs = ops.rmsnorm_fwd(x, m.weight, eps)
        xf = x.float()
        ref = torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + eps)[:, 0]
        _bits_equal(rs, ref, f"rs (eps {eps})")


def test_frozen_weight_writes_no_product():
    """With w frozen the backward writes no dy * hb product and returns no dw; dx is still the stock one."""
    from sow_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(2)
    m = _norm(1024, torch.bfloat16)
    x = torch.randn(64, 1024, device=DEV, generator=gen).to(torch.bfloat16)
    dy = torch.randn(64, 1024, device=DEV, generator=gen).to(torch.bfloat16)
    _check(m, x, dy, train_w=False)
    _, rs = ops.rmsnorm_fwd(x, m.weight, EPS)
    _, p = ops.rmsnorm_bwd(dy, x, m.weight, rs, want_p=False)
    assert p is None


def test_non_contiguous_gradient_runs_the_stock_backward():
    from sow_b200.llama_glue import _RMSNorm
    gen = torch.Generator(device=DEV).manual_seed(4)
    m = _norm(512, torch.float16)
    x = torch.randn(32, 512, device=DEV, generator=gen).to(torch.float16)
    dy_t = torch.randn(512, 32, device=DEV, generator=gen).to(torch.float16)
    res = []
    for native in (False, True):
        xi = x.clone().requires_grad_(True)
        y = _RMSNorm.apply(xi, m.weight, EPS) if native else _stock_forward()(m, xi)
        res.append(torch.autograd.grad(y, (xi, m.weight), dy_t.t()))
    _bits_equal(res[1][0], res[0][0], "dx")
    _bits_equal(res[1][1], res[0][1], "dw")


def test_rmsnorm_under_cuda_graph_capture():
    from sow_b200.llama_glue import _RMSNorm
    gen = torch.Generator(device=DEV).manual_seed(6)
    m = _norm(1024, torch.bfloat16)
    x = torch.randn(256, 1024, device=DEV, generator=gen).to(torch.bfloat16).requires_grad_(True)
    dy = torch.randn(256, 1024, device=DEV, generator=gen).to(torch.bfloat16)

    def run():
        y = _RMSNorm.apply(x, m.weight, EPS)
        # detached: no autograd node made outside the capture (and its stream) outlives this call
        return [t.detach() for t in (y,) + torch.autograd.grad(y, (x, m.weight), dy)]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ref = [t.clone() for t in run()]
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = run()
    with torch.no_grad():
        x.copy_(torch.randn(x.shape, device=DEV, generator=gen).to(torch.bfloat16))
    g.replay()
    torch.cuda.synchronize()
    ys, dxs, dws = _both(m, x.detach(), dy)[0]     # the stock chain on the new input
    _bits_equal(outs[0], ys, "graphed y")
    _bits_equal(outs[1], dxs, "graphed dx")
    _bits_equal(outs[2], dws, "graphed dw")
    assert not torch.equal(outs[0], ref[0])


def _count_norm(monkeypatch):
    from sow_b200 import ops
    calls = {"fwd": 0, "bwd": 0}
    f, b = ops.rmsnorm_fwd, ops.rmsnorm_bwd

    def fwd(*a, **k):
        calls["fwd"] += 1
        return f(*a, **k)

    def bwd(*a, **k):
        calls["bwd"] += 1
        return b(*a, **k)
    monkeypatch.setattr(ops, "rmsnorm_fwd", fwd)
    monkeypatch.setattr(ops, "rmsnorm_bwd", bwd)
    return calls


def test_every_norm_of_the_bench_model_runs_native(monkeypatch):
    """Llama-350M as the bench builds it: 24 layers x 2 norms + the final norm, one forward and one backward each."""
    from sow_b200.trainer import SoWTrainer, TrainConfig
    calls = _count_norm(monkeypatch)
    tr = SoWTrainer(TrainConfig(batch_size=2), torch.device(DEV, 0))
    ids = torch.randint(1, 32000, (2, 256), generator=torch.Generator().manual_seed(0)).to(DEV)
    tr.step(ids)
    assert calls == {"fwd": 49, "bwd": 49}


def test_fp32_and_compiled_models_make_no_native_norm_call(monkeypatch):
    import torch._dynamo
    from sow_b200.trainer import build_llama, LLAMA_TARGETS
    from tn_gradient.prepare import SoWConfig, prepare_sow
    calls = _count_norm(monkeypatch)
    ids = torch.randint(1, 32000, (2, 64), generator=torch.Generator().manual_seed(0)).to(DEV)
    model = prepare_sow(build_llama("llama_60m"), SoWConfig(target_modules=LLAMA_TARGETS, rank=8, init_method="normal",
                                                            device=DEV))
    model.to(DEV, torch.float32)(input_ids=ids, labels=ids).loss.backward()
    assert calls == {"fwd": 0, "bwd": 0}
    model.to(DEV, torch.bfloat16)
    torch._dynamo.reset()
    ex = torch._dynamo.explain(model)(input_ids=ids)
    assert ex.graph_break_count == 0, ex.break_reasons
    assert calls == {"fwd": 0, "bwd": 0}
