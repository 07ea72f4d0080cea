"""GPU: the native rotary embedding and SwiGLU kernels (csrc/glue.cu) against the stock HF / torch functions, bit for bit.

Adam at lr 1e-2 turns a one-ulp gradient difference into a 2 lr weight difference, so nothing short of bit equality is
accepted: every comparison goes through .view(torch.int16) and covers signed zeros, inf and NaN patterns too."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _bits_equal(a, b, what):
    assert a.shape == b.shape and a.dtype == b.dtype, (what, a.shape, b.shape, a.dtype, b.dtype)
    it = {1: torch.int8, 2: torch.int16, 4: torch.int32}[a.element_size()]
    ai, bi = a.contiguous().view(it), b.contiguous().view(it)
    bad = (ai != bi).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.shape[0]} elements differ, first at {bad[0].tolist()}: " \
                             f"{a[tuple(bad[0])].item()} vs {b[tuple(bad[0])].item()}"


def _stock_rope():
    from transformers.models.llama import modeling_llama as ml
    f = ml.apply_rotary_pos_emb
    return getattr(f, "stock", f)


def _cos_sin(B, S, D, dt, batched):
    """HF's LlamaRotaryEmbedding tables (position 0: sin == 0 exactly); batched -> one row of positions per sequence."""
    inv = 1.0 / (10000.0 ** (torch.arange(0, D, 2, device=DEV, dtype=torch.float32) / D))
    pos = torch.arange(S, device=DEV, dtype=torch.float32)[None].expand(B if batched else 1, S)
    if batched:
        pos = pos + torch.arange(B, device=DEV, dtype=torch.float32)[:, None] * 3
    fr = pos[..., None] * inv
    emb = torch.cat((fr, fr), dim=-1)
    return emb.cos().to(dt), emb.sin().to(dt)


ROPE_CASES = [   # B, Hq, Hk, S, D, dtype, batched cos/sin
    (128, 16, 16, 256, 64, torch.bfloat16, False),     # the bench shape
    (3, 5, 5, 77, 64, torch.bfloat16, False),          # S not a multiple of anything
    (4, 4, 4, 33, 64, torch.bfloat16, True),           # per-sequence cos / sin
    (2, 8, 8, 50, 128, torch.bfloat16, False),         # D = 128
    (2, 8, 2, 40, 64, torch.bfloat16, False),          # GQA: fewer k heads
    (8, 16, 16, 96, 64, torch.float16, False),         # fp16
    (3, 4, 4, 21, 128, torch.float16, True),
]


@pytest.mark.parametrize("g_layout", ["bhsd", "bshd"])
@pytest.mark.parametrize("case", ROPE_CASES, ids=lambda c: "x".join(str(v) for v in c[:5]) + f"-{str(c[5])[6:]}-{c[6]}")
def test_rope_matches_stock_bit_for_bit(case, g_layout):
    from sow_b200.llama_glue import _RoPE, rope_native_ok
    B, Hq, Hk, S, D, dt, batched = case
    gen = torch.Generator(device=DEV).manual_seed(B * 1000 + S)
    # q, k as HF makes them: (B, S, H*D) projections viewed (B, S, H, D) and transposed to (B, H, S, D)
    q0 = torch.randn(B, S, Hq * D, device=DEV, generator=gen).to(dt)
    k0 = torch.randn(B, S, Hk * D, device=DEV, generator=gen).to(dt)
    q0[0, :2, :16] = -0.0                                   # signed zeros through the products
    k0[-1, 0, :8] = 0.0
    cos, sin = _cos_sin(B, S, D, dt, batched)
    g_shape = (B, Hq, S, D)
    gq = torch.randn(B, Hq, S, D, device=DEV, generator=gen).to(dt)
    gk = torch.randn(B, Hk, S, D, device=DEV, generator=gen).to(dt)
    gq[:, :, 0] = -0.0                                       # -0 gradients at position 0, where sin == 0
    gq[0, 0, 1, ::3] = -0.0
    if g_layout == "bshd":
        gq = gq.transpose(1, 2).contiguous().transpose(1, 2)
        gk = gk.transpose(1, 2).contiguous().transpose(1, 2)
    outs = []
    for native in (False, True):
        q = q0.clone().view(B, S, Hq, D).transpose(1, 2).requires_grad_(True)
        k = k0.clone().view(B, S, Hk, D).transpose(1, 2).requires_grad_(True)
        if native:
            assert rope_native_ok(q, k, cos, sin)
            qe, ke = _RoPE.apply(q, k, cos, sin)
        else:
            qe, ke = _stock_rope()(q, k, cos, sin)
        dq, dk = torch.autograd.grad((qe, ke), (q, k), (gq, gk))
        outs.append((qe, ke, dq, dk))
    (qs, ks, dqs, dks), (qn, kn, dqn, dkn) = outs
    assert qn.stride() == qs.stride() and kn.stride() == ks.stride(), (qn.stride(), qs.stride())
    _bits_equal(qn, qs, "q_embed")
    _bits_equal(kn, ks, "k_embed")
    _bits_equal(dqn, dqs, "dq")
    _bits_equal(dkn, dks, "dk")
    assert g_shape == tuple(dqn.shape)


def _all_patterns(dt, reps, gen):
    """Every 16-bit pattern of dt (all finite values of both signs, subnormals, +-0, +-inf, NaNs) in random order, reps
    times, plus an odd tail so the element-by-element path runs too."""
    pats = torch.arange(-32768, 32768, device=DEV, dtype=torch.int32).to(torch.int16).view(dt)
    parts = [pats[torch.randperm(65536, device=DEV, generator=gen)] for _ in range(reps)]
    return torch.cat(parts + [pats[:5]])


def _mixed(n, dt, gen):
    """Random values over the whole range: normal draws at several scales, subnormals, +-0, +-inf, NaN."""
    v = torch.randn(n, device=DEV, generator=gen) * torch.exp2(torch.randint(-30, 30, (n,), device=DEV, generator=gen).float())
    v = v.to(dt)
    sel = torch.randint(0, 16, (n,), device=DEV, generator=gen)
    tiny = torch.finfo(dt).tiny
    v = torch.where(sel == 0, torch.zeros_like(v), v)
    v = torch.where(sel == 1, -torch.zeros_like(v), v)
    v = torch.where(sel == 2, torch.full_like(v, float("inf")), v)
    v = torch.where(sel == 3, torch.full_like(v, float("-inf")), v)
    v = torch.where(sel == 4, torch.full_like(v, float("nan")), v)
    v = torch.where(sel == 5, (torch.rand(n, device=DEV, generator=gen) * tiny).to(dt), v)   # subnormals
    return v


def _swiglu_both(gate, up, dh):
    from sow_b200.llama_glue import _SwiGLU, swiglu_native_ok
    res = []
    for native in (False, True):
        g = gate.clone().requires_grad_(True)
        u = up.clone().requires_grad_(True)
        if native:
            assert swiglu_native_ok(g, u)
            h = _SwiGLU.apply(g, u)
        else:
            h = F.silu(g) * u
        dg, du = torch.autograd.grad(h, (g, u), dh)
        res.append((h, dg, du))
    return res


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_swiglu_matches_stock_over_every_16bit_pattern(dt):
    """gate runs through all 65536 patterns (|x| > 88 where expf overflows, subnormals, +-0, +-inf, NaN) against up and dh
    drawn over the whole range as well."""
    gen = torch.Generator(device=DEV).manual_seed(7)
    gate = _all_patterns(dt, 8, gen)
    n = gate.numel()
    up = _mixed(n, dt, gen)
    dh = _mixed(n, dt, gen)
    (hs, dgs, dus), (hn, dgn, dun) = _swiglu_both(gate, up, dh)
    _bits_equal(hn, hs, "h")
    _bits_equal(dgn, dgs, "dgate")
    _bits_equal(dun, dus, "dup")
    # and with up = dh = 1: the bare silu / silu_backward of every pattern
    ones = torch.ones_like(gate)
    (hs, dgs, dus), (hn, dgn, dun) = _swiglu_both(gate, ones, ones)
    _bits_equal(hn, hs, "silu")
    _bits_equal(dgn, dgs, "silu_backward")
    _bits_equal(dun, dus, "silu (dup)")


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_swiglu_matches_stock_at_the_bench_shape(dt):
    gen = torch.Generator(device=DEV).manual_seed(3)
    shape = (128, 256, 2736)
    gate = (torch.randn(shape, device=DEV, generator=gen) * 2).to(dt)
    up = torch.randn(shape, device=DEV, generator=gen).to(dt)
    dh = (torch.randn(shape, device=DEV, generator=gen) * 1e-3).to(dt)
    (hs, dgs, dus), (hn, dgn, dun) = _swiglu_both(gate, up, dh)
    _bits_equal(hn, hs, "h")
    _bits_equal(dgn, dgs, "dgate")
    _bits_equal(dun, dus, "dup")


# ---------------------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------------------

class _Stock:
    """Within the block the Llama glue is switched off: the stock apply_rotary_pos_emb global, no MLP forward override."""

    def __init__(self, *models):
        self.models = models

    def __enter__(self):
        from transformers.models.llama import modeling_llama as ml
        self.ml, self.disp = ml, ml.apply_rotary_pos_emb
        ml.apply_rotary_pos_emb = _stock_rope()
        self.saved = []
        for model in self.models:
            for m in model.modules():
                if "forward" in m.__dict__:
                    self.saved.append((m, m.__dict__.pop("forward")))
        return self

    def __exit__(self, *exc):
        self.ml.apply_rotary_pos_emb = self.disp
        for m, f in self.saved:
            m.forward = f


def _count_native(monkeypatch):
    from sow_b200 import ops
    calls = {"rope": 0, "swiglu": 0}
    rf, sf = ops.rope_fwd, ops.swiglu_fwd

    def rope(*a):
        calls["rope"] += 1
        return rf(*a)

    def swiglu(*a):
        calls["swiglu"] += 1
        return sf(*a)
    monkeypatch.setattr(ops, "rope_fwd", rope)
    monkeypatch.setattr(ops, "swiglu_fwd", swiglu)
    return calls


def _llama350m_2layers(dtype):
    from sow_b200.trainer import LLAMA_TARGETS
    from tn_gradient.prepare import SoWConfig, prepare_sow
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(vocab_size=32000, hidden_size=1024, intermediate_size=2736, num_hidden_layers=2,
                      num_attention_heads=16, max_position_embeddings=1024, rms_norm_eps=1e-6, hidden_act="silu",
                      use_cache=False, tie_word_embeddings=False)
    torch.manual_seed(0)
    model = LlamaForCausalLM(cfg)
    model = prepare_sow(model, SoWConfig(target_modules=LLAMA_TARGETS, rank=50, init_method="normal", device=DEV))
    return model.to(DEV, dtype)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_llama_350m_shaped_loss_and_grads_are_identical(dtype, monkeypatch):
    calls = _count_native(monkeypatch)
    model = _llama350m_2layers(dtype)
    ids = torch.randint(1, 32000, (8, 256), generator=torch.Generator().manual_seed(1)).to(DEV)
    res = []
    for stock in (True, False):
        model.zero_grad(set_to_none=True)
        if stock:
            with _Stock(model):
                loss = model(input_ids=ids, labels=ids).loss
                loss.backward()
        else:
            loss = model(input_ids=ids, labels=ids).loss
            loss.backward()
        res.append((loss.detach().clone(), {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}))
    assert calls == {"rope": 2, "swiglu": 2}
    (ls, gs), (ln, gn) = res
    _bits_equal(ln.reshape(1), ls.reshape(1), "loss")
    assert set(gs) == set(gn) and len(gs) > 0
    for n in gs:
        _bits_equal(gn[n], gs[n], n)


def _trainer_run(stock, graphed=False, sow_accumulation=3, steps=6):
    """Six steps of a llama_60m SoW trainer (capturable optimizer); graphed: capture step 3 and replay from there."""
    from sow_b200.trainer import SoWTrainer, TrainConfig
    cfg = TrainConfig(model="llama_60m", rank=16, seq_len=128, batch_size=4, lr=1e-2, sow_lr=1e-3,
                      sow_accumulation=sow_accumulation, init_method="normal", seed=1, cuda_graph=True)
    torch.manual_seed(0)
    tr = SoWTrainer(cfg, torch.device(DEV, 0))
    tr.cfg.cuda_graph = graphed
    g = torch.Generator().manual_seed(3)
    losses = []
    ctx = _Stock(tr.model) if stock else None
    if ctx:
        ctx.__enter__()
    try:
        for _ in range(steps):
            ids = torch.randint(1, 32000, (4, 128), generator=g).to(DEV)
            losses.append(tr.step(ids).detach().clone())
        torch.cuda.synchronize()
    finally:
        if ctx:
            ctx.__exit__(None, None, None)
    return tr, losses, {n: p.detach().clone() for n, p in tr.model.named_parameters()}


def _same_run(a, b):
    (_, la, pa), (_, lb, pb) = a, b
    for i, (x, y) in enumerate(zip(la, lb)):
        _bits_equal(y.reshape(1), x.reshape(1), f"loss of step {i}")
    assert set(pa) == set(pb)
    for n in pa:
        _bits_equal(pb[n], pa[n], n)


def test_trainer_parameters_identical_after_six_steps_across_a_merge(monkeypatch):
    calls = _count_native(monkeypatch)
    stock = _trainer_run(stock=True)
    assert calls["rope"] == 0 and calls["swiglu"] == 0
    native = _trainer_run(stock=False)
    assert calls["rope"] > 0 and calls["swiglu"] > 0
    assert stock[0].merges == native[0].merges == 1
    _same_run(stock, native)


def test_cuda_graph_replay_matches_eager_with_native_glue(monkeypatch):
    calls = _count_native(monkeypatch)
    eager = _trainer_run(stock=False, sow_accumulation=100)
    graphed = _trainer_run(stock=False, graphed=True, sow_accumulation=100)
    assert eager[0]._graph is None and graphed[0]._graph is not None
    assert calls["rope"] > 0 and calls["swiglu"] > 0
    _same_run(eager, graphed)


def test_dynamo_traces_the_glued_model_without_graph_breaks(monkeypatch):
    """Under torch.compile the dispatchers run the stock functions (inductor fuses them itself): no graph break, no
    native call."""
    import torch._dynamo
    calls = _count_native(monkeypatch)
    from sow_b200.trainer import build_llama, LLAMA_TARGETS
    from tn_gradient.prepare import SoWConfig, prepare_sow
    model = prepare_sow(build_llama("llama_60m"), SoWConfig(target_modules=LLAMA_TARGETS, rank=8, init_method="normal",
                                                            device=DEV)).to(DEV, torch.bfloat16)
    ids = torch.randint(1, 32000, (2, 64), generator=torch.Generator().manual_seed(0)).to(DEV)
    torch._dynamo.reset()
    ex = torch._dynamo.explain(model)(input_ids=ids)
    assert ex.graph_break_count == 0, ex.break_reasons
    assert calls == {"rope": 0, "swiglu": 0}


def test_fp32_model_takes_the_stock_path(monkeypatch):
    calls = _count_native(monkeypatch)
    from sow_b200.trainer import build_llama, LLAMA_TARGETS
    from tn_gradient.prepare import SoWConfig, prepare_sow
    model = prepare_sow(build_llama("llama_60m"), SoWConfig(target_modules=LLAMA_TARGETS, rank=8, init_method="normal",
                                                            device=DEV)).to(DEV, torch.float32)
    ids = torch.randint(1, 32000, (2, 64), generator=torch.Generator().manual_seed(0)).to(DEV)
    model(input_ids=ids, labels=ids).loss.backward()
    assert calls == {"rope": 0, "swiglu": 0}
