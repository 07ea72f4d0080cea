"""GPU: the native causal-LM cross-entropy (csrc/glue.cu ce_fwd_kernel / ce_bwd_kernel behind llama_glue.CausalLMLoss)
against HF's stock ForCausalLMLoss, bit for bit: the loss and the bf16 / fp16 gradient of the logits.

Every comparison goes through an integer view, so signed zeros and inf count too; NaN matches NaN (where stock gives
NaN, so must the native path)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
V = 32000
HALF = [torch.bfloat16, torch.float16]
HALF_IDS = ["bf16", "fp16"]


def _same(a, b, what):
    assert a.shape == b.shape and a.dtype == b.dtype, (what, a.shape, b.shape, a.dtype, b.dtype)
    it = {2: torch.int16, 4: torch.int32}[a.element_size()]
    nan = torch.isnan(a)
    assert torch.equal(nan, torch.isnan(b)), f"{what}: NaN patterns differ"
    ai, bi = a.contiguous().view(it), b.contiguous().view(it)
    bad = ((ai != bi) & ~nan).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.shape[0]} elements differ, first at {bad[0].tolist()}: " \
                             f"{a[tuple(bad[0])].item()} vs {b[tuple(bad[0])].item()}"


def _both(logits, labels, grad_out=1.0, **kw):
    """(loss, logits.grad) of the stock ForCausalLMLoss and of the native dispatcher on the same inputs."""
    from transformers.loss.loss_utils import ForCausalLMLoss
    from sow_b200.llama_glue import CausalLMLoss, loss_native_ok
    vocab = logits.shape[-1]
    lab = kw.get("shift_labels", labels)
    assert loss_native_ok(logits, lab, vocab, kw.get("ignore_index", -100), shifted="shift_labels" in kw)
    out = []
    for fn in (ForCausalLMLoss, CausalLMLoss(ForCausalLMLoss)):
        lg = logits.detach().clone().requires_grad_(True)
        loss = fn(logits=lg, labels=labels, vocab_size=vocab, **kw)
        (g,) = torch.autograd.grad(loss, lg, torch.tensor(grad_out, device=DEV))
        out.append((loss.detach(), g))
    return out


def _check(logits, labels, grad_out=1.0, **kw):
    (ls, gs), (ln, gn) = _both(logits, labels, grad_out, **kw)
    _same(ln, ls, "loss")
    _same(gn, gs, "logits.grad")
    return ls


def _labels(shape, gen, vocab=V, ignored=0.1):
    lab = torch.randint(0, vocab, shape, device=DEV, generator=gen)
    return torch.where(torch.rand(shape, device=DEV, generator=gen) < ignored, -100, lab)


@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_loss_matches_stock_at_the_bench_shape(dt):
    gen = torch.Generator(device=DEV).manual_seed(1)
    logits = (torch.randn(128, 256, V, device=DEV, generator=gen) * 3).to(dt)
    labels = _labels((128, 256), gen)
    loss = _check(logits, labels)
    assert torch.isfinite(loss)


@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("rows", [1, 7, 300])
@pytest.mark.parametrize("scale", [1e-2, 1.0, 30.0])
def test_loss_matches_stock_at_small_row_counts(rows, scale, dt):
    gen = torch.Generator(device=DEV).manual_seed(rows * 3 + int(scale))
    logits = (torch.randn(1, rows, V, device=DEV, generator=gen) * scale).to(dt)
    labels = _labels((1, rows), gen, ignored=0.2)
    labels[0, 0] = 0
    for go in (1.0, 1.0 / 3.0, 2.0 ** 16):
        _check(logits, labels, go)


@pytest.mark.parametrize("vocab", [16384, 24008, 32768])
def test_loss_matches_stock_at_other_vocabulary_sizes(vocab):
    gen = torch.Generator(device=DEV).manual_seed(vocab)
    logits = (torch.randn(3, 40, vocab, device=DEV, generator=gen) * 4).to(torch.bfloat16)
    labels = _labels((3, 40), gen, vocab)
    labels[0, 1], labels[1, 2] = 0, vocab - 1
    _check(logits, labels)
    _check(logits, labels, 0.25, num_items_in_batch=50)


@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_loss_edge_rows(dt):
    """Targets at 0 and V - 1, constant rows, the max first and last, -inf entries, rows of +inf and NaN results."""
    gen = torch.Generator(device=DEV).manual_seed(7)
    logits = torch.randn(1, 64, V, device=DEV, generator=gen).to(dt)
    labels = _labels((1, 64), gen, ignored=0.0)
    labels[0, :8] = 0
    labels[0, 8:16] = V - 1
    logits[0, 1] = 0.0                              # constant rows
    logits[0, 2] = 5.0
    logits[0, 3, 0] = 20.0                          # max first, at the target (0)
    logits[0, 9, V - 1] = 20.0                      # max last, at the target (V - 1)
    logits[0, 4, V - 1] = 20.0                      # max last, target elsewhere
    logits[0, 20, ::3] = float("-inf")
    logits[0, 21, 17] = float("-inf")
    _check(logits, labels)
    logits[0, 30, 5] = float("inf")                 # a row of NaN log-probabilities: NaN loss and NaN gradient rows
    logits[0, 31] = float("-inf")
    _check(logits, labels)


@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_ignored_labels_and_num_items_in_batch(dt):
    gen = torch.Generator(device=DEV).manual_seed(9)
    logits = (torch.randn(4, 100, V, device=DEV, generator=gen) * 2).to(dt)
    labels = _labels((4, 100), gen, ignored=0.5)
    _check(logits, labels)
    _check(logits, labels, 1.0 / 3.0, num_items_in_batch=torch.tensor(123, device=DEV))
    _check(logits, labels, 2.0 ** 16, num_items_in_batch=77)
    shift = _labels((4, 100), gen, ignored=0.3)
    _check(logits, labels, 1.0, shift_labels=shift)
    _check(logits, labels, 1.0, ignore_index=-1, shift_labels=torch.where(shift < 0, -1, shift))
    # every label ignored: a NaN mean (0 / 0) and an all-zero gradient, as stock
    ls = _check(logits, torch.full_like(labels, -100))
    assert torch.isnan(ls)
    _check(logits, torch.full_like(labels, -100), 1.0, num_items_in_batch=5)


def test_loss_under_cuda_graph_capture():
    from transformers.loss.loss_utils import ForCausalLMLoss
    from sow_b200.llama_glue import CausalLMLoss
    gen = torch.Generator(device=DEV).manual_seed(6)
    logits = (torch.randn(2, 128, V, device=DEV, generator=gen) * 3).to(torch.bfloat16).requires_grad_(True)
    labels = _labels((2, 128), gen)
    native = CausalLMLoss(ForCausalLMLoss)

    def run():
        loss = native(logits=logits, labels=labels, vocab_size=V)
        # detached: no autograd node made outside the capture (and its stream) outlives this call
        return [t.detach() for t in (loss,) + torch.autograd.grad(loss, logits)]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ref = [t.clone() for t in run()]
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = run()
    with torch.no_grad():
        logits.copy_((torch.randn(logits.shape, device=DEV, generator=gen) * 3).to(torch.bfloat16))
        labels.copy_(_labels((2, 128), gen))
    g.replay()
    torch.cuda.synchronize()
    ls, gs = _both(logits, labels)[0]       # the stock loss on the new inputs
    _same(outs[0], ls, "graphed loss")
    _same(outs[1], gs, "graphed logits.grad")
    assert not torch.equal(outs[0], ref[0])


def _count_loss(monkeypatch):
    from sow_b200 import ops
    calls = {"fwd": 0, "bwd": 0}
    f, b = ops.ce_fwd, ops.ce_bwd

    def fwd(*a, **k):
        calls["fwd"] += 1
        return f(*a, **k)

    def bwd(*a, **k):
        calls["bwd"] += 1
        return b(*a, **k)
    monkeypatch.setattr(ops, "ce_fwd", fwd)
    monkeypatch.setattr(ops, "ce_bwd", bwd)
    return calls


def test_the_bench_model_loss_runs_native(monkeypatch):
    from sow_b200.trainer import SoWTrainer, TrainConfig
    calls = _count_loss(monkeypatch)
    tr = SoWTrainer(TrainConfig(batch_size=2), torch.device(DEV, 0))
    ids = torch.randint(1, 32000, (2, 256), generator=torch.Generator().manual_seed(0)).to(DEV)
    tr.step(ids)
    assert calls == {"fwd": 1, "bwd": 1}
    monkeypatch.setenv("SOWB_NATIVE_LOSS", "0")
    tr.step(ids)
    assert calls == {"fwd": 1, "bwd": 1}


def test_fp32_and_compiled_models_make_no_native_loss_call(monkeypatch):
    import torch._dynamo
    from sow_b200.trainer import build_llama, LLAMA_TARGETS
    from tn_gradient.prepare import SoWConfig, prepare_sow
    calls = _count_loss(monkeypatch)
    ids = torch.randint(1, 32000, (2, 64), generator=torch.Generator().manual_seed(0)).to(DEV)
    model = prepare_sow(build_llama("llama_60m"), SoWConfig(target_modules=LLAMA_TARGETS, rank=8, init_method="normal",
                                                            device=DEV))
    model.to(DEV, torch.float32)(input_ids=ids, labels=ids).loss.backward()
    assert calls == {"fwd": 0, "bwd": 0}
    model.to(DEV, torch.bfloat16)
    torch._dynamo.reset()
    torch._dynamo.explain(model)(input_ids=ids, labels=ids)
    assert calls == {"fwd": 0, "bwd": 0}
