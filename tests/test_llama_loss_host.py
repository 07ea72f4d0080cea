"""CPU: installation and dispatch of the native causal-LM loss, its label handling, and the argument checks of its C ABI.
On CPU tensors, for fp32 logits and under torch.compile the stock ForCausalLMLoss runs."""
import ctypes

import pytest
import torch

from conftest import ROOT  # noqa: F401  (puts the repository on sys.path)

V = 32000


def _tiny_llama(vocab=128, seed=0):
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(vocab_size=vocab, hidden_size=128, intermediate_size=96, num_hidden_layers=2, num_attention_heads=4,
                      max_position_embeddings=64, rms_norm_eps=1e-6, hidden_act="silu", use_cache=False,
                      tie_word_embeddings=False)
    torch.manual_seed(seed)
    return LlamaForCausalLM(cfg)


def test_the_loss_is_installed_once_and_keeps_the_stock_function():
    from transformers.loss.loss_utils import ForCausalLMLoss
    from sow_b200 import llama_glue
    model = _tiny_llama()
    assert model.loss_function is ForCausalLMLoss
    llama_glue.install_llama_glue(model)
    fn = model.loss_function
    assert isinstance(fn, llama_glue.CausalLMLoss) and fn.stock is ForCausalLMLoss
    llama_glue.install_llama_glue(model)
    assert model.loss_function is fn
    assert _tiny_llama().loss_function is ForCausalLMLoss          # other instances stay stock


def test_a_custom_loss_function_is_left_alone():
    from sow_b200 import llama_glue
    model = _tiny_llama()
    custom = lambda logits, labels, vocab_size, **kw: logits.sum()    # noqa: E731
    model.loss_function = custom
    llama_glue.install_llama_glue(model)
    assert model.loss_function is custom


def test_cpu_loss_takes_the_stock_path_and_matches_it():
    from transformers.loss.loss_utils import ForCausalLMLoss
    from sow_b200 import llama_glue
    model = _tiny_llama()
    llama_glue.install_llama_glue(model)
    ids = torch.randint(0, 128, (2, 16), generator=torch.Generator().manual_seed(1))
    ref = _tiny_llama()
    assert torch.equal(model(input_ids=ids, labels=ids).loss, ref(input_ids=ids, labels=ids).loss)
    assert model.loss_function.stock is ForCausalLMLoss


def test_native_ok_rejects_what_the_kernels_do_not_compute():
    from sow_b200.llama_glue import loss_native_ok
    logits = torch.zeros(2, 8, V, dtype=torch.bfloat16)
    labels = torch.zeros(2, 8, dtype=torch.int64)
    assert not loss_native_ok(logits, labels, V)                                   # CPU
    assert not loss_native_ok(logits.float(), labels, V)


def _emulated(monkeypatch):
    """Let the dispatcher take its native branch on CPU, with the gather computed by torch: what is left to check is
    the label handling and the NLL reduction around it."""
    from sow_b200 import llama_glue

    class Gather:
        @staticmethod
        def apply(logits, targets):
            lp = torch.log_softmax(logits.float(), -1)
            ok = (targets >= 0) & (targets < logits.shape[-1])
            return torch.where(ok, lp.gather(1, torch.where(ok, targets, 0)[:, None])[:, 0], 0.0)[:, None]
    monkeypatch.setattr(llama_glue, "_CausalLMLoss", Gather)
    monkeypatch.setattr(llama_glue, "loss_native_ok", lambda *a, **k: True)


def test_label_shift_ignore_index_and_num_items_match_the_stock_loss(monkeypatch):
    from transformers.loss.loss_utils import ForCausalLMLoss
    from sow_b200.llama_glue import CausalLMLoss
    _emulated(monkeypatch)
    gen = torch.Generator().manual_seed(3)
    logits = torch.randn(3, 10, 50, generator=gen).to(torch.bfloat16)
    labels = torch.randint(0, 50, (3, 10), generator=gen)
    labels[0, 4] = labels[2, 0] = -100
    native = CausalLMLoss(ForCausalLMLoss)
    shift = torch.randint(0, 50, (3, 10), generator=gen)
    shift[1, 1] = -100
    cases = [(labels, {}), (labels, {"num_items_in_batch": 11}), (labels, {"num_items_in_batch": torch.tensor(11)}),
             (labels, {"shift_labels": shift}), (labels, {"shift_labels": torch.where(shift < 0, -7, shift), "ignore_index": -7}),
             (torch.where(labels < 0, -5, labels), {"ignore_index": -5})]
    for lab, kw in cases:
        a = native(logits=logits, labels=lab, vocab_size=50, **kw)
        b = ForCausalLMLoss(logits=logits, labels=lab, vocab_size=50, **kw)
        torch.testing.assert_close(a, b, rtol=1e-6, atol=0, msg=str(kw))
    # a label that is neither in range nor ignore_index is rejected by nll_loss on both paths
    bad = labels.clone()
    bad[1, 3] = 50
    for fn in (native, ForCausalLMLoss):
        with pytest.raises(IndexError):
            fn(logits=logits, labels=bad, vocab_size=50)


def test_the_knob_selects_the_stock_loss(monkeypatch):
    from sow_b200 import llama_glue
    _emulated(monkeypatch)
    seen = []
    native = llama_glue.CausalLMLoss(lambda *a, **k: seen.append(k) or torch.tensor(0.0))
    logits, labels = torch.zeros(1, 4, 50), torch.zeros(1, 4, dtype=torch.int64)
    native(logits=logits, labels=labels, vocab_size=50)
    assert seen == []
    monkeypatch.setenv("SOWB_NATIVE_LOSS", "0")
    native(logits=logits, labels=labels, vocab_size=50, num_items_in_batch=3)
    assert seen == [{"num_items_in_batch": 3, "ignore_index": -100, "shift_labels": None}]


def test_loss_traces_without_graph_breaks():
    import torch._dynamo
    from sow_b200 import llama_glue
    model = _tiny_llama()
    llama_glue.install_llama_glue(model)
    ids = torch.randint(0, 128, (2, 16), generator=torch.Generator().manual_seed(0))
    torch._dynamo.reset()
    ex = torch._dynamo.explain(model)(input_ids=ids, labels=ids)
    assert ex.graph_break_count == 0, ex.break_reasons


@pytest.mark.parametrize("fn", ["sow_ce_fwd", "sow_ce_bwd"])
def test_loss_entry_points_reject_bad_arguments_before_any_work(fn):
    """Vocabulary / row count / dtype / alignment errors come back as SOWB_EINVAL from host checks (the fake pointers
    are never touched)."""
    from sow_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(1 << 20)
    odd = ctypes.c_void_p((1 << 20) + 8)
    bf16 = _lib.SOWB_BF16

    def call(rows, vocab, dtype=bf16, logits=p, last=p):
        if fn == "sow_ce_fwd":
            return lib.sow_ce_fwd(logits, p, p, p, last, rows, vocab, dtype, None)
        return lib.sow_ce_bwd(logits, p, p, p, p, last, rows, vocab, dtype, None)
    assert call(64, 32001) == -1                 # not a multiple of 8
    assert call(64, 12288) == -1                 # torch reduces narrower rows in another order
    assert call(64, 32776) == -1                 # a row no longer fits the registers
    assert call(64, V, _lib.SOWB_F32) == -1      # fp32 logits are not a glue dtype
    assert call(-1, V) == -1
    assert call(64, V, logits=odd) == -1         # misaligned
    assert call(64, V, last=None) == -1
    assert fn.encode() in lib.sow_last_error()
    assert call(0, V) == 0                       # empty: a no-op
