"""CPU: installation of the native LlamaRMSNorm and the argument checks of its C ABI.  On CPU tensors, and under
torch.compile, the stock forward runs."""
import ctypes

import torch

from conftest import ROOT  # noqa: F401  (puts the repository on sys.path)


def _tiny_llama(seed=0):
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(vocab_size=128, hidden_size=128, intermediate_size=96, num_hidden_layers=2, num_attention_heads=4,
                      max_position_embeddings=64, rms_norm_eps=1e-6, hidden_act="silu", use_cache=False,
                      tie_word_embeddings=False)
    torch.manual_seed(seed)
    return LlamaForCausalLM(cfg)


def test_every_norm_gets_the_native_forward_once():
    from transformers.models.llama import modeling_llama as ml
    from sow_b200 import llama_glue
    model = _tiny_llama()
    llama_glue.install_llama_glue(model)
    norms = [m for m in model.modules() if isinstance(m, ml.LlamaRMSNorm)]
    assert len(norms) == 5
    for m in norms:
        assert m.forward.__func__ is llama_glue._llama_rmsnorm_forward and m.forward.__self__ is m
    before = [m.__dict__["forward"] for m in norms]
    llama_glue.install_llama_glue(model)
    assert [m.__dict__["forward"] for m in norms] == before
    assert ml.LlamaRMSNorm.forward is not llama_glue._llama_rmsnorm_forward     # the class itself stays stock


def test_subclasses_with_their_own_forward_are_left_alone():
    from transformers.models.llama import modeling_llama as ml
    from sow_b200 import llama_glue

    class Other(ml.LlamaRMSNorm):
        def forward(self, h):
            return h

    wrap = torch.nn.Sequential(Other(128))
    llama_glue.install_llama_glue(wrap)
    assert "forward" not in wrap[0].__dict__


def test_cpu_norm_takes_the_stock_path_and_matches_it():
    from transformers.models.llama import modeling_llama as ml
    from sow_b200 import llama_glue
    model = _tiny_llama()
    llama_glue.install_llama_glue(model)
    m = model.model.norm
    for dt in (torch.float32, torch.bfloat16):
        m.to(dt)
        x = torch.randn(4, 16, 128, generator=torch.Generator().manual_seed(1)).to(dt)
        assert not llama_glue.rmsnorm_native_ok(x, m.weight, m.variance_epsilon)
        assert torch.equal(m(x), ml.LlamaRMSNorm.forward(m, x))


def test_native_ok_rejects_what_the_kernels_do_not_compute():
    from sow_b200.llama_glue import rmsnorm_native_ok
    w = torch.ones(1024, dtype=torch.bfloat16)
    x = torch.zeros(64, 1024, dtype=torch.bfloat16)
    assert not rmsnorm_native_ok(x, w, 1e-6)                                       # CPU
    assert not rmsnorm_native_ok(x.float(), w.float(), 1e-6)


def test_norm_traces_without_graph_breaks():
    import torch._dynamo
    from sow_b200 import llama_glue
    model = _tiny_llama()
    llama_glue.install_llama_glue(model)
    ids = torch.randint(0, 128, (2, 16), generator=torch.Generator().manual_seed(0))
    torch._dynamo.reset()
    ex = torch._dynamo.explain(model)(input_ids=ids)
    assert ex.graph_break_count == 0, ex.break_reasons


def test_rmsnorm_entry_points_reject_bad_arguments_before_any_work():
    """Width / row count / dtype / alignment errors come back as SOWB_EINVAL from host checks (the fake pointers are
    never touched)."""
    from sow_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(1 << 20)
    odd = ctypes.c_void_p((1 << 20) + 8)
    bf16 = _lib.SOWB_BF16
    fwd = lambda rows, width, dtype=bf16, x=p: lib.sow_rmsnorm_fwd(x, p, p, p, rows, width, 1e-6, dtype, None)
    bwd = lambda rows, width, dtype=bf16, pp=p: lib.sow_rmsnorm_bwd(p, p, p, p, p, pp, rows, width, dtype, None)
    for fn in (fwd, bwd):
        assert fn(64, 1000) == -1                      # no kernel for this width
        assert fn(64, 1024, _lib.SOWB_F32) == -1       # fp32 is not a glue dtype
        assert fn(15, 1024) == -1                      # torch sums fewer than 16 rows in another order
        assert fn(-1, 1024) == -1
        assert b"sow_rmsnorm" in lib.sow_last_error()
    assert fwd(64, 1024, x=odd) == -1                  # misaligned
    assert bwd(64, 1024, pp=odd) == -1
    assert lib.sow_rmsnorm_fwd(None, p, p, p, 64, 1024, 1e-6, bf16, None) == -1
    assert lib.sow_rmsnorm_bwd(p, p, p, p, None, None, 64, 1024, bf16, None) == -1
    # empty tensors are a no-op; H = 128 has torch's order at any row count
    assert fwd(0, 1024) == 0 and bwd(0, 1024, pp=None) == 0
    assert fwd(0, 128) == 0
