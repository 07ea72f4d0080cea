"""CPU: installation of the native Llama glue (rotary embedding, SwiGLU) and its argument checks.  On CPU tensors, and
under torch.compile, the stock HF functions run."""
import ctypes

import pytest
import torch

from conftest import ROOT  # noqa: F401  (puts the repository on sys.path)


def _tiny_llama(seed=0):
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(vocab_size=128, hidden_size=64, intermediate_size=96, num_hidden_layers=2, num_attention_heads=4,
                      max_position_embeddings=64, rms_norm_eps=1e-6, hidden_act="silu", use_cache=False,
                      tie_word_embeddings=False)
    torch.manual_seed(seed)
    return LlamaForCausalLM(cfg)


def _prepared(seed=0):
    from tn_gradient.prepare import SoWConfig, prepare_sow
    return prepare_sow(_tiny_llama(seed), SoWConfig(target_modules=["q_proj", "k_proj", "v_proj", "o_proj", "gate_proj",
                                                                    "up_proj", "down_proj"], rank=4, init_method="normal"))


def test_prepare_sow_installs_the_glue_once():
    from transformers.models.llama import modeling_llama as ml
    from sow_b200 import llama_glue
    model = _prepared()
    mlps = [m for m in model.modules() if isinstance(m, ml.LlamaMLP)]
    assert len(mlps) == 2
    for m in mlps:
        assert m.forward.__func__ is llama_glue._llama_mlp_forward and m.forward.__self__ is m
    disp = ml.apply_rotary_pos_emb
    stock = disp.stock
    assert getattr(stock, "stock", None) is None          # the dispatcher wraps the stock function, not itself
    # installing again (same model, or another one) changes nothing
    assert llama_glue.install_llama_glue(model) == 0
    assert llama_glue.install_rope(ml) is False
    _prepared(1)
    assert ml.apply_rotary_pos_emb is disp and disp.stock is stock


def _glued(seed=0):
    """A plain HF Llama with the glue installed (SoW layers themselves run on CUDA only)."""
    from sow_b200.llama_glue import install_llama_glue
    model = _tiny_llama(seed)
    assert install_llama_glue(model) == 2
    return model


def test_cpu_model_takes_the_stock_path_and_matches_it():
    """On CPU the dispatchers run the stock functions: loss and gradients equal those of the unpatched model."""
    from transformers.models.llama import modeling_llama as ml
    ids = torch.randint(0, 128, (2, 16), generator=torch.Generator().manual_seed(0))
    model = _glued()
    loss = model(input_ids=ids, labels=ids).loss
    loss.backward()
    grads = {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}
    model.zero_grad(set_to_none=True)
    disp = ml.apply_rotary_pos_emb
    try:
        ml.apply_rotary_pos_emb = disp.stock
        for m in model.modules():
            m.__dict__.pop("forward", None)
        loss2 = model(input_ids=ids, labels=ids).loss
        loss2.backward()
    finally:
        ml.apply_rotary_pos_emb = disp
    assert torch.equal(loss, loss2)
    for n, p in model.named_parameters():
        if n in grads:
            assert torch.equal(grads[n], p.grad), n


def test_dispatchers_trace_without_graph_breaks():
    import torch._dynamo
    model = _glued()
    ids = torch.randint(0, 128, (2, 16), generator=torch.Generator().manual_seed(0))
    torch._dynamo.reset()
    ex = torch._dynamo.explain(model)(input_ids=ids)
    assert ex.graph_break_count == 0, ex.break_reasons


def test_glue_entry_points_reject_bad_arguments_before_any_work():
    """Shape / dtype / alignment errors come back as SOWB_EINVAL from host checks (the fake pointers are never touched)."""
    from sow_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(1 << 20)
    ok_strides = (16 * 8 * 64, 64, 16 * 64)
    args = lambda D, dtype, strides=ok_strides, ptr=p: (ptr, ptr, ptr, ptr, ptr, ptr, 2, 8, 16, 16, D, *strides, *strides,
                                                        0, dtype, None)
    for fn in (lib.sow_rope_fwd, lib.sow_rope_bwd):
        assert fn(*args(24, _lib.SOWB_BF16)) == -1                       # D not a multiple of 16
        assert fn(*args(64, _lib.SOWB_F32)) == -1                        # fp32 is not a glue dtype
        assert fn(*args(64, _lib.SOWB_BF16, (100, 64, 1028))) == -1      # stride not a multiple of 8
        assert fn(*args(64, _lib.SOWB_BF16, ptr=ctypes.c_void_p((1 << 20) + 2))) == -1   # misaligned
        assert b"sow_rope" in lib.sow_last_error()
    assert lib.sow_swiglu_fwd(p, p, p, 1000, _lib.SOWB_F32, None) == -1
    assert lib.sow_swiglu_fwd(p, p, ctypes.c_void_p((1 << 20) + 8), 1000, _lib.SOWB_BF16, None) == -1
    assert lib.sow_swiglu_bwd(p, p, p, p, None, 1000, _lib.SOWB_F16, None) == -1
    assert lib.sow_swiglu_bwd(p, p, p, p, p, -1, _lib.SOWB_F16, None) == -1
    # empty tensors are a no-op
    assert lib.sow_swiglu_fwd(p, p, p, 0, _lib.SOWB_BF16, None) == 0


def test_ops_refuse_cpu_tensors():
    from sow_b200 import ops
    from sow_b200._lib import SowB200Error
    x = torch.zeros(2, 4, 8, 64, dtype=torch.bfloat16)
    cs = torch.zeros(1, 8, 64, dtype=torch.bfloat16)
    with pytest.raises(SowB200Error, match="no CPU fallback"):
        ops.rope_fwd(x, x, cs, cs)
    with pytest.raises(SowB200Error, match="no CPU fallback"):
        ops.swiglu_fwd(x, x)
