"""Native rotary embedding and SwiGLU for HF Llama blocks on the eager training path.

Eager HF code runs ``q * cos + rotate_half(q) * sin`` (for q and k) and ``act_fn(gate) * up`` as about a dozen element-wise
kernels per layer on strided views, with zero-filled slice-backward buffers in the backward pass.  The kernels of
``csrc/glue.cu`` do each chain in one pass per direction and reproduce eager's rounding sequence exactly, so the results
are bit-identical to the stock functions (and a training run is unchanged bit for bit).

``install_llama_glue(model)`` (called by ``prepare_sow``) routes a model's Llama blocks through them:
  * SwiGLU: every ``LlamaMLP`` with a silu activation gets a per-instance ``forward`` that calls ``gate_proj(x)`` then
    ``up_proj(x)`` (the order eager uses, which the shared-input SoW group relies on) and the fused gate.
  * RoPE: HF's attention looks ``apply_rotary_pos_emb`` up in the ``modeling_llama`` module globals; that global is
    replaced by a dispatcher that keeps the stock function.  Installing twice changes nothing.
  * RMSNorm: every ``LlamaRMSNorm`` gets a per-instance ``forward``.
  * Loss: every ``LlamaForCausalLM`` whose ``loss_function`` is HF's ``ForCausalLMLoss`` gets ``CausalLMLoss`` (which
    keeps the stock function as ``.stock``) through the ``loss_function`` setter.
The native path runs only for CUDA bf16 / fp16 tensors of the expected layouts, cos / sin without grad,
``unsqueeze_dim == 1``, and outside ``torch.compile`` tracing; every other call runs the stock function, so compiled
models (inductor fuses these chains itself) and fp32 models are exactly as before.
"""
from __future__ import annotations

import os
import types

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops

_HALF = (torch.bfloat16, torch.float16)


# ---- rotary embedding ----------------------------------------------------------------------------------------------

class _RoPE(torch.autograd.Function):
    """(q, k, cos, sin) -> (q * cos + rotate_half(q) * sin, the same for k).  Saves only cos / sin, as eager does."""

    @staticmethod
    def forward(ctx, q, k, cos, sin):
        ctx.save_for_backward(cos, sin)
        return ops.rope_fwd(q, k, cos, sin)

    @staticmethod
    def backward(ctx, gq, gk):
        cos, sin = ctx.saved_tensors
        dq, dk = ops.rope_bwd(gq, gk, cos, sin)
        return dq, dk, None, None


def _aligned_rows(t: torch.Tensor) -> bool:
    return t.stride(-1) == 1 and t.data_ptr() % 16 == 0 and all(s % 8 == 0 for s in t.stride()[:-1])


def rope_native_ok(q, k, cos, sin, unsqueeze_dim=1) -> bool:
    """True when the native kernel computes apply_rotary_pos_emb(q, k, cos, sin, unsqueeze_dim) for these arguments."""
    if unsqueeze_dim != 1 or not all(isinstance(t, torch.Tensor) for t in (q, k, cos, sin)):
        return False
    if not q.is_cuda or q.dtype not in _HALF or not (k.dtype == cos.dtype == sin.dtype == q.dtype):
        return False
    if not (k.device == cos.device == sin.device == q.device) or cos.requires_grad or sin.requires_grad:
        return False
    if q.dim() != 4 or k.dim() != 4 or cos.dim() != 3:
        return False
    B, _, S, D = q.shape
    if D % 16 or k.shape[0] != B or tuple(k.shape[2:]) != (S, D):
        return False
    if cos.shape != sin.shape or tuple(cos.shape) not in ((1, S, D), (B, S, D)):
        return False
    if not (cos.is_contiguous() and sin.is_contiguous() and cos.data_ptr() % 16 == 0 and sin.data_ptr() % 16 == 0):
        return False
    return _aligned_rows(q) and _aligned_rows(k)


def make_rope_dispatcher(stock):
    """apply_rotary_pos_emb with HF's signature: the native kernel where rope_native_ok holds, ``stock`` otherwise."""

    def apply_rotary_pos_emb(q, k, cos, sin, unsqueeze_dim=1):
        if not torch.compiler.is_compiling() and rope_native_ok(q, k, cos, sin, unsqueeze_dim):
            return _RoPE.apply(q, k, cos, sin)
        return stock(q, k, cos, sin, unsqueeze_dim)

    apply_rotary_pos_emb.__doc__ = getattr(stock, "__doc__", None)
    apply_rotary_pos_emb.stock = stock
    return apply_rotary_pos_emb


def install_rope(modeling_module) -> bool:
    """Replace ``modeling_module.apply_rotary_pos_emb`` by the dispatcher (once).  Returns True if it was installed now."""
    cur = modeling_module.apply_rotary_pos_emb
    if getattr(cur, "stock", None) is not None:
        return False
    modeling_module.apply_rotary_pos_emb = make_rope_dispatcher(cur)
    return True


# ---- SwiGLU ----------------------------------------------------------------------------------------------------------

class _SwiGLU(torch.autograd.Function):
    """(gate, up) -> silu(gate) * up.  Saves gate and up; eager also keeps silu(gate), one more activation per layer."""

    @staticmethod
    def forward(ctx, gate, up):
        ctx.save_for_backward(gate, up)
        return ops.swiglu_fwd(gate, up)

    @staticmethod
    def backward(ctx, dh):
        gate, up = ctx.saved_tensors
        return ops.swiglu_bwd(dh, gate, up)


def swiglu_native_ok(gate, up) -> bool:
    return (isinstance(gate, torch.Tensor) and isinstance(up, torch.Tensor) and gate.is_cuda and gate.dtype in _HALF
            and up.dtype == gate.dtype and up.device == gate.device and gate.shape == up.shape
            and gate.is_contiguous() and up.is_contiguous() and gate.data_ptr() % 16 == 0 and up.data_ptr() % 16 == 0)


def _is_silu(act) -> bool:
    try:
        from transformers.activations import SiLUActivation
    except Exception:  # pragma: no cover - older transformers
        SiLUActivation = ()
    return isinstance(act, SiLUActivation) or (isinstance(act, nn.SiLU) and not act.inplace)


def _llama_mlp_forward(self, x):
    """LlamaMLP.forward with the silu gate fused: down_proj(silu(gate_proj(x)) * up_proj(x))."""
    if torch.compiler.is_compiling():
        return type(self).forward(self, x)
    gate = self.gate_proj(x)
    up = self.up_proj(x)
    h = _SwiGLU.apply(gate, up) if swiglu_native_ok(gate, up) else self.act_fn(gate) * up
    return self.down_proj(h)


# ---- RMSNorm ---------------------------------------------------------------------------------------------------------

_NORM_WIDTHS = (128, 256, 512, 768, 1024, 2048, 3072, 4096)   # the widths csrc/glue.cu has kernels for


def _stock_rmsnorm(x, w, eps):
    """LlamaRMSNorm.forward, op for op."""
    h = x.to(torch.float32)
    h = h * torch.rsqrt(h.pow(2).mean(-1, keepdim=True) + eps)
    return w * h.to(x.dtype)


class _RMSNorm(torch.autograd.Function):
    """(x, w) -> w * (x * rsqrt(mean(x^2) + eps)) in one pass each way.  Saves x, w and one fp32 value per row, where
    eager saves several fp32 copies of x."""

    @staticmethod
    def forward(ctx, x, w, eps):
        y, rs = ops.rmsnorm_fwd(x, w, eps)
        ctx.save_for_backward(x, w, rs)
        ctx.eps = eps
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, rs = ctx.saved_tensors
        want_w = ctx.needs_input_grad[1]
        if not (dy.is_contiguous() and dy.data_ptr() % 16 == 0):
            # eager's row sums follow the layout of dy: replay the stock chain for such a gradient
            with torch.enable_grad():
                xd, wd = x.detach().requires_grad_(True), w.detach().requires_grad_(want_w)
                ins = (xd, wd) if want_w else (xd,)
                gs = torch.autograd.grad(_stock_rmsnorm(xd, wd, ctx.eps), ins, dy)
            return gs[0], gs[1] if want_w else None, None
        dx, p = ops.rmsnorm_bwd(dy, x, w, rs, want_p=want_w)
        # dw as eager's engine forms it: torch's own reduction of the bf16 / fp16 product over the leading dims
        return dx, p.sum_to_size(w.shape) if want_w else None, None


def rmsnorm_native_ok(x, w, eps) -> bool:
    """True when the native kernels compute LlamaRMSNorm (weight w, epsilon eps) of x bit for bit."""
    if not (isinstance(x, torch.Tensor) and isinstance(w, torch.Tensor) and isinstance(eps, (float, int))):
        return False
    if not x.is_cuda or x.dtype not in _HALF or w.dtype != x.dtype or w.device != x.device or w.dim() != 1:
        return False
    H = x.shape[-1] if x.dim() else 0
    if H not in _NORM_WIDTHS or w.shape[0] != H or not (x.is_contiguous() and w.is_contiguous()):
        return False
    rows = x.numel() // H
    # below 16 rows torch's row sums take another order (except at H = 128, where the order is the same)
    return (rows >= 16 or H == 128) and x.data_ptr() % 16 == 0 and w.data_ptr() % 16 == 0


def _llama_rmsnorm_forward(self, hidden_states):
    """LlamaRMSNorm.forward through the native kernels where rmsnorm_native_ok holds."""
    if not torch.compiler.is_compiling() and rmsnorm_native_ok(hidden_states, self.weight, self.variance_epsilon):
        return _RMSNorm.apply(hidden_states, self.weight, self.variance_epsilon)
    return type(self).forward(self, hidden_states)


# ---- causal-LM loss --------------------------------------------------------------------------------------------------

_LOSS_VOCAB = (16384, 32768)   # widths (multiples of 8) whose torch log_softmax sums in ce_fwd_kernel's order (glue.cu)


class _CausalLMLoss(torch.autograd.Function):
    """(logits (N, V) bf16 / fp16, targets (N,) int64) -> logp_t (N, 1) fp32, log_softmax(logits.float()) at each row's
    target.  Saves the logits and two fp32 values per row, where eager keeps an fp32 copy of the logits and their fp32
    log_softmax."""

    @staticmethod
    def forward(ctx, logits, targets):
        row_max, row_logsum, logp_t = ops.ce_fwd(logits, targets)
        ctx.save_for_backward(logits, targets, row_max, row_logsum)
        return logp_t.unsqueeze(1)

    @staticmethod
    def backward(ctx, g):
        logits, targets, row_max, row_logsum = ctx.saved_tensors
        return ops.ce_bwd(logits, row_max, row_logsum, targets, g[:, 0]), None


def loss_native_ok(logits, labels, vocab_size, ignore_index=-100, shifted=False) -> bool:
    """True when the native kernels compute ForCausalLMLoss(logits, labels, vocab_size, ignore_index=ignore_index) bit
    for bit (``shifted``: labels are the already shifted ``shift_labels``)."""
    if not (isinstance(logits, torch.Tensor) and isinstance(labels, torch.Tensor) and isinstance(vocab_size, int)
            and isinstance(ignore_index, int)):
        return False
    if not logits.is_cuda or logits.dtype not in _HALF or labels.dtype != torch.int64 or logits.dim() < 2:
        return False
    V = logits.shape[-1]
    if V != vocab_size or V % 8 or not _LOSS_VOCAB[0] <= V <= _LOSS_VOCAB[1] or 0 <= ignore_index < V:
        return False
    if labels.numel() != logits.numel() // V or (not shifted and labels.shape != logits.shape[:-1]):
        return False
    return logits.is_contiguous() and logits.data_ptr() % 16 == 0


class CausalLMLoss:
    """ForCausalLMLoss with HF's signature: the native kernels where loss_native_ok holds (and SOWB_NATIVE_LOSS is not
    0), ``stock`` otherwise.

    The native path shifts the labels as HF does, gathers logp_t = log_softmax(logits.float())[i, t_i] for every row
    (ops.ce_fwd) and hands that (N, 1) column to torch's own nll_loss, with target 0 for a valid row and the label itself
    otherwise.  nll_loss sums over the rows in an order that depends on N only, so the loss, its total weight and the
    per-row gradient it passes back are torch's, bit for bit; ops.ce_bwd turns that gradient into the logits' gradient."""

    def __init__(self, stock):
        self.stock = stock

    def __call__(self, logits, labels, vocab_size, num_items_in_batch=None, ignore_index=-100, shift_labels=None,
                 **kwargs):
        if (torch.compiler.is_compiling() or os.environ.get("SOWB_NATIVE_LOSS", "1") == "0"
                or not loss_native_ok(logits, labels if shift_labels is None else shift_labels, vocab_size,
                                      ignore_index, shifted=shift_labels is not None)):
            return self.stock(logits, labels, vocab_size, num_items_in_batch=num_items_in_batch,
                              ignore_index=ignore_index, shift_labels=shift_labels, **kwargs)
        if shift_labels is None:
            labels = F.pad(labels, (0, 1), value=ignore_index)
            shift_labels = labels[..., 1:].contiguous()
        logits = logits.view(-1, vocab_size)
        targets = shift_labels.view(-1).to(logits.device)
        logp_t = _CausalLMLoss.apply(logits, targets)
        # a label outside [0, V) is ignore_index (ignored here too) or invalid (nll_loss rejects it, as it does in eager)
        nll_targets = torch.where((targets >= 0) & (targets < vocab_size), 0, targets)
        reduction = "sum" if num_items_in_batch is not None else "mean"
        loss = F.nll_loss(logp_t, nll_targets, ignore_index=ignore_index, reduction=reduction)
        if reduction == "sum":
            if torch.is_tensor(num_items_in_batch):
                num_items_in_batch = num_items_in_batch.to(loss.device)
            loss = loss / num_items_in_batch
        return loss


def install_loss(model: nn.Module) -> bool:
    """Route ``model.loss_function`` (HF's ForCausalLMLoss) through CausalLMLoss, once.  Returns True if installed now."""
    try:
        from transformers.loss.loss_utils import ForCausalLMLoss
    except Exception:  # pragma: no cover - older transformers
        return False
    cur = model.loss_function
    if cur is not ForCausalLMLoss:    # another loss, or already installed
        return False
    model.loss_function = CausalLMLoss(cur)
    return True


# ---- installation ----------------------------------------------------------------------------------------------------

def install_llama_glue(model: nn.Module) -> int:
    """Route the Llama blocks of ``model`` through the native glue.  Returns the number of MLPs newly switched over
    (the RMSNorms and the causal-LM loss are switched over as well, uncounted)."""
    try:
        from transformers.models.llama import modeling_llama as ml
    except Exception:  # pragma: no cover - transformers is optional for the kernels themselves
        return 0
    n, has_attention = 0, False
    for m in model.modules():
        if isinstance(m, ml.LlamaAttention):
            has_attention = True
        elif isinstance(m, ml.LlamaForCausalLM):
            install_loss(m)
        elif type(m).forward is ml.LlamaMLP.forward and isinstance(m, ml.LlamaMLP) and _is_silu(m.act_fn):
            if getattr(m.__dict__.get("forward"), "__func__", None) is not _llama_mlp_forward:
                m.forward = types.MethodType(_llama_mlp_forward, m)
                n += 1
        elif type(m).forward is ml.LlamaRMSNorm.forward and isinstance(m, ml.LlamaRMSNorm):
            if getattr(m.__dict__.get("forward"), "__func__", None) is not _llama_rmsnorm_forward:
                m.forward = types.MethodType(_llama_rmsnorm_forward, m)
    if has_attention:
        install_rope(ml)
    return n
