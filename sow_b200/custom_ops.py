"""torch.library registration of the SoW linear so that ``torch.compile(model)`` (scripts/finetune.py:486-487) traces
THROUGH the kernel-backed layers instead of breaking the graph at each of them (SURVEY.md 8f-4).

Two opaque ops, ``sow_b200::linear_fwd`` and ``sow_b200::linear_bwd``, with fake (meta) implementations and an autograd
formula; their real implementations call the same C-ABI entry points as the eager path (ops.group_fwd / group_bwd with
a group of one).  ``SoWLinear.forward`` takes this route only while dynamo is tracing; eager execution keeps the
autograd.Function path (shared-input groups, gradients written straight into the flat buckets).
"""
from __future__ import annotations

from typing import List, Optional

import torch
from torch import Tensor

from . import ops


def _bf16c(t: Optional[Tensor], dt: torch.dtype = torch.bfloat16) -> Optional[Tensor]:
    """``t`` as a contiguous tensor of the 16-bit compute dtype ``dt`` (bf16, or fp16 on the fp16 path)."""
    if t is None:
        return None
    if t.dtype != dt:
        t = t.to(dt)
    return t if t.is_contiguous() else t.contiguous()


def _half_dtype(x: Tensor, Ws, f32: bool) -> torch.dtype:
    """16-bit compute dtype of a call: fp16 when x and every dense W are fp16 (layer._native_f16), else bf16."""
    f16 = not f32 and x.dtype == torch.float16 and all(w is None or w.dtype == torch.float16 for w in Ws)
    return torch.float16 if f16 else torch.bfloat16


# bf16 pieces of fp32 accumulation weights, keyed by storage address.  The ops take the user-visible W (any dtype) so
# that the traced graph holds no Python-side cache logic; the real implementations look the pieces up here.  Cleared
# whenever a W changes under the same address (in-place merge, checkpoint load): invalidate_weight_cache().
_w_pieces = {}


def invalidate_weight_cache() -> None:
    _w_pieces.clear()


def _weight_pieces(W: Optional[Tensor], want_f32: bool, hdt: torch.dtype = torch.bfloat16):
    """(W_c, W_lo): W of the compute dtype ``hdt`` (bf16, or fp16 on the fp16 path) -> (W, None); fp32 W with an fp32
    caller -> its two bf16 pieces (cached); else one bf16 copy."""
    if W is None or W.numel() == 0:
        return None, None
    if W.dtype == hdt and W.is_contiguous():
        return W, None
    key = (W.data_ptr(), W._version, W.dtype, want_f32)
    hit = _w_pieces.get(W.data_ptr())
    if hit is not None and hit[0] == key:
        return hit[1]
    Wd = W.detach()
    if want_f32 and W.dtype == torch.float32:
        pieces = ops.split_f32(Wd if Wd.is_contiguous() else Wd.contiguous())
    else:
        pieces = (Wd.to(torch.bfloat16).contiguous(), None)
    _w_pieces[W.data_ptr()] = (key, pieces)
    return pieces


@torch.library.custom_op("sow_b200::linear_fwd", mutates_args=())
def linear_fwd(x: Tensor, W: Optional[Tensor], A: Tensor, B: Tensor, bias: Optional[Tensor], scale: float) -> List[Tensor]:
    """[y (..., out) in x.dtype, A_pad (in, r_pad), t (T, r_pad)] with A_pad / t fp16 on the fp16 path, else bf16.
    W: acc_downweight (any dtype) or None."""
    fin = A.shape[0]
    lead = x.shape[:-1]
    f32 = x.dtype == torch.float32 and W is not None and W.dtype == torch.float32 and (bias is None or bias.dtype == torch.float32)
    hdt = _half_dtype(x, [W], f32)
    if x.numel() == 0:
        rp = ops.rank_pad(A.shape[1])
        return [x.new_zeros(*lead, B.shape[1]), x.new_zeros((fin, rp), dtype=hdt), x.new_zeros((0, rp), dtype=hdt)]
    W, W_lo = _weight_pieces(W, f32, hdt)
    if f32:
        xf = x.reshape(-1, fin)
        x_hi, x_lo = ops.split_f32(xf if xf.is_contiguous() else xf.contiguous())
        ys, A_cat, t_cat = ops.group_fwd(x_hi, [(W, _bf16c(A), _bf16c(B), None if bias is None else bias.contiguous(),
                                                 scale, W_lo)], x_lo=x_lo)
    else:
        ys, A_cat, t_cat = ops.group_fwd(_bf16c(x.reshape(-1, fin), hdt),
                                         [(_bf16c(W, hdt), _bf16c(A, hdt), _bf16c(B, hdt), _bf16c(bias, hdt), scale)])
    y = ys[0].reshape(*lead, B.shape[1])
    return [y if y.dtype == x.dtype else y.to(x.dtype), A_cat, t_cat]


@linear_fwd.register_fake
def _(x, W, A, B, bias, scale):
    fin = A.shape[0]
    rp = (A.shape[1] + 63) // 64 * 64
    T = x.numel() // fin
    f32 = x.dtype == torch.float32 and W is not None and W.dtype == torch.float32 and (bias is None or bias.dtype == torch.float32)
    hdt = _half_dtype(x, [W], f32)
    return [x.new_empty((*x.shape[:-1], B.shape[1])), x.new_empty((fin, rp), dtype=hdt), x.new_empty((T, rp), dtype=hdt)]


@torch.library.custom_op("sow_b200::linear_bwd", mutates_args=())
def linear_bwd(dy: Tensor, x: Tensor, W: Optional[Tensor], A_pad: Tensor, t: Tensor, B: Tensor, scale: float, r: int,
               need_dx: bool, need_dbias: bool, f32: bool) -> List[Tensor]:
    """[dx (x.shape, x.dtype; empty if not needed), dA (in, r), dB (r, out), dbias (out) or empty]; the gradients have t's
    dtype (fp16 on the fp16 path, else bf16)."""
    fin = A_pad.shape[0]
    fout = B.shape[1]
    dev = x.device
    hdt = t.dtype
    if x.numel() == 0:
        return [x.new_zeros(x.shape if need_dx else (0,)), torch.zeros((fin, r), dtype=hdt, device=dev),
                torch.zeros((r, fout), dtype=hdt, device=dev), torch.zeros((fout if need_dbias else 0,), dtype=hdt, device=dev)]
    W, W_lo = _weight_pieces(W, f32, hdt)
    dy2 = dy.reshape(-1, fout)
    if f32:
        xf = x.reshape(-1, fin)
        x_hi, _ = ops.split_f32(xf if xf.is_contiguous() else xf.contiguous())
        dyf = dy2 if dy2.dtype == torch.float32 else dy2.float()
        dy_hi, dy_lo = ops.split_f32(dyf if dyf.is_contiguous() else dyf.contiguous())
        member = (W, _bf16c(B), dy_hi, scale, True, True, need_dbias, W_lo, dy_lo)
        dx, dAs, dBs, dbs = ops.group_bwd(x_hi, A_pad, t, [member], need_dx, f32=True)
    else:
        member = (_bf16c(W, hdt), _bf16c(B, hdt), _bf16c(dy2, hdt), scale, True, True, need_dbias)
        dx, dAs, dBs, dbs = ops.group_bwd(_bf16c(x.reshape(-1, fin), hdt), A_pad, t, [member], need_dx)
    if dx is None:
        dx = x.new_zeros((0,))
    else:
        dx = dx.reshape(x.shape)
        dx = dx if dx.dtype == x.dtype else dx.to(x.dtype)
    db = dbs[0] if dbs[0] is not None else torch.zeros((0,), dtype=hdt, device=dev)
    return [dx, dAs[0], dBs[0], db]


@linear_bwd.register_fake
def _(dy, x, W, A_pad, t, B, scale, r, need_dx, need_dbias, f32):
    fin, fout = A_pad.shape[0], B.shape[1]
    return [x.new_empty(x.shape if need_dx else (0,)), x.new_empty((fin, r), dtype=t.dtype),
            x.new_empty((r, fout), dtype=t.dtype), x.new_empty((fout if need_dbias else 0,), dtype=t.dtype)]


def _setup_context(ctx, inputs, output):
    x, W, A, B, bias, scale = inputs
    _, A_pad, t = output
    ctx.save_for_backward(x, W, A_pad, t, B)
    ctx.scale = float(scale)
    ctx.r = int(A.shape[1])
    ctx.dtypes = (A.dtype, B.dtype, None if bias is None else bias.dtype)
    ctx.f32 = bool(x.dtype == torch.float32 and W is not None and W.dtype == torch.float32
                   and (bias is None or bias.dtype == torch.float32))


def _backward(ctx, grads):
    dy = grads[0]
    x, W, A_pad, t, B = ctx.saved_tensors
    need_x, _, need_A, need_B, need_bias, _ = ctx.needs_input_grad
    a_dt, b_dt, bias_dt = ctx.dtypes
    dx, dA, dB, db = linear_bwd(dy, x, W, A_pad, t, B, ctx.scale, ctx.r, bool(need_x),
                                bool(need_bias) and bias_dt is not None, ctx.f32)
    return (dx if need_x else None, None,
            (dA if dA.dtype == a_dt else dA.to(a_dt)) if need_A else None,
            (dB if dB.dtype == b_dt else dB.to(b_dt)) if need_B else None,
            (db if db.dtype == bias_dt else db.to(bias_dt)) if (need_bias and bias_dt is not None) else None, None)


linear_fwd.register_autograd(_backward, setup_context=_setup_context)


def sow_linear_traceable(x: Tensor, W: Optional[Tensor], A: Tensor, B: Tensor, bias: Optional[Tensor],
                         scale: float) -> Tensor:
    """y = x.W + scale*(x.A).B + bias through the registered ops (what SoWLinear.forward calls under torch.compile)."""
    return linear_fwd(x, W, A, B, bias, float(scale))[0]


# ---------------------------------------------------------------------------------------------------------
# projection GROUPS as one traceable op (q/k/v, gate/up: one t_cat / dA_cat / dX launch per group also when compiled)
# ---------------------------------------------------------------------------------------------------------
from typing import Sequence  # noqa: E402


def _group_f32(x: Tensor, Ws, biases) -> bool:
    """The fp32-faithful (bf16x3) path of a group: fp32 x, at least one dense W, and every W and bias fp32."""
    return bool(x.dtype == torch.float32 and any(w is not None for w in Ws)
                and all(w is None or w.dtype == torch.float32 for w in Ws)
                and all(b is None or b.dtype == torch.float32 for b in biases))


@torch.library.custom_op("sow_b200::group_fwd", mutates_args=())
def group_fwd(x: Tensor, Ws: Sequence[Optional[Tensor]], As: Sequence[Tensor], Bs: Sequence[Tensor],
              biases: Sequence[Optional[Tensor]], scales: Sequence[float]) -> List[Tensor]:
    """[y_0 .. y_{n-1} (x.dtype), A_cat (in, R), t_cat (T, R)] for n projections that read the same x; A_cat / t_cat
    fp16 on the fp16 path, else bf16."""
    n = len(As)
    fin = As[0].shape[0]
    lead = x.shape[:-1]
    R = sum(ops.rank_pad(a.shape[1]) for a in As)
    f32 = _group_f32(x, Ws, biases)
    hdt = _half_dtype(x, Ws, f32)
    if x.numel() == 0:
        return [x.new_zeros(*lead, b.shape[1]) for b in Bs] + [x.new_zeros((fin, R), dtype=hdt), x.new_zeros((0, R), dtype=hdt)]
    pieces = [_weight_pieces(w, f32, hdt) for w in Ws]
    if f32:
        xf = x.reshape(-1, fin)
        x_hi, x_lo = ops.split_f32(xf if xf.is_contiguous() else xf.contiguous())
        ys, A_cat, t_cat = ops.group_fwd(
            x_hi, [(pieces[i][0], _bf16c(As[i]), _bf16c(Bs[i]), None if biases[i] is None else biases[i].contiguous(),
                    scales[i], pieces[i][1]) for i in range(n)], x_lo=x_lo)
    else:
        ys, A_cat, t_cat = ops.group_fwd(
            _bf16c(x.reshape(-1, fin), hdt),
            [(pieces[i][0], _bf16c(As[i], hdt), _bf16c(Bs[i], hdt), _bf16c(biases[i], hdt), scales[i]) for i in range(n)])
    outs = []
    for y, b in zip(ys, Bs):
        y = y.reshape(*lead, b.shape[1])
        outs.append(y if y.dtype == x.dtype else y.to(x.dtype))
    return outs + [A_cat, t_cat]


@group_fwd.register_fake
def _(x, Ws, As, Bs, biases, scales):
    fin = As[0].shape[0]
    R = sum((a.shape[1] + 63) // 64 * 64 for a in As)
    T = x.numel() // fin
    hdt = _half_dtype(x, Ws, _group_f32(x, Ws, biases))
    return [x.new_empty((*x.shape[:-1], b.shape[1])) for b in Bs] + [x.new_empty((fin, R), dtype=hdt),
                                                                    x.new_empty((T, R), dtype=hdt)]


@torch.library.custom_op("sow_b200::group_bwd", mutates_args=())
def group_bwd(dys: Sequence[Tensor], x: Tensor, Ws: Sequence[Optional[Tensor]], A_cat: Tensor, t_cat: Tensor,
              Bs: Sequence[Tensor], scales: Sequence[float], ranks: Sequence[int], need_dx: bool,
              need_dbias: Sequence[bool], f32: bool) -> List[Tensor]:
    """[dx (empty if not needed)] + [dA_i (in, r_i)] + [dB_i (r_i, out_i)] + [dbias_i (out_i) or empty]; the gradients
    have t_cat's dtype (fp16 on the fp16 path, else bf16)."""
    n = len(Bs)
    fin = A_cat.shape[0]
    dev = x.device
    hdt = t_cat.dtype
    if x.numel() == 0:
        return ([x.new_zeros(x.shape if need_dx else (0,))]
                + [torch.zeros((fin, ranks[i]), dtype=hdt, device=dev) for i in range(n)]
                + [torch.zeros((ranks[i], Bs[i].shape[1]), dtype=hdt, device=dev) for i in range(n)]
                + [torch.zeros((Bs[i].shape[1] if need_dbias[i] else 0,), dtype=hdt, device=dev) for i in range(n)])
    pieces = [_weight_pieces(w, f32, hdt) for w in Ws]
    members = []
    if f32:
        xf = x.reshape(-1, fin)
        x2, _ = ops.split_f32(xf if xf.is_contiguous() else xf.contiguous())
    else:
        x2 = _bf16c(x.reshape(-1, fin), hdt)
    for i in range(n):
        dy2 = dys[i].reshape(-1, Bs[i].shape[1])
        if f32:
            dyf = dy2 if dy2.dtype == torch.float32 else dy2.float()
            dy_hi, dy_lo = ops.split_f32(dyf if dyf.is_contiguous() else dyf.contiguous())
            members.append((pieces[i][0], _bf16c(Bs[i]), dy_hi, scales[i], True, True, need_dbias[i], pieces[i][1],
                            dy_lo if pieces[i][0] is not None else None))
        else:
            members.append((pieces[i][0], _bf16c(Bs[i], hdt), _bf16c(dy2, hdt), scales[i], True, True, need_dbias[i]))
    dx, dAs, dBs, dbs = ops.group_bwd(x2, A_cat, t_cat, members, need_dx, f32=f32)
    if dx is None:
        dx = x.new_zeros((0,))
    else:
        dx = dx.reshape(x.shape)
        dx = dx if dx.dtype == x.dtype else dx.to(x.dtype)
    dbs = [d if d is not None else torch.zeros((0,), dtype=hdt, device=dev) for d in dbs]
    return [dx] + list(dAs) + list(dBs) + dbs


@group_bwd.register_fake
def _(dys, x, Ws, A_cat, t_cat, Bs, scales, ranks, need_dx, need_dbias, f32):
    n = len(Bs)
    fin = A_cat.shape[0]
    hdt = t_cat.dtype
    return ([x.new_empty(x.shape if need_dx else (0,))]
            + [x.new_empty((fin, ranks[i]), dtype=hdt) for i in range(n)]
            + [x.new_empty((ranks[i], Bs[i].shape[1]), dtype=hdt) for i in range(n)]
            + [x.new_empty((Bs[i].shape[1] if need_dbias[i] else 0,), dtype=hdt) for i in range(n)])


def _group_setup_context(ctx, inputs, output):
    x, Ws, As, Bs, biases, scales = inputs
    n = len(As)
    ctx.n = n
    ctx.save_for_backward(x, output[n], output[n + 1], *Bs, *[w for w in Ws if w is not None])
    ctx.has_w = [w is not None for w in Ws]
    ctx.scales = [float(s) for s in scales]
    ctx.ranks = [int(a.shape[1]) for a in As]
    ctx.dtypes = ([a.dtype for a in As], [b.dtype for b in Bs], [None if b is None else b.dtype for b in biases])
    ctx.f32 = _group_f32(x, Ws, biases)


def _group_backward(ctx, grads):
    n = ctx.n
    saved = ctx.saved_tensors
    x, A_cat, t_cat = saved[0], saved[1], saved[2]
    Bs = list(saved[3:3 + n])
    w_it = iter(saved[3 + n:])
    Ws = [next(w_it) if h else None for h in ctx.has_w]
    a_dts, b_dts, bias_dts = ctx.dtypes
    need_x = ctx.needs_input_grad[0]
    need_bias = [bias_dts[i] is not None for i in range(n)]      # frozen biases: their gradients are simply dropped
    dys = [grads[i] if grads[i] is not None else torch.zeros((*x.shape[:-1], Bs[i].shape[1]), dtype=x.dtype, device=x.device)
           for i in range(n)]
    outs = group_bwd(dys, x, Ws, A_cat, t_cat, Bs, ctx.scales, ctx.ranks, bool(need_x), need_bias, ctx.f32)
    dx = outs[0] if need_x else None
    dAs = [d if d.dtype == a_dts[i] else d.to(a_dts[i]) for i, d in enumerate(outs[1:1 + n])]
    dBs = [d if d.dtype == b_dts[i] else d.to(b_dts[i]) for i, d in enumerate(outs[1 + n:1 + 2 * n])]
    dbs = [None if bias_dts[i] is None else (d if d.dtype == bias_dts[i] else d.to(bias_dts[i]))
           for i, d in enumerate(outs[1 + 2 * n:1 + 3 * n])]
    # the returned structure mirrors the inputs: a list argument that held no tensor at all (no dense W yet, no biases)
    # is a plain constant to the dispatcher and takes a single None
    return (dx, [None] * n if any(ctx.has_w) else None, dAs, dBs,
            dbs if any(d is not None for d in bias_dts) else None, None)


group_fwd.register_autograd(_group_backward, setup_context=_group_setup_context)


def sow_group_traceable(x: Tensor, Ws, As, Bs, biases, scales):
    """Outputs of a projection group through the registered group op (SharedInputGroup under torch.compile)."""
    return group_fwd(x, list(Ws), list(As), list(Bs), list(biases), [float(s) for s in scales])[:len(As)]
