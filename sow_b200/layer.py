"""SoW linear layer on sm_100a kernels -- host-side mirror of ``tn_gradient.layer.sow`` (reference file
tn_gradient/layer/sow.py).

Same constructor, attributes, parameter names and state-dict keys as the reference (SURVEY.md 8b):
``acc_downweight`` / ``acc_upweight`` (frozen accumulation, empty until the first merge), ``downscale_weights[i]``
(in, r), ``upscale_weights[i]`` (r, out), ``bias``.  The math is not PyTorch: ``forward`` dispatches to one
autograd Function whose forward/backward call the C ABI (fused tcgen05 GEMMs), ``accumulate`` to the grouped
merge kernel.  CUDA only -- CPU tensors raise (no fallback).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence

import torch
import torch.nn as nn

from . import ops
from ._lib import SowB200Error


@dataclass
class SoWArgs:
    """Legacy argument bundle that scripts/run_glue.py:54,564 imports from ``tn_gradient.layer.sow`` (it only
    survives as a commented-out dataclass in the reference, tn_gradient/prepare.py:16-25)."""
    device: Optional[str] = None
    dtype: Optional[torch.dtype] = None
    init_method: str = "normal_QR"
    rank: int = 16
    n_iter: int = 5
    scale: float = 1


class SoWParameter(nn.ParameterList):
    """``n_iter`` factor matrices of one shape; ``from_weights`` swaps ``.data`` so that Parameter identity (held by
    optimizers and DDP) survives a merge.  Mirrors tn_gradient/layer/sow.py:15-42."""

    def __init__(self, in_features: int, out_features: int, n_iter: int = 1, device=None, dtype=None) -> None:
        super().__init__(
            [nn.Parameter(torch.empty(in_features, out_features, device=device, dtype=dtype)) for _ in range(n_iter)]
        )
        self.in_features = in_features
        self.out_features = out_features
        self.n_iter = n_iter

    def from_weights(self, weights: Sequence[torch.Tensor]) -> None:
        for i, w in enumerate(weights):
            self[i].data = w.data

    def extra_repr(self) -> str:
        return f"{self.n_iter} x ({self.in_features}, {self.out_features})"


# ---------------------------------------------------------------------------------------------------------
# autograd bridge
# ---------------------------------------------------------------------------------------------------------

def _halfc(t: Optional[torch.Tensor], dt: torch.dtype) -> Optional[torch.Tensor]:
    """``t`` as a contiguous tensor of the 16-bit compute dtype ``dt`` (no copy when it already is one)."""
    if t is None:
        return None
    if t.dtype != dt:
        t = t.to(dt)
    return t if t.is_contiguous() else t.contiguous()


def _bf16c(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    return _halfc(t, torch.bfloat16)


def _native_f16(x_dtype: torch.dtype, Ws) -> bool:
    """The fp16 path: fp16 activations and every dense W of the group fp16 (no W yet counts as fp16)."""
    return x_dtype == torch.float16 and all(w is None or w.dtype == torch.float16 for w in Ws)


def _grad_dst(param: Optional[torch.Tensor], dt: torch.dtype = torch.bfloat16):
    """Where the kernels should write the gradient of a factor: the parameter's view into a flat gradient bucket
    (``_sow_grad_view``, set by parallel.FlatGradSync) when the parameter has no gradient yet -- autograd's AccumulateGrad
    then adopts the returned view as ``param.grad`` without a copy or an add -- else a fresh tensor.  ``dt``: the dtype
    the kernels write (bf16, or fp16 on the fp16 path)."""
    if param is None:
        return True
    view = getattr(param, "_sow_grad_view", None)
    if view is not None and param.grad is None and view.dtype == dt:
        return view
    return True


class _SoWGroupFn(torch.autograd.Function):
    """y_i = x.W_i + scale_i*(x.A_i).B_i + bias_i for the n projections of a group that read the same x, W_i frozen.
    Saves x, the packed factors A_cat and t_cat = scale_i*x.A_cat (T x R); never forms dW.

    Positional inputs after ``scales``: for each member (W_c or None, A, B, bias or None, W_lo or None).
      * bf16 modules: ``W_c`` is W itself, everything runs in bf16 with fp32 accumulation.
      * fp16 modules (fp16 x and every dense W fp16): the same in fp16 -- no cast of x, dY or W; factors and biases of
        another dtype are rounded to fp16 once per call and their gradients returned in their own dtype.
      * fp32 modules (fp32 x, and every dense W given as its two bf16 pieces W_c + W_lo, see SoWLinear._compute_weight):
        the fp32-faithful path -- x and dY are split into two bf16 pieces on the fly, the base products run as bf16x3
        tensor-core contractions, outputs and dX are fp32; the small rank-r factors are rounded to bf16 once.
      * anything else (mixed dtypes) follows the bf16 compute policy: cast in, cast back."""

    @staticmethod
    def forward(ctx, x, scales, *params):
        n = len(scales)
        out_dtype = x.dtype
        Ws, As, Bs, biases, Wlos = params[0::5], params[1::5], params[2::5], params[3::5], params[4::5]
        fin = As[0].shape[0]
        lead = x.shape[:-1]
        ctx.n = n
        ctx.meta = (out_dtype, [a.dtype for a in As], [b.dtype for b in Bs],
                    [None if b is None else b.dtype for b in biases], lead, fin,
                    [a.shape for a in As], [b.shape for b in Bs])
        if x.numel() == 0:                      # empty batch: nothing to launch (the reference returns an empty tensor too)
            ctx.empty = True
            return tuple(x.new_zeros(*lead, b.shape[1]) for b in Bs)
        ctx.empty = False
        f32 = (x.dtype == torch.float32 and all((w is None) == (wl is None) for w, wl in zip(Ws, Wlos))
               and all(b is None or b.dtype == torch.float32 for b in biases) and any(w is not None for w in Ws))
        ctx.f32 = f32
        hdt = torch.float16 if (not f32 and _native_f16(x.dtype, Ws)) else torch.bfloat16
        ctx.hdt = hdt
        Bc = [_halfc(b, hdt) for b in Bs]
        if f32:
            xf = x.reshape(-1, fin)
            x2, x_lo = ops.split_f32(xf if xf.is_contiguous() else xf.contiguous())
            Wc, Wl = list(Ws), list(Wlos)
            ys, A_cat, t_cat = ops.group_fwd(
                x2, [(Wc[i], _bf16c(As[i]), Bc[i], None if biases[i] is None else biases[i].contiguous(), scales[i], Wl[i])
                     for i in range(n)], x_lo=x_lo)
        else:
            x2 = _halfc(x.reshape(-1, fin), hdt)
            Wc = [_halfc(w, hdt) for w in Ws]
            Wl = [None] * n
            ys, A_cat, t_cat = ops.group_fwd(
                x2, [(Wc[i], _halfc(As[i], hdt), Bc[i], _halfc(biases[i], hdt), scales[i]) for i in range(n)])
        ctx.has_w = [w is not None for w in Wc]
        ctx.save_for_backward(x2, A_cat, t_cat, *[w for w in Wc if w is not None], *[w for w in Wl if w is not None], *Bc)
        ctx.scales = tuple(float(s) for s in scales)
        # leaf factor Parameters: their gradients may be written straight into a flat bucket view
        ctx.leaves = [(a if isinstance(a, nn.Parameter) else None, b if isinstance(b, nn.Parameter) else None)
                      for a, b in zip(As, Bs)]
        outs = []
        for y, b in zip(ys, Bs):
            y = y.reshape(*lead, b.shape[1])
            outs.append(y if y.dtype == out_dtype else y.to(out_dtype))
        return tuple(outs)

    @staticmethod
    def backward(ctx, *dys):
        n = ctx.n
        out_dtype, a_dts, b_dts, bias_dts, lead, fin, a_shapes, b_shapes = ctx.meta
        need = ctx.needs_input_grad
        need_x = need[0]
        grads = [None, None]
        if ctx.empty:
            for i in range(n):
                nW, nA, nB, nb, _ = need[2 + 5 * i: 7 + 5 * i]
                grads += [None,
                          torch.zeros(a_shapes[i], dtype=a_dts[i], device=dys[0].device) if nA else None,
                          torch.zeros(b_shapes[i], dtype=b_dts[i], device=dys[0].device) if nB else None,
                          torch.zeros(b_shapes[i][1], dtype=bias_dts[i], device=dys[0].device) if (nb and bias_dts[i] is not None) else None,
                          None]
            grads[0] = dys[0].new_zeros(*lead, fin) if need_x else None
            return tuple(grads)
        saved = list(ctx.saved_tensors)
        x2, A_cat, t_cat = saved[0], saved[1], saved[2]
        nw = sum(ctx.has_w)
        w_it = iter(saved[3:3 + nw])
        wl_it = iter(saved[3 + nw:3 + 2 * nw]) if ctx.f32 else iter(())
        Bc = saved[-n:]
        Wc = [next(w_it) if h else None for h in ctx.has_w]
        Wl = [(next(wl_it) if h else None) if ctx.f32 else None for h in ctx.has_w]
        members = []
        for i in range(n):
            nW, nA, nB, nb, _ = need[2 + 5 * i: 7 + 5 * i]
            dyi = dys[i].reshape(-1, dys[i].shape[-1])
            if ctx.f32:
                dyi = dyi if dyi.dtype == torch.float32 else dyi.float()
                dy2, dy_lo = ops.split_f32(dyi if dyi.is_contiguous() else dyi.contiguous())
            else:
                dy2, dy_lo = _halfc(dyi, ctx.hdt), None
            pa, pb = ctx.leaves[i]
            gdt = torch.bfloat16 if ctx.f32 else ctx.hdt          # dtype the kernels write the factor gradients in
            dA_dst = (_grad_dst(pa, gdt) if a_dts[i] == gdt else True) if nA else None
            dB_dst = (_grad_dst(pb, gdt) if b_dts[i] == gdt else True) if nB else None
            members.append((Wc[i], Bc[i], dy2, ctx.scales[i], dA_dst, dB_dst, bool(nb) and bias_dts[i] is not None,
                            Wl[i], dy_lo if Wc[i] is not None else None))
        dx, dAs, dBs, dbs = ops.group_bwd(x2, A_cat, t_cat, members, bool(need_x), f32=ctx.f32)
        if dx is not None:
            dx = dx.reshape(*lead, fin)
            if dx.dtype != out_dtype:
                dx = dx.to(out_dtype)
        grads[0] = dx
        for i in range(n):
            dA, dB, db = dAs[i], dBs[i], dbs[i]
            grads += [None,
                      None if dA is None else (dA if a_dts[i] == dA.dtype else dA.to(a_dts[i])),
                      None if dB is None else (dB if b_dts[i] == dB.dtype else dB.to(b_dts[i])),
                      None if db is None else (db if bias_dts[i] == db.dtype else db.to(bias_dts[i])),
                      None]
        return tuple(grads)


@torch.compiler.disable
def sow_linear_group(x, scales, params):
    """Kernel-backed SoW projections sharing one input.  Opaque to torch.compile (scripts/finetune.py:486-487 compiles
    the model): the C-ABI calls are not traceable, so dynamo breaks the graph here and runs this call eagerly."""
    return _SoWGroupFn.apply(x, tuple(scales), *params)


def sow_linear(x, W_c, A, B, bias, scale, W_lo=None):
    """One projection = a group of one."""
    return sow_linear_group(x, (scale,), (W_c, A, B, bias, W_lo))[0]


class SharedInputGroup:
    """SoW projections of one block that are called with the SAME input tensor (q/k/v, gate/up; SURVEY.md 8f-4:
    simple_train.py:318 lists them as separate target modules).  The first member called with a new x runs the whole
    group through ONE autograd node (one pass over x for all t_i and dA_i, one dX for all members) and parks the other
    members' outputs; the siblings, called with the identical tensor object, pick theirs up.  User-visible parameters and
    module call sites stay untouched.  If the siblings turn out to be called with different tensors the group switches
    itself off (each member then runs as a group of one)."""

    MAX_MISSES = 4

    def __init__(self, members: Sequence["SoWLinear"]):
        self.members = list(members)
        self.index = {id(m): i for i, m in enumerate(self.members)}
        self.cache = None            # (x, x._version, grad_mode, {member index: parked output})
        self.misses = 0
        self.enabled = True
        # a member's factors enter the group call concatenated (rank * n_iter columns); too wide a group runs its members
        # one by one, each of which fits on its own
        self.rank_fits = ops.group_rank_fits(m.rank * m.n_iter for m in self.members)

    def usable_traced(self) -> bool:
        ms = self.members
        return (self.enabled and self.rank_fits and 2 <= len(ms) <= 4
                and all(m.n_iter == 1 and m.acc_upweight.numel() == 0 for m in ms))

    def usable(self) -> bool:
        ms = self.members
        if not self.enabled or not self.rank_fits or len(ms) < 2 or len(ms) > 4:
            return False
        m0 = ms[0]
        n_dense = 0
        for m in ms:
            if (m.in_features != m0.in_features or m.acc_upweight.numel() != 0 or
                    m.downscale_weights[0].device != m0.downscale_weights[0].device):
                return False
            n_dense += m.acc_downweight.numel() != 0
        return n_dense <= 3

    def forward_traced(self, idx: int, x: torch.Tensor) -> torch.Tensor:
        """Same protocol while dynamo traces (torch.compile): tensor identity is the identity of the traced value, the
        whole group is ONE sow_b200::group_fwd node in the graph."""
        c = self.cache
        if c is not None and c[0] is x and idx in c[3]:
            y = c[3].pop(idx)
            if not c[3]:
                self.cache = None
            return y
        from .custom_ops import sow_group_traceable
        ms = self.members
        Ws = [m.acc_downweight if m.acc_downweight.numel() != 0 else None for m in ms]
        ys = sow_group_traceable(x, Ws, [m.downscale_weights[0] for m in ms], [m.upscale_weights[0] for m in ms],
                                 [m.bias for m in ms], [m.scale for m in ms])
        self.cache = (x, 0, True, {i: y for i, y in enumerate(ys) if i != idx})
        return ys[idx]

    def forward(self, mod: "SoWLinear", x: torch.Tensor) -> torch.Tensor:
        idx = self.index[id(mod)]
        c = self.cache
        if c is not None and c[0] is x and c[1] == x._version and c[2] == torch.is_grad_enabled() and idx in c[3]:
            y = c[3].pop(idx)
            if not c[3]:
                self.cache = None
            return y
        if c is not None and c[3]:
            self.misses += 1         # parked outputs were never picked up: the members do not share their input
            if self.misses >= self.MAX_MISSES:
                self.enabled = False
                self.cache = None
                return _forward_modules([mod], x)[0]
        ys = _forward_modules(self.members, x)
        self.cache = (x, x._version, torch.is_grad_enabled(), {i: y for i, y in enumerate(ys) if i != idx})
        return ys[idx]


def _forward_modules(mods: Sequence["SoWLinear"], x: torch.Tensor):
    params, scales = [], []
    f16 = _native_f16(x.dtype, [m.acc_downweight if m.acc_downweight.numel() != 0 else None for m in mods])
    for m in mods:
        A_list, B_list = list(m.downscale_weights), list(m.upscale_weights)
        if len(A_list) == 1:
            A, B = A_list[0], B_list[0]
        else:
            # sum_i (x.A_i).B_i == (x.[A_1|..|A_n]).[B_1;..;B_n]: one fused call; autograd splits the grads
            A = torch.cat(A_list, dim=1)
            B = torch.cat(B_list, dim=0)
        W_c, W_lo = m._compute_weight(native_f16=f16)
        params += [W_c, A, B, m.bias, W_lo]
        scales.append(m.scale)
    return sow_linear_group(x, scales, params)


# ---------------------------------------------------------------------------------------------------------
# QR initialisation helpers (thin-QR kernel instead of a full in x out QR)
# ---------------------------------------------------------------------------------------------------------

def _cuda_device_for(t: torch.Tensor) -> torch.device:
    if t.is_cuda:
        return t.device
    if not torch.cuda.is_available():
        raise SowB200Error(
            'init_method="normal_QR" runs its QR on the GPU (the reference hard-codes .to("cuda") too, '
            "tn_gradient/layer/sow.py:91) and no CUDA device is available"
        )
    return torch.device("cuda", torch.cuda.current_device())


def qr_init_factors(in_features: int, out_features: int, rank: int, device: torch.device, want_b: bool,
                    std: float = 0.02, generator: Optional[torch.Generator] = None):
    """A = first ``rank`` columns of Q of QR(G), G ~ N(0, std) (in x out); B = A^T G (= R[:rank]) if requested.

    Q[:, :rank] of a Householder QR depends on the first ``rank`` columns only (SURVEY.md section 7), so the thin-QR
    kernel on those columns yields the same subspace at 1/(out/rank) of the cost; columns are sign-normalised
    (diag(R) >= 0) whereas LAPACK's signs vary, which leaves A.B and the distribution of A unchanged.
    """
    if want_b:
        G = torch.empty((in_features, out_features), dtype=torch.float32, device=device).normal_(0.0, std, generator=generator)
        A = ops.thin_qr(G, rank)
        B = ops.project(G, A)
        return A, B
    G = torch.empty((in_features, rank), dtype=torch.float32, device=device).normal_(0.0, std, generator=generator)
    return ops.thin_qr(G, rank), None


class SoWLinear(nn.Module):
    """Drop-in for tn_gradient.layer.sow.SoWLinear (tn_gradient/layer/sow.py:45-181)."""

    def __init__(self, in_features: int, out_features: int, bias: bool = True, rank: int = 16, n_iter: int = 1,
                 scale: float = 1, init_method: str = "normal_QR", device=None, dtype=None, init_params=True) -> None:
        super().__init__()
        fk = {"device": device, "dtype": dtype}
        self.in_features = in_features
        self.out_features = out_features
        self.n_iter = n_iter
        self.rank = rank
        self.scale = scale
        self.virtual_rank = min(rank * n_iter, in_features, out_features)
        self.init_method = init_method

        self.acc_upweight = nn.Parameter(torch.empty(0), requires_grad=False)
        self.acc_downweight = nn.Parameter(torch.empty(0), requires_grad=False)
        self.downscale_weights = SoWParameter(in_features, rank, n_iter=n_iter, device=device, dtype=dtype)
        self.upscale_weights = SoWParameter(rank, out_features, n_iter=n_iter, device=device, dtype=dtype)
        if bias:
            self.bias = nn.Parameter(torch.empty(out_features, **fk))
        else:
            self.register_parameter("bias", None)
        self._w_shadow = None       # compute copy of acc_downweight: bf16x3 pieces of fp32, bf16 copy of a mixed-dtype W
        self._w_shadow_key = None
        self._group = None          # SharedInputGroup of the projections that read the same input (surgery.group_shared_inputs)
        self._group_index = -1
        if init_params:
            self.reset_parameters()

    # ---- initialisation (sow.py:89-105) ------------------------------------------------------------------
    def reset_parameters(self, reset_scale=1.0) -> None:
        for i in range(self.n_iter):
            if i / self.n_iter >= 1 - reset_scale:
                A_p, B_p = self.downscale_weights[i], self.upscale_weights[i]
                if self.init_method == "normal_QR":
                    dev = _cuda_device_for(A_p)
                    A, B = qr_init_factors(self.in_features, self.out_features, self.rank, dev, want_b=True)
                    with torch.no_grad():
                        A_p.copy_(A.to(A_p.device))
                        B_p.copy_(B.to(B_p.device))
                else:
                    nn.init.normal_(A_p, std=0.02)
                    nn.init.normal_(B_p, std=0.02)
        if self.bias is not None:
            nn.init.zeros_(self.bias)

    # ---- forward (sow.py:107-126) ---------------------------------------------------------------------------
    def _compute_weight(self, native_f16: bool = False):
        """(W_c, W_lo): the operand(s) the kernels read for the frozen accumulation.  bf16 W: (W, None), no copy.  fp16 W
        of a call on the fp16 path (``native_f16``): (W, None), no copy.  fp32 W: its two bf16 pieces (W ~ W_c + W_lo,
        2^-17 relative) for the bf16x3 path, cached until W changes (merge, load).  Other dtypes: one bf16 copy (bf16
        compute policy)."""
        W = self.acc_downweight
        if W.numel() == 0:
            return None, None
        if W.is_contiguous() and (W.dtype == torch.bfloat16 or (native_f16 and W.dtype == torch.float16)):
            return W, None
        key = (W.data_ptr(), W._version, W.dtype)
        if self._w_shadow is None or self._w_shadow_key != key:
            Wd = W.detach()
            if W.dtype == torch.float32 and W.is_cuda:
                self._w_shadow = ops.split_f32(Wd if Wd.is_contiguous() else Wd.contiguous())
            else:
                self._w_shadow = (Wd.to(torch.bfloat16).contiguous(), None)
            self._w_shadow_key = key
        return self._w_shadow

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if not x.is_cuda:
            raise SowB200Error("SoWLinear.forward needs CUDA tensors (sm_100a kernels only, no CPU fallback)")
        factored = self.acc_downweight.numel() != 0 and self.acc_upweight.numel() != 0
        if factored:
            # compat branch (direct construction with virtual_rank < min(in,out); never reached through
            # prepare_sow, prepare.py:120): the frozen factored accumulation goes through cuBLAS
            A_list, B_list = list(self.downscale_weights), list(self.upscale_weights)
            A = A_list[0] if len(A_list) == 1 else torch.cat(A_list, dim=1)
            B = B_list[0] if len(B_list) == 1 else torch.cat(B_list, dim=0)
            out = sow_linear(x, None, A, B, None, self.scale)
            out = out + (x @ self.acc_downweight.to(x.dtype)) @ self.acc_upweight.to(x.dtype)
            if self.bias is not None:
                out = out + self.bias.to(out.dtype)
            return out
        if torch.compiler.is_compiling():
            # torch.compile(model) (scripts/finetune.py:486-487): registered custom ops, traced without a graph break
            grp = self._group
            if grp is not None and self._group_index >= 0 and self.n_iter == 1 and grp.usable_traced():
                return grp.forward_traced(self._group_index, x)
            from .custom_ops import sow_linear_traceable
            A_list, B_list = list(self.downscale_weights), list(self.upscale_weights)
            A = A_list[0] if len(A_list) == 1 else torch.cat(A_list, dim=1)
            B = B_list[0] if len(B_list) == 1 else torch.cat(B_list, dim=0)
            W = self.acc_downweight if self.acc_downweight.numel() != 0 else None
            return sow_linear_traceable(x, W, A, B, self.bias, self.scale)
        grp = self._group
        if grp is not None and grp.usable():
            return grp.forward(self, x)
        return _forward_modules([self], x)[0]

    # ---- merge (sow.py:128-178) ---------------------------------------------------------------------------
    def accumulate(self) -> None:
        accumulate_modules([self])

    def extra_repr(self) -> str:
        return (f"in_features={self.in_features}, out_features={self.out_features}, bias={self.bias is not None}, "
                f"rank={self.rank}, n_iter={self.n_iter}")


# ---------------------------------------------------------------------------------------------------------
# grouped merge + re-initialisation over many modules
# ---------------------------------------------------------------------------------------------------------

def _merge_dense(mods: List[SoWLinear]) -> None:
    """Dense branch (sow.py:151-153) for all modules: one grouped launch per dtype class (and per 64-wide rank chunk).

    bf16 and fp16 modules: tcgen05 kernel in the module's dtype, W updated IN PLACE (pointer-stable).  fp32 modules: exact
    fp32 kernel, in place -- the pretrained weights keep their full precision, as in the reference (sow.py:131-153 stays in
    the parameter dtype).  Anything else (mixed dtypes, other devices) goes through a bf16 compute copy and is cast back."""
    items = {torch.bfloat16: [], torch.float16: [], torch.float32: []}
    post = []
    for mod in mods:
        A_list = [a.detach() for a in mod.downscale_weights]
        B_list = [b.detach() for b in mod.upscale_weights]
        dev = A_list[0].device
        if not dev.type == "cuda":
            raise SowB200Error("SoWLinear.accumulate needs the module on a CUDA device (no CPU fallback)")
        A = A_list[0] if len(A_list) == 1 else torch.cat(A_list, dim=1)
        B = B_list[0] if len(B_list) == 1 else torch.cat(B_list, dim=0)
        pdtype = A.dtype
        W_old = mod.acc_downweight
        expanded = W_old.numel() != 0 and mod.acc_upweight.numel() != 0
        if expanded:
            # last QR-growth step reached full rank: expand the factored accumulation once (sow.py:137-138); the
            # product is a temporary, so the merged result must be bound as the new acc_downweight below
            tgt = W_old.dtype
            W_tmp = (W_old.detach() @ mod.acc_upweight.detach()).to(dev)
            cls = torch.float32 if (tgt == torch.float32 and pdtype == torch.float32) else torch.bfloat16
            W_tmp = W_tmp.to(cls).contiguous()
            items[cls].append((W_tmp, W_tmp, A.to(cls).contiguous(), B.to(cls).contiguous(), mod.scale))
            post.append((mod, W_tmp, tgt))
            continue
        has_prev = W_old.numel() != 0
        wdt = W_old.dtype if has_prev else pdtype
        native = wdt in items and pdtype == wdt and (not has_prev or (W_old.is_contiguous() and W_old.device == dev))
        if native:
            A_c, B_c = A.contiguous(), B.contiguous()
            if has_prev:
                items[wdt].append((W_old.data, W_old.data, A_c, B_c, mod.scale))      # in-place RMW: pointer stays stable
                post.append((mod, None, None))
            else:
                W_new = torch.empty((mod.in_features, mod.out_features), dtype=wdt, device=dev)
                items[wdt].append((W_new, None, A_c, B_c, mod.scale))
                post.append((mod, W_new, wdt))
        else:
            W_new = torch.empty((mod.in_features, mod.out_features), dtype=torch.bfloat16, device=dev)
            prev = _bf16c(W_old.detach().to(dev)) if has_prev else None
            items[torch.bfloat16].append((W_new, prev, _bf16c(A), _bf16c(B), mod.scale))
            post.append((mod, W_new, wdt))
    for lst in items.values():
        ops.merge_grouped(lst)
    for mod, W_new, tgt_dtype in post:
        if W_new is not None:
            W_final = W_new if tgt_dtype == W_new.dtype else W_new.to(tgt_dtype)
            mod.acc_downweight = nn.Parameter(W_final, requires_grad=False)
            mod.acc_upweight = nn.Parameter(torch.empty(0, device=W_final.device), requires_grad=False)
        mod._w_shadow = None
        mod._w_shadow_key = None
    from .custom_ops import invalidate_weight_cache
    invalidate_weight_cache()


def _merge_factored(mod: SoWLinear) -> None:
    """Factored / QR-growth branch (sow.py:137-150), only reachable by direct construction with
    virtual_rank < min(in, out).  One-off compat path: cuBLAS + cuSOLVER through torch (SURVEY.md 8f rank 3)."""
    from .utils import qr_weight
    acc = None
    for a, b in zip(mod.downscale_weights, mod.upscale_weights):
        term = a.detach() @ b.detach()
        acc = term if acc is None else acc + term
    acc = mod.scale * acc
    if mod.acc_downweight.numel() != 0 and mod.acc_upweight.numel() != 0:
        acc = acc + mod.acc_downweight @ mod.acc_upweight
    elif mod.acc_downweight.numel() != 0:
        acc = acc + mod.acc_downweight
    Q, R = qr_weight(acc, rank=mod.virtual_rank)
    mod.acc_downweight = nn.Parameter(Q.contiguous(), requires_grad=False)
    mod.acc_upweight = nn.Parameter(R.contiguous(), requires_grad=False)
    mod.virtual_rank = min(mod.virtual_rank + mod.rank * mod.n_iter, mod.in_features, mod.out_features)


def _reinit(mods: List[SoWLinear], sync: bool) -> None:
    """A <- QR-init / N(0, .02), B <- 0 (sow.py:157-178).  The new values are copied INTO the existing factor storage
    (one multi-tensor copy, one multi-tensor zero fill): Parameter identity is preserved as with the reference's
    ``.data`` swap, every factor keeps its own storage, and the addresses the fused optimizer / gradient buckets / CUDA
    graphs hold stay valid.

    With torch.distributed initialised and ``sync`` the new A is broadcast from rank 0 -- ONE broadcast per batch of
    same-shaped factors -- which makes the replicas consistent by construction (the reference relies on identical RNG
    state on every rank, SURVEY.md 8e)."""
    import torch.distributed as dist
    do_sync = sync and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    # batch the thin QRs of all normal_QR modules that share (in, rank, device)
    groups = {}
    for mod in mods:
        if mod.init_method == "normal_QR":
            dev = mod.downscale_weights[0].device
            groups.setdefault((mod.in_features, mod.rank, dev), []).append(mod)
    dst, src, zeros = [], [], []
    for (fin, r, dev), ms in groups.items():
        n = sum(m.n_iter for m in ms)
        # the reference draws in the accumulation dtype (bf16-rounded Gaussian, sow.py:163-165,170)
        wdt = ms[0].acc_downweight.dtype if ms[0].acc_downweight.numel() else ms[0].downscale_weights[0].dtype
        G = torch.empty((n, fin, r), dtype=torch.float32, device=dev).normal_(0.0, 0.02)
        if wdt != torch.float32:
            G = G.to(wdt).to(torch.float32)
        Q = ops.thin_qr(G, r)
        if do_sync:
            dist.broadcast(Q, src=0)
        k = 0
        for m in ms:
            for i in range(m.n_iter):
                dst.append(m.downscale_weights[i].data)
                src.append(Q[k])
                k += 1
    for mod in mods:
        if mod.init_method != "normal_QR":
            for a in mod.downscale_weights:
                a.data.normal_(std=0.02)
                if do_sync:
                    dist.broadcast(a.data, src=0)
        zeros += [b.data for b in mod.upscale_weights]
    if dst:
        try:
            torch._foreach_copy_(dst, src)
        except Exception:                                  # older torch: no mixed-dtype foreach copy
            for d, s_ in zip(dst, src):
                d.copy_(s_)
    if zeros:
        torch._foreach_zero_(zeros)


@torch.no_grad()
def accumulate_modules(mods: Sequence[SoWLinear], sync_reinit: bool = True) -> None:
    """SoWLinear.accumulate over a list of modules: grouped merge, then factor re-initialisation."""
    mods = list(mods)
    for m in mods:
        if not m.downscale_weights[0].is_cuda:
            raise SowB200Error("SoWLinear.accumulate needs the module on a CUDA device (sm_100a kernels only, no CPU fallback)")
    dense = [m for m in mods if m.virtual_rank >= min(m.in_features, m.out_features)]
    fact = [m for m in mods if m.virtual_rank < min(m.in_features, m.out_features)]
    by_dev = {}
    for m in dense:
        by_dev.setdefault(m.downscale_weights[0].device, []).append(m)
    for ms in by_dev.values():
        _merge_dense(ms)
    for m in fact:
        _merge_factored(m)
    _reinit(mods, sync_reinit)
