"""Optimizers -- host-side mirrors of ``tn_gradient.optimizer.ttadam`` / ``ttsgd`` (reference files
tn_gradient/optimizer/ttadam.py, ttsgd.py) plus the fused multi-tensor AdamW used for the factor group.

TTAdam keeps the reference's state layout (``step``, ``exp_avg``, ``exp_avg_sq`` as TensorTrain objects after a
step with "ranks", ``exp_avg_expr`` / ``exp_avg_sq_expr``) but executes each parameter's update as
    order 2 : tt_adam2_step through a per-parameter ops.TTAdam2Plan (head -> thin QR -> fused reconstruct + Adam + projection;
              the dense moments never reach HBM; rank > 64: tt_adam_fused2 -> thin-QR + projection)
    order>2 : tt_matmul_rk chain + tt_deinterleave -> tt_adam_dense -> tt_interleave -> thin-QR + projection sweep
instead of ~8 elementwise launches, two einsum reconstructions and two complete QRs.
"""
from __future__ import annotations

import math
from math import ceil
from typing import Callable, Iterable, Tuple

import torch
import torch.nn as nn

from . import ops
from ._lib import SowB200Error
from .tt import TensorTrain, reconstruct_interleaved


class TTAdam(torch.optim.Optimizer):
    """tn_gradient/optimizer/ttadam.py:10-117."""

    def __init__(self, params: Iterable[nn.parameter.Parameter], lr: float = 1e-3,
                 betas: Tuple[float, float] = (0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0,
                 amsgrad: bool = False, correct_bias: bool = True):
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=amsgrad,
                        correct_bias=correct_bias)
        super().__init__(params, defaults)

    @torch.no_grad()
    def step(self, closure: Callable = None):
        loss = None
        if closure is not None:
            loss = closure()
        # Tensor-train parameters are independent of each other and each one's step is a chain of small dependent kernels (head,
        # Cholesky-QR) in front of one large kernel: consecutive parameters alternate between side streams, so the chain of
        # one overlaps the large kernel of another.  The side streams fork from / join the caller's stream around the step.
        n_side = self._side_stream_count()
        side, used, forked, tt_index = None, set(), None, 0
        for group in self.param_groups:
            beta1, beta2 = group["betas"]
            for p in group["params"]:
                if p.grad is None:
                    continue
                grad = p.grad
                if grad.is_sparse:
                    raise RuntimeError("TTAdam does not support sparse gradients, please consider SparseAdam instead")
                if not p.is_cuda:
                    raise SowB200Error("TTAdam needs CUDA parameters (sm_100a kernels only, no CPU fallback)")
                state = self.state[p]
                if "step" not in state:
                    state["step"] = 0
                first = "exp_avg" not in state or "exp_avg_sq" not in state
                state["step"] += 1
                step_size = group["lr"]
                if group["correct_bias"]:                                       # ttadam.py:97-100
                    bc1 = 1.0 - beta1 ** state["step"]
                    bc2 = 1.0 - beta2 ** state["step"]
                    step_size = step_size * math.sqrt(bc2) / bc1
                lr_wd = group["lr"] * group["weight_decay"] if group["weight_decay"] > 0.0 else 0.0
                if "ranks" in group and grad.dim() == 2:
                    if not hasattr(self, "_tt2_plans"):
                        self._tt2_plans = {}           # per-parameter plans of the fused order-2 path (not part of state_dict)
                    stream = None
                    if n_side > 1:
                        if side is None:
                            side = self._side_streams(p.device, n_side)
                            forked = torch.cuda.current_stream(p.device).record_event()
                        k = tt_index % n_side
                        tt_index += 1
                        if k not in used:
                            side[k].wait_event(forked)
                            used.add(k)
                        stream = side[k]
                    # steady state: a live plan takes the step as one C-ABI call on the given stream (no stream switch, no
                    # shape arithmetic); everything else (first step, re-seeding, ranks without a plan) goes the long way
                    if self._plan_step(p, grad, state, group["ranks"], first, beta1, beta2, group["eps"], step_size, lr_wd,
                                       stream):
                        continue
                    if stream is not None:
                        with torch.cuda.stream(stream):
                            self._tt_update(p, grad, state, list(group["ranks"]), first, beta1, beta2, group["eps"], step_size,
                                            lr_wd, self._tt2_plans)
                    else:
                        self._tt_update(p, grad, state, list(group["ranks"]), first, beta1, beta2, group["eps"], step_size, lr_wd,
                                        self._tt2_plans)
                else:
                    self._dense_update(p, grad, state, first, beta1, beta2, group["eps"], step_size, lr_wd)
        if side is not None:
            cur = torch.cuda.current_stream(side[0].device)
            for k in used:
                cur.wait_event(side[k].record_event())
        return loss

    def _plan_step(self, p, grad, state, ranks, first, beta1, beta2, eps, step_size, lr_wd, stream) -> bool:
        """The step through an existing, live per-parameter plan (see _tt_update for how plans are made and re-seeded)."""
        if first or grad.dtype != p.dtype or not grad.is_contiguous():
            return False
        order = len(ranks) - 1
        plan = self._tt2_plans.get(p) if order == 2 else self._tt2_plans.get("_order_n", {}).get(p)
        if plan is None or plan.cur < 0 or not getattr(plan, "supported", True):
            return False
        if (plan.r != ranks[1]) if order == 2 else (plan.ranks != [int(r) for r in ranks]):
            return False
        tts = plan.tts[plan.cur]
        if state.get("exp_avg") is not tts[0] or state.get("exp_avg_sq") is not tts[1]:
            return False
        pd = p.data
        if not pd.is_contiguous():
            return False
        state["exp_avg_expr"] = tts[0].contract_expr                      # ttadam.py:73,81
        state["exp_avg_sq_expr"] = tts[1].contract_expr
        k = plan.step(pd, grad, beta1, beta2, eps, step_size, lr_wd, stream=stream)
        state["exp_avg"], state["exp_avg_sq"] = plan.tts[k]
        return True

    def _side_stream_count(self) -> int:
        """Streams the tensor-train parameters alternate on (SOWB_TT_STREAMS, default 4; 1 = everything on the caller's
        stream).  Only worth it with more than one tensor-train parameter."""
        import os
        n = int(os.environ.get("SOWB_TT_STREAMS", "4"))
        if n <= 1:
            return 1
        n_tt = sum(1 for g in self.param_groups if "ranks" in g for p in g["params"] if p.grad is not None and p.grad.dim() == 2)
        return n if n_tt > 1 else 1

    def _side_streams(self, device, n):
        cache = self.__dict__.setdefault("_tt_streams", {})
        key = (device.index, n)
        if key not in cache:
            cache[key] = [torch.cuda.Stream(device=device, priority=-1) for _ in range(n)]
        return cache[key]

    @staticmethod
    def _dense_update(p, grad, state, first, beta1, beta2, eps, step_size, lr_wd):
        if first:
            state["exp_avg"] = torch.zeros(grad.shape, dtype=torch.float32, device=grad.device)
            state["exp_avg_sq"] = torch.zeros(grad.shape, dtype=torch.float32, device=grad.device)
            state["exp_avg_expr"] = None
            state["exp_avg_sq_expr"] = None
        pd = p.data
        if not pd.is_contiguous():
            raise SowB200Error("TTAdam needs contiguous parameters")
        g = grad if grad.dtype == pd.dtype else grad.to(pd.dtype)
        ops.tt_adam_dense(pd, g, state["exp_avg"], state["exp_avg_sq"], beta1, beta2, eps, step_size, lr_wd)

    @staticmethod
    def _tt_update(p, grad, state, ranks, first, beta1, beta2, eps, step_size, lr_wd, plans=None):
        plans = {} if plans is None else plans
        order = len(ranks) - 1
        M, N = grad.shape
        mm = ceil(M ** (1 / order))
        nn_ = ceil(N ** (1 / order))
        pd = p.data
        if not pd.is_contiguous():
            raise SowB200Error("TTAdam needs contiguous parameters")
        g = grad if grad.dtype == pd.dtype else grad.to(pd.dtype)
        if not first:
            state["exp_avg_expr"] = state["exp_avg"].contract_expr          # ttadam.py:73,81
            state["exp_avg_sq_expr"] = state["exp_avg_sq"].contract_expr
        else:
            state["exp_avg_expr"] = None
            state["exp_avg_sq_expr"] = None
        if order == 2 and ranks[1] <= 64 and ranks[1] <= mm * nn_ and g.is_contiguous():
            # fused path, Adam + re-compression in one pass over p and g (the dense moments never reach HBM), through a
            # per-parameter plan: persistent core buffers (ping-pong), pre-built TensorTrain views, one C-ABI call
            plan = plans.get(p)
            if plan is not None and first:
                plan.cur = -1                                                   # state was reset: start from zero moments
            live = (plan is not None and not first and plan.cur >= 0 and state["exp_avg"] is plan.tts[plan.cur][0]
                    and state["exp_avg_sq"] is plan.tts[plan.cur][1])
            if plan is None or (plan.mm, plan.nn, plan.r) != (mm, nn_, ranks[1]) or not (first or live):
                plan = ops.TTAdam2Plan(pd.device, mm, nn_, ranks[1])
                plan.tts = []
                for k in range(2):
                    pair = []
                    for cores in plan.cores(k):
                        tt = TensorTrain(list(ranks), (mm, mm), (nn_, nn_), device=pd.device)
                        tt.cores = list(cores)
                        pair.append(tt)
                    plan.tts.append(pair)
                plans[p] = plan
                if not first:
                    # moments that did not come from this plan (loaded checkpoint, replaced by the caller): copy them in
                    P = mm * nn_
                    for b, key in enumerate(("exp_avg", "exp_avg_sq")):
                        plan.Q[0][b].copy_(state[key].cores[0].reshape(P, -1))
                        plan.R[0][b].copy_(state[key].cores[1].reshape(-1, P))
                    plan.cur = 0
            k = plan.step(pd, g, beta1, beta2, eps, step_size, lr_wd)
            state["exp_avg"], state["exp_avg_sq"] = plan.tts[k]
            return
        if order == 2:
            r = ranks[1]
            P = mm * nn_
            cm = cv = None
            if not first:
                tm, tv = state["exp_avg"], state["exp_avg_sq"]
                cm = (tm.cores[0].reshape(P, -1).contiguous(), tm.cores[1].reshape(-1, P).contiguous())
                cv = (tv.cores[0].reshape(P, -1).contiguous(), tv.cores[1].reshape(-1, P).contiguous())
            if r > P:
                raise RuntimeError(f"TT rank {r} exceeds the unfolding row count {P}")
            if r <= 64:
                # fused path: Adam + re-compression in one pass over p and g (dense moments never reach HBM)
                (Qm, Rm), (Qv, Rv) = ops.tt_adam2_step(pd, g, cm, cv, mm, nn_, r, beta1, beta2, eps, step_size, lr_wd, first)
                Q, R = (Qm, Qv), (Rm, Rv)
            else:
                m_new, v_new = ops.tt_adam_fused2(pd, g, cm, cv, mm, nn_, beta1, beta2, eps, step_size, lr_wd, first)
                L = torch.stack([m_new, v_new])                              # (2, P, P): one batched sweep
                Q = ops.thin_qr(L, r)
                R = ops.project(L, Q)
            for key, b in (("exp_avg", 0), ("exp_avg_sq", 1)):
                tt = TensorTrain(list(ranks), (mm, mm), (nn_, nn_), device=pd.device)
                tt.cores = [Q[b].reshape(1, mm, nn_, r), R[b].reshape(r, mm, nn_, 1)]
                state[key] = tt
            return
        if order > 2 and g.is_contiguous():
            # the whole step as one C-ABI call (reconstruction chains, interleaved Adam, one batched decomposition sweep)
            # through a per-parameter plan, like the order-2 path above
            nplans = plans.setdefault("_order_n", {})
            plan = nplans.get(p)
            if plan is not None and first:
                plan.cur = -1
            if plan is None or (plan.mm, plan.nn, plan.ranks) != (mm, nn_, [int(r) for r in ranks]):
                plan = ops.TTAdamNPlan(pd.device, mm, nn_, ranks)
                nplans[p] = plan
                if plan.supported:
                    plan.tts = []
                    for s_ in range(2):
                        pair = []
                        for b in range(2):
                            tt = TensorTrain(list(ranks), (mm,) * order, (nn_,) * order, device=pd.device)
                            tt.cores = plan.cores(s_, b)
                            pair.append(tt)
                        plan.tts.append(pair)
            if plan.supported:
                live = (not first and plan.cur >= 0 and state["exp_avg"] is plan.tts[plan.cur][0]
                        and state["exp_avg_sq"] is plan.tts[plan.cur][1])
                if not first and not live:
                    # moments that did not come from this plan (loaded checkpoint, replaced by the caller): copy them in
                    for b, key in enumerate(("exp_avg", "exp_avg_sq")):
                        for k in range(order):
                            plan.bufs[0][k][b].copy_(state[key].cores[k].reshape(-1))
                    plan.cur = 0
                k_out = plan.step(pd, g, beta1, beta2, eps, step_size, lr_wd)
                state["exp_avg"], state["exp_avg_sq"] = plan.tts[k_out]
                return
        # order > 2, op by op (ranks the one-call path does not take): the moments stay in the interleaved layout between the
        # reconstruction chain, the Adam kernel and the decomposition sweep (no de-interleave / interleave passes;
        # ttadam.py:71-84,113-115)
        total = (mm * nn_) ** order
        if first:
            m = torch.zeros((total,), dtype=torch.float32, device=pd.device)
            v = torch.zeros((total,), dtype=torch.float32, device=pd.device)
        else:
            m = reconstruct_interleaved(state["exp_avg"].cores)
            v = reconstruct_interleaved(state["exp_avg_sq"].cores)
        ops.tt_adam_interleaved(pd, g, m, v, mm, nn_, order, beta1, beta2, eps, step_size, lr_wd)
        for key, flat in (("exp_avg", m), ("exp_avg_sq", v)):
            tt = TensorTrain(list(ranks), (mm,) * order, (nn_,) * order, device=pd.device)
            tt._decompose_interleaved(flat)
            state[key] = tt


class TTRAdam(torch.optim.Optimizer):
    """Empty in the reference as well (tn_gradient/optimizer/ttadam.py:120-121)."""
    pass


class TTSGD(torch.optim.Optimizer):
    """tn_gradient/optimizer/ttsgd.py:8-86: SGD whose gradient / momentum live in TT format.  Compression and
    reconstruction use the CUDA kernels; the TT algebra in between is the (compat) PyTorch path of TensorTrain."""

    def __init__(self, params, lr: float = 1e-3, momentum: float = 0.9, dampening: float = 0,
                 weight_decay: float = 0, nesterov: bool = False):
        defaults = dict(lr=lr, momentum=momentum, dampening=dampening, weight_decay=weight_decay, nesterov=nesterov)
        super().__init__(params, defaults)

    @torch.no_grad()
    def step(self, closure: Callable = None):
        loss = None
        if closure is not None:
            loss = closure()
        for group in self.param_groups:
            for p in group["params"]:
                if p.grad is None:
                    continue
                grad = p.grad
                grad_shape = grad.shape
                if grad.is_sparse:
                    raise RuntimeError("TTSGD does not support sparse gradients, please consider SparseAdam instead")
                state = self.state[p]
                if "step" not in state:
                    state["step"] = 0
                use_tt = "ranks" in group
                d_p = TensorTrain.from_matrix(grad, ranks=list(group["ranks"]), padding=True) if use_tt else grad
                if group["weight_decay"] != 0:
                    if use_tt:
                        raise RuntimeError("TTSGD: weight_decay with TT gradients is unsupported "
                                           "(the reference calls a non-existent TensorTrain.add here, ttsgd.py:61)")
                    d_p = d_p.add(p, alpha=group["weight_decay"])
                if group["momentum"] != 0:
                    if "momentum_buffer" not in state:
                        buf = state["momentum_buffer"] = d_p.clone().detach()
                    else:
                        buf = state["momentum_buffer"]
                        buf = group["momentum"] * buf + (1 - group["dampening"]) * d_p
                    d_p = d_p + group["momentum"] * buf if group["nesterov"] else buf
                if use_tt:
                    d_p = d_p.to_matrix(grad_shape).to(p.dtype)
                p.add_(-group["lr"] * d_p)
                if group["weight_decay"] > 0.0:
                    p.add_(p, alpha=(-group["lr"] * group["weight_decay"]))
        return loss


def _check_state_dtype(param_dtype: torch.dtype, state_dtype) -> None:
    """FusedAdamW's moments: the parameter dtype (``None``), or fp32 for bf16 / fp16 parameters."""
    if state_dtype is None or state_dtype == param_dtype:
        return
    if state_dtype == torch.float32 and param_dtype in (torch.bfloat16, torch.float16):
        return
    raise SowB200Error(f"FusedAdamW: state_dtype {state_dtype} is not supported for {param_dtype} parameters "
                       "(None = the parameter dtype, or torch.float32 for bf16 / fp16 parameters)")


def _check_max_grad_norm(max_grad_norm):
    """FusedAdamW's per-group clipping threshold: ``None`` (no clipping) or a finite number > 0, returned as a float."""
    if max_grad_norm is None:
        return None
    if (isinstance(max_grad_norm, bool) or not isinstance(max_grad_norm, (int, float)) or not math.isfinite(max_grad_norm)
            or max_grad_norm <= 0):
        raise SowB200Error(f"FusedAdamW: max_grad_norm must be None or a finite float > 0, not {max_grad_norm!r}")
    return float(max_grad_norm)


class FusedAdamW(torch.optim.Optimizer):
    """Multi-tensor AdamW / Adam on one kernel launch per param group (SURVEY.md 8f rank 1).

    State layout is torch.optim.AdamW's (``state[p]["step"]`` tensor, ``exp_avg``, ``exp_avg_sq`` in the parameter
    dtype), so ``reset_optimizer`` (scripts/utils/training_utils.py:257-277), which REBINDS those tensors and zeroes
    ``step``, keeps working: pointers are re-resolved whenever a state tensor or gradient was rebound.

    ``capturable=True`` (as in torch.optim.AdamW): ``state[p]["step"]`` lives on the device -- one fp32 counter shared by
    the parameters of a group -- the kernels advance it and derive the bias corrections from it, and ``step()`` performs
    no host-side arithmetic on it, so the whole optimizer step can be captured in a CUDA graph and replayed.

    ``state_dtype`` (per group): ``torch.float32`` keeps ``exp_avg`` / ``exp_avg_sq`` in fp32 for bf16 / fp16
    parameters.  fp16 moments underflow ((1 - beta2) * g^2 is 0 below |g| ~ 8e-3), so training fp16 weights needs them.
    Moments that ``reset_optimizer`` rebinds in the parameter dtype are converted back (exactly: they are zeros) on the
    next step, and ``load_state_dict`` keeps them in fp32.

    torch.amp.GradScaler: ``step()`` takes the ``grad_scale`` / ``found_inf`` tensors GradScaler.step sets on the
    optimizer (``_step_supports_amp_scaling``).  The kernel unscales the gradients (and writes them back unscaled, as
    torch's fused AdamW does) and, for capturable groups, skips a step with found_inf on the device: no host sync, so a
    loss-scaled step can be captured in a CUDA graph.  Non-capturable groups read found_inf once on the host and leave
    parameters, moments and ``step`` untouched when it is set.

    ``max_grad_norm`` (per group): clip the group's gradients by their global 2-norm before the update, as
    ``torch.nn.utils.clip_grad_norm_(params, max_grad_norm)`` would, with the norm and the coefficient computed on the
    device (fp32 sums of squares, reduced in a fixed order: bit-reproducible, no host sync, graph-capturable).  The norm
    covers every gradient of the group and, under GradScaler, is that of the unscaled gradients; the clipped (and unscaled)
    gradients are written back to ``p.grad``.  ``grad_norm(group_index)`` returns the pre-clip norm of the last step.
    """

    _step_supports_amp_scaling = True

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, amsgrad=False,
                 decoupled=True, capturable=False, state_dtype=None, max_grad_norm=None):
        if amsgrad:
            raise SowB200Error("FusedAdamW: amsgrad is not implemented")
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=amsgrad, decoupled=decoupled,
                        capturable=capturable, state_dtype=state_dtype, max_grad_norm=max_grad_norm)
        super().__init__(params, defaults)
        self._tables = {}
        self._clip = {}                         # group index -> partials buffer, total_norm and clip_coef (device)

    def add_param_group(self, param_group):
        super().add_param_group(param_group)
        group = self.param_groups[-1]
        for p in group["params"]:
            _check_state_dtype(p.dtype, group.get("state_dtype"))
        _check_max_grad_norm(group.get("max_grad_norm"))

    def grad_norm(self, group_index: int):
        """The total 2-norm of group ``group_index``'s gradients before clipping, at its last clipped step (unscaled under
        GradScaler; what ``clip_grad_norm_`` returns), as a 0-dim fp32 device tensor that the next clipped step overwrites.
        No host sync.  ``None`` before the group's first clipped step."""
        st = self._clip.get(group_index)
        return None if st is None else st["total_norm"]

    def _clip_coef(self, gi, tables, max_norm, grad_scale):
        """Norm of the group's gradients over all its chunk tables ``(chunks, dtype)`` and the clip coefficient, into
        per-group device buffers that are reused from step to step (a captured step keeps their addresses; the partials
        are reallocated only when the row count changes, which rebuilds the chunk tables too)."""
        device = tables[0][0].device
        rows = max(1, sum(t.shape[0] for t, _ in tables))
        st = self._clip.get(gi)
        if st is None or st["total_norm"].device != device:
            st = {"total_norm": torch.zeros((), dtype=torch.float32, device=device),
                  "clip_coef": torch.ones((), dtype=torch.float32, device=device), "partials": None}
            self._clip[gi] = st
        if st["partials"] is None or st["partials"].numel() != rows:
            st["partials"] = torch.zeros(rows, dtype=torch.float32, device=device)
        ops.grad_norm(tables, st["partials"], st["total_norm"], st["clip_coef"], max_norm, grad_scale)
        return st["clip_coef"]

    def load_state_dict(self, state_dict):
        """torch's load_state_dict casts every floating-point state tensor to the parameter dtype (through
        ``Optimizer._process_value_according_to_param_policy``, called by class name, so a subclass cannot override it);
        the moments of groups with a ``state_dtype`` are taken from the checkpoint in that dtype instead."""
        keep = {}
        for group, saved in zip(self.param_groups, state_dict["param_groups"]):
            sdt = saved.get("state_dtype")
            if sdt is None:
                continue
            for p, pid in zip(group["params"], saved["params"]):
                st = state_dict["state"].get(pid, {})
                keep[p] = (sdt, {k: st[k] for k in ("exp_avg", "exp_avg_sq") if isinstance(st.get(k), torch.Tensor)})
        super().load_state_dict(state_dict)
        for p, (sdt, moments) in keep.items():
            for k, v in moments.items():
                self.state[p][k] = v.to(device=p.device, dtype=sdt)

    @staticmethod
    def _init_state(p, st, sdt):
        """Moments of dtype ``sdt``, created on the first step (``step`` None) or converted after reset_optimizer rebound
        them."""
        if len(st) == 0 or "exp_avg" not in st:
            st["step"] = None
            st["exp_avg"] = torch.zeros_like(p, dtype=sdt, memory_format=torch.preserve_format)
            st["exp_avg_sq"] = torch.zeros_like(p, dtype=sdt, memory_format=torch.preserve_format)
        for k in ("exp_avg", "exp_avg_sq"):
            if st[k].dtype != sdt:
                st[k] = st[k].to(sdt)

    @staticmethod
    def _grad(p, grad_scale, clip=False):
        if p.grad.dtype == p.dtype:
            return p.grad
        if grad_scale is not None:
            raise SowB200Error("FusedAdamW: loss-scaled gradients must have the parameter dtype (they are unscaled in place)")
        if clip:
            raise SowB200Error("FusedAdamW: the gradients of a max_grad_norm group must have the parameter dtype (they are "
                               "clipped in place)")
        return p.grad.to(p.dtype)

    def _step_capturable(self, gi, group, grad_scale=None, found_inf=None):
        """One device counter per (group, dtype); parameters whose ``step`` was rebound by reset_optimizer (a fresh zero
        tensor) are folded back onto a shared counter restarted from that value."""
        beta1, beta2 = group["betas"]
        gsdt = group.get("state_dtype")
        max_norm = _check_max_grad_norm(group.get("max_grad_norm"))
        by_dtype = {}
        for p in group["params"]:
            if p.grad is None:
                continue
            if not p.is_cuda:
                raise SowB200Error("FusedAdamW needs CUDA parameters (no CPU fallback)")
            st = self.state[p]
            self._init_state(p, st, gsdt or p.dtype)
            g = self._grad(p, grad_scale, max_norm is not None)
            by_dtype.setdefault(p.dtype, []).append((p, g, st))
        launches = []
        for dtype, items in by_dtype.items():
            ckey = ("counter", gi, dtype)
            counter = self._tables.get(ckey)
            steps = [st["step"] for _, _, st in items]
            if counter is None or any(s is not counter for s in steps):
                # (re)build the shared counter: happens outside graph capture (first step, or the step after a reset)
                start = 0.0
                for s_ in steps:
                    if s_ is not None and s_ is not counter:
                        start = float(s_)                       # rebound by reset_optimizer: restart from its value
                        break
                else:
                    start = float(counter) if counter is not None else 0.0
                counter = torch.full((1,), start, dtype=torch.float32, device=items[0][0].device)
                self._tables[ckey] = counter
                for _, _, st in items:
                    st["step"] = counter
            sig = tuple((p.data_ptr(), g.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(), p.numel())
                        for p, g, st in items)
            key = (gi, dtype, len(items))
            cached = self._tables.get(key)
            if cached is None or cached[0] != sig:
                cached = (sig, ops.build_adam_chunks([p.data for p, _, _ in items], [g for _, g, _ in items],
                                                     [st["exp_avg"] for _, _, st in items],
                                                     [st["exp_avg_sq"] for _, _, st in items]))
                self._tables[key] = cached
            launches.append((dtype, items[0][2]["exp_avg"].dtype, counter, cached[1]))
        # clipping: the norm spans every dtype bucket of the group, so it is complete before the first update
        clip = (self._clip_coef(gi, [(t, d) for d, _, _, t in launches], max_norm, grad_scale)
                if max_norm is not None and launches else None)
        for dtype, sdt, counter, table in launches:
            if clip is not None:
                ops.adam_multi_clip(table, dtype, sdt, group["lr"], beta1, beta2, group["eps"], group["weight_decay"],
                                    group["decoupled"], clip, step_dev=counter, grad_scale=grad_scale, found_inf=found_inf)
            elif sdt == dtype and grad_scale is None and found_inf is None:
                ops.adam_multi_dev(table, dtype, group["lr"], beta1, beta2, group["eps"], group["weight_decay"],
                                   counter, group["decoupled"])
            else:
                ops.adam_multi_amp(table, dtype, sdt, group["lr"], beta1, beta2, group["eps"], group["weight_decay"],
                                   group["decoupled"], step_dev=counter, grad_scale=grad_scale, found_inf=found_inf)

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        # set by torch.amp.GradScaler.step for the duration of this call; grad_scale is None after an explicit unscale_
        grad_scale = getattr(self, "grad_scale", None)
        found_inf = getattr(self, "found_inf", None)
        skip = None                             # found_inf read on the host, once, for the non-capturable groups
        for gi, group in enumerate(self.param_groups):
            if group.get("capturable", False):
                self._step_capturable(gi, group, grad_scale, found_inf)
                continue
            if found_inf is not None:
                if skip is None:
                    skip = bool(found_inf.item())
                if skip:
                    continue
            buckets = {}
            gsdt = group.get("state_dtype")
            max_norm = _check_max_grad_norm(group.get("max_grad_norm"))
            for p in group["params"]:
                if p.grad is None:
                    continue
                if not p.is_cuda:
                    raise SowB200Error("FusedAdamW needs CUDA parameters (no CPU fallback)")
                st = self.state[p]
                self._init_state(p, st, gsdt or p.dtype)
                if st["step"] is None:
                    st["step"] = torch.zeros((), dtype=torch.float32)
                st["step"] += 1
                g = self._grad(p, grad_scale, max_norm is not None)
                buckets.setdefault((int(st["step"]), p.dtype), []).append((p, g, st["exp_avg"], st["exp_avg_sq"]))
            beta1, beta2 = group["betas"]
            launches = []
            for (step, dtype), items in buckets.items():
                sig = tuple((p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel()) for p, g, m, v in items)
                key = (gi, dtype, len(items))
                cached = self._tables.get(key)
                if cached is None or cached[0] != sig:
                    ps, gs, ms, vs = zip(*items)
                    cached = (sig, ops.build_adam_chunks([p.data for p in ps], list(gs), list(ms), list(vs)))
                    self._tables[key] = cached
                launches.append((step, dtype, items[0][2].dtype, cached[1]))
            clip = (self._clip_coef(gi, [(t, d) for _, d, _, t in launches], max_norm, grad_scale)
                    if max_norm is not None and launches else None)
            for step, dtype, sdt, table in launches:
                if clip is not None:
                    ops.adam_multi_clip(table, dtype, sdt, group["lr"], beta1, beta2, group["eps"], group["weight_decay"],
                                        group["decoupled"], clip, 1.0 - beta1 ** step, 1.0 - beta2 ** step,
                                        grad_scale=grad_scale)
                elif sdt == dtype and grad_scale is None:
                    ops.adam_multi(table, dtype, group["lr"], beta1, beta2, group["eps"], group["weight_decay"],
                                   1.0 - beta1 ** step, 1.0 - beta2 ** step, group["decoupled"])
                else:
                    ops.adam_multi_amp(table, dtype, sdt, group["lr"], beta1, beta2, group["eps"],
                                       group["weight_decay"], group["decoupled"], 1.0 - beta1 ** step, 1.0 - beta2 ** step,
                                       grad_scale=grad_scale)
        return loss
