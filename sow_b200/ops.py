"""torch-level wrappers over the C ABI (include/sow_b200.h).

PyTorch is plumbing here: it owns device memory and streams.  All device math happens inside libsow_b200.so.
Every wrapper requires CUDA tensors and raises otherwise -- there is no CPU path.
"""
from __future__ import annotations

import ctypes
import os
import threading
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import SOWB_BF16, SOWB_F16, SOWB_F32, MergeEntry, SowB200Error, check

# count of kernel-launching C-ABI calls, for bench.py's `gpu_launches` accounting (approximate kernels per call
# are listed next to each call site)
launch_counter = {"kernels": 0}

_ws_lock = threading.Lock()
_workspaces = {}


def _stream_ptr(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _p(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise SowB200Error(
                "sow_b200 ops need CUDA tensors: the SoW hot path is implemented as sm_100a kernels only "
                "(no CPU fallback).  Move the module / tensors to a B200 device."
            )


def _dtype_code(dt: torch.dtype) -> int:
    if dt == torch.bfloat16:
        return SOWB_BF16
    if dt == torch.float32:
        return SOWB_F32
    if dt == torch.float16:
        return SOWB_F16
    raise SowB200Error(f"unsupported dtype {dt}")


def _tt_dtype_code(dt: torch.dtype) -> int:
    """dtype code of the tensor-train entry points, which take bf16 and fp32 only."""
    if dt not in (torch.bfloat16, torch.float32):
        raise SowB200Error(f"unsupported dtype {dt}")
    return _dtype_code(dt)


def workspace(device: torch.device, nbytes: int, stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
    """Per-(device, stream) scratch buffer, grown on demand.  Kernels that share a stream are serialised, so one
    buffer per stream is enough; a bigger request replaces the buffer (the old one stays alive until the work
    queued on it finishes because the caching allocator is stream-ordered).  ``stream``: the stream the caller will
    launch on when that is not the current one (the buffer is then allocated under it)."""
    sp = stream.cuda_stream if stream is not None else torch.cuda.current_stream(device).cuda_stream
    key = (device.index if device.index is not None else torch.cuda.current_device(), sp)
    with _ws_lock:
        buf = _workspaces.get(key)
        if buf is None or buf.numel() < nbytes:
            if stream is not None:
                with torch.cuda.stream(stream):
                    buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
            else:
                buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
            _workspaces[key] = buf
    return buf


def rank_pad(r: int) -> int:
    return (r + 63) // 64 * 64


# Widest concatenated padded rank R = sum_i rank_pad(r_i) one sow_group_fwd / sow_group_bwd call takes: the skinny GEMM
# keeps one scale per 64 columns of t_cat in a table of kMaxAlphaBlocks = 16 entries (csrc/gemm.cuh), and group_layout
# (csrc/linear.cu) rejects anything wider.
MAX_GROUP_RANK = 64 * 16


def group_rank_fits(ranks) -> bool:
    """True when projections of these ranks can run as ONE group call (sum of their padded ranks <= MAX_GROUP_RANK)."""
    return sum(rank_pad(int(r)) for r in ranks) <= MAX_GROUP_RANK


# ---------------------------------------------------------------------------------------------------------
# SoW linear
# ---------------------------------------------------------------------------------------------------------

_HALF_NAMES = {torch.bfloat16: "bf16", torch.float16: "fp16"}


def _check_bf16c(name: str, t: Optional[torch.Tensor], dt: torch.dtype = torch.bfloat16):
    if t is not None and (t.dtype != dt or not t.is_contiguous()):
        raise SowB200Error(f"{name} must be a contiguous {_HALF_NAMES[dt]} tensor")


def split_f32(t: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """fp32 tensor -> (hi, lo) bf16 pieces with t ~ hi + lo (relative error 2^-17): the operands of the bf16x3 tensor-core
    products that give fp32 modules an fp32-faithful path (include/sow_b200.h: sow_split_bf16x2)."""
    _require_cuda(t)
    if t.dtype != torch.float32 or not t.is_contiguous():
        raise SowB200Error("split_f32 expects a contiguous fp32 tensor")
    hi = torch.empty(t.shape, dtype=torch.bfloat16, device=t.device)
    lo = torch.empty(t.shape, dtype=torch.bfloat16, device=t.device)
    check(_lib.load().sow_split_bf16x2(_p(t), _p(hi), _p(lo), t.numel(), _stream_ptr(t.device)), "sow_split_bf16x2")
    launch_counter["kernels"] += 1
    return hi, lo


def group_fwd(x: torch.Tensor, members, x_lo: Optional[torch.Tensor] = None):
    """Forward of a group of SoW projections that read the same x (T,in) bf16 or fp16 contiguous (include/sow_b200.h:
    sow_group_fwd).  members: (W (in,out) or None, A (in,r), B (r,out), bias or None, scale[, W_lo]), all of x's dtype.
    With ``x_lo`` (SOWB_F32 mode) x / x_lo and W / W_lo are the bf16 pieces of fp32 operands, bias is fp32 and the outputs
    are fp32.  Returns ([y_i (T,out_i)], A_cat (in,R), t_cat (T,R)); A_cat / t_cat (x's dtype) are what autograd saves for
    group_bwd."""
    lib = _lib.load()
    n = len(members)
    T, fin = x.shape
    f32 = x_lo is not None
    hdt = torch.float16 if (x.dtype == torch.float16 and not f32) else torch.bfloat16
    _require_cuda(x, x_lo)
    _check_bf16c("x", x, hdt)
    _check_bf16c("x_lo", x_lo)
    arr = (_lib.GroupMember * n)()
    ys = []
    R = 0
    keep = []
    for i, mem in enumerate(members):
        W, A, B, bias, scale = mem[:5]
        W_lo = mem[5] if len(mem) > 5 else None
        _require_cuda(W, A, B, bias, W_lo)
        for nm, t in (("W", W), ("A", A), ("B", B), ("W_lo", W_lo)):
            _check_bf16c(nm, t, hdt)
        if f32:
            if bias is not None and (bias.dtype != torch.float32 or not bias.is_contiguous()):
                raise SowB200Error("group_fwd: fp32 mode needs a contiguous fp32 bias")
            if (W is None) != (W_lo is None):
                raise SowB200Error("group_fwd: fp32 mode needs both pieces of W")
        else:
            _check_bf16c("bias", bias, hdt)
        r, fout = B.shape
        if A.shape != (fin, r) or (W is not None and tuple(W.shape) != (fin, fout)):
            raise SowB200Error("group_fwd: shape mismatch")
        y = torch.empty((T, fout), dtype=torch.float32 if f32 else hdt, device=x.device)
        ys.append(y)
        arr[i].W, arr[i].W_lo, arr[i].A, arr[i].B, arr[i].bias = _p(W), _p(W_lo), _p(A), _p(B), _p(bias)
        arr[i].y = _p(y)
        arr[i].out_features, arr[i].r, arr[i].scale = fout, r, float(scale)
        R += rank_pad(r)
        keep.append((W, W_lo, A, B, bias))
    A_cat = torch.empty((fin, R), dtype=hdt, device=x.device)
    t_cat = torch.empty((T, R), dtype=hdt, device=x.device)
    rc = lib.sow_group_fwd(_p(x), _p(x_lo), arr, n, _p(A_cat), _p(t_cat), T, fin, SOWB_F32 if f32 else _dtype_code(hdt),
                           _stream_ptr(x.device))
    check(rc, "sow_group_fwd")
    launch_counter["kernels"] += 2 + n
    return ys, A_cat, t_cat


def group_bwd(x: torch.Tensor, A_cat: torch.Tensor, t_cat: torch.Tensor, members, need_dx: bool, f32: bool = False):
    """Backward of a group (sow_group_bwd).  members: (W or None, B (r,out), dy (T,out), scale, dA_dst, dB_dst,
    want_dbias[, W_lo, dy_lo]) where dA_dst / dB_dst are None (not needed), True (allocate) or a preallocated contiguous
    tensor of the gradient's shape and the 16-bit dtype (e.g. a view into a flat gradient bucket) that the kernels write in
    place.  The 16-bit dtype is x's: bf16, or fp16 (every operand and gradient fp16).
    ``f32``: W / W_lo and dy / dy_lo are bf16 pieces of fp32 operands and dx is fp32.
    Returns (dx or None, [dA_i], [dB_i], [dbias_i])."""
    lib = _lib.load()
    n = len(members)
    T, fin = x.shape
    dev = x.device
    hdt = torch.float16 if (x.dtype == torch.float16 and not f32) else torch.bfloat16
    _check_bf16c("x", x, hdt)
    _check_bf16c("A_cat", A_cat, hdt)
    _check_bf16c("t_cat", t_cat, hdt)
    R = t_cat.shape[1]
    arr = (_lib.GroupMember * n)()
    dAs, dBs, dbs = [], [], []
    keep = []
    for i, mem in enumerate(members):
        W, B, dy, scale, dA_dst, dB_dst, want_dbias = mem[:7]
        W_lo = mem[7] if len(mem) > 7 else None
        dy_lo = mem[8] if len(mem) > 8 else None
        _require_cuda(W, B, dy, W_lo, dy_lo)
        for nm, t in (("W", W), ("B", B), ("dy", dy), ("W_lo", W_lo), ("dy_lo", dy_lo)):
            _check_bf16c(nm, t, hdt)
        r, fout = B.shape
        if tuple(dy.shape) != (T, fout):
            raise SowB200Error("group_bwd: dy shape mismatch")

        def out_buf(dst, shape):
            if dst is None:
                return None
            if dst is True:
                return torch.empty(shape, dtype=hdt, device=dev)
            if tuple(dst.shape) != tuple(shape) or dst.dtype != hdt or not dst.is_contiguous() or dst.device != dev:
                raise SowB200Error(f"group_bwd: gradient destination must be a contiguous {_HALF_NAMES[hdt]} tensor of the "
                                   "gradient's shape")
            return dst.detach()          # fresh alias of the same memory: AccumulateGrad can adopt it as param.grad
        dA = out_buf(dA_dst, (fin, r))
        dB = out_buf(dB_dst, (r, fout))
        db = torch.empty((fout,), dtype=hdt, device=dev) if want_dbias else None
        dAs.append(dA)
        dBs.append(dB)
        dbs.append(db)
        arr[i].W, arr[i].W_lo, arr[i].B, arr[i].dy, arr[i].dy_lo = _p(W), _p(W_lo), _p(B), _p(dy), _p(dy_lo)
        arr[i].A = _p(A_cat)       # not read by the backward (A_cat carries the factors); must be non-null
        arr[i].dA, arr[i].dB, arr[i].dbias = _p(dA), _p(dB), _p(db)
        arr[i].out_features, arr[i].r, arr[i].scale = fout, r, float(scale)
        keep.append((W, W_lo, B, dy, dy_lo))
    dt_cat = torch.empty((T, R), dtype=hdt, device=dev)
    dx = torch.empty((T, fin), dtype=torch.float32 if f32 else hdt, device=dev) if need_dx else None
    nws = lib.sow_group_workspace_bytes(_lib.OP_LINEAR_BWD, T, fin, arr, n)
    ws = workspace(dev, nws)
    rc = lib.sow_group_bwd(_p(x), _p(A_cat), _p(t_cat), arr, n, _p(dt_cat), _p(dx), T, fin, SOWB_F32 if f32 else _dtype_code(hdt),
                           _p(ws), ws.numel(), _stream_ptr(dev))
    check(rc, "sow_group_bwd")
    # K2 (one launch when the members share a cluster size, else n) + split-K dA + finalize + dX + colsum pairs
    uniform = len({(m[1].shape[1], rank_pad(m[1].shape[0])) for m in members}) == 1
    launch_counter["kernels"] += (1 if uniform else n) + 2 + (1 if need_dx else 0) + 2 * sum(1 for d in dbs if d is not None)
    return dx, dAs, dBs, dbs


def linear_fwd(x: torch.Tensor, W: Optional[torch.Tensor], A: torch.Tensor, B: torch.Tensor,
               bias: Optional[torch.Tensor], scale: float) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Single projection = group of one.  Returns (y (T,out), A_pad (in,r_pad), t (T,r_pad))."""
    _require_cuda(x, W, A, B, bias)
    ys, A_cat, t_cat = group_fwd(x, [(W, A, B, bias, scale)])
    return ys[0], A_cat, t_cat


def linear_bwd(dy, x, A_pad, t, W, B, scale: float, want_dbias: bool, need_dx: bool = True):
    """Returns (dx (T,in) or None, dA (in,r), dB (r,out), dbias or None)."""
    dx, dAs, dBs, dbs = group_bwd(x, A_pad, t, [(W, B, dy, scale, True, True, want_dbias)], need_dx)
    return dx, dAs[0], dBs[0], dbs[0]


# ---------------------------------------------------------------------------------------------------------
# grouped merge
# ---------------------------------------------------------------------------------------------------------

def merge_grouped(items: Sequence[Tuple[torch.Tensor, Optional[torch.Tensor], torch.Tensor, torch.Tensor, float]]):
    """items: (W_out (in,out), W_prev or None, A (in,r), B (r,out), scale), all CUDA contiguous on one device and all
    of ONE dtype: bf16 or fp16 (tcgen05 path, one launch per 64-wide rank chunk for the whole list) or fp32 (exact fp32
    path)."""
    if not items:
        return
    lib = _lib.load()
    dev = items[0][0].device
    n = len(items)
    dt = items[0][0].dtype
    if dt not in (torch.bfloat16, torch.float16, torch.float32):
        raise SowB200Error(f"merge_grouped: unsupported dtype {dt}")
    arr = (MergeEntry * n)()
    for i, (W, Wp, A, B, s) in enumerate(items):
        _require_cuda(W, Wp, A, B)
        for tname, tt in (("W", W), ("W_prev", Wp), ("A", A), ("B", B)):
            if tt is not None and (tt.dtype != dt or not tt.is_contiguous()):
                raise SowB200Error(f"merge_grouped: {tname} must be a contiguous {dt} tensor")
        fin, r = A.shape
        fout = B.shape[1]
        if tuple(W.shape) != (fin, fout) or B.shape[0] != r:
            raise SowB200Error("merge_grouped: shape mismatch")
        arr[i].W = W.data_ptr()
        arr[i].W_prev = Wp.data_ptr() if Wp is not None else None
        arr[i].A = A.data_ptr()
        arr[i].B = B.data_ptr()
        arr[i].in_features, arr[i].out_features, arr[i].r = fin, fout, r
        arr[i].scale = float(s)
    stride = lib.sow_merge_table_stride()
    table = workspace(dev, n * stride + 256)
    base = table.data_ptr()
    aligned = (base + 127) // 128 * 128
    rc = lib.sow_merge_grouped(arr, n, _dtype_code(dt), ctypes.c_void_p(aligned), table.numel() - (aligned - base),
                               _stream_ptr(dev))
    check(rc, "sow_merge_grouped")
    launch_counter["kernels"] += max((a[2].shape[1] + 63) // 64 for a in items)


# ---------------------------------------------------------------------------------------------------------
# thin QR / TT pieces
# ---------------------------------------------------------------------------------------------------------

def thin_qr(X: torch.Tensor, r: int) -> torch.Tensor:
    """Orthonormal basis Q (.., m, r) of the first r columns of X (.., m, n) fp32; batched over leading dims."""
    _require_cuda(X)
    if X.dtype != torch.float32:
        raise SowB200Error("thin_qr expects fp32 input")
    lib = _lib.load()
    squeeze = X.dim() == 2
    Xb = X.unsqueeze(0) if squeeze else X
    if Xb.dim() != 3 or Xb.stride(2) != 1 or Xb.stride(1) < Xb.shape[2]:
        Xb = Xb.contiguous()
    b, m, n = Xb.shape
    Q = torch.empty((b, m, r), dtype=torch.float32, device=X.device)
    # scratch: for r <= 64 two Cholesky blocks per matrix (the second for the CholeskyQR2 pass of ill-conditioned
    # inputs), one flag per matrix and the fp64 Gram partials; above that the column-major Gram-Schmidt work copy
    if r > m:
        raise SowB200Error(f"thin_qr: rank {r} exceeds the row count {m} (the reference fails here too: tt.py:135)")
    work = workspace(X.device, lib.sow_thin_qr_workspace_bytes(m, r, b))
    rc = lib.sow_thin_qr(_p(Xb), Xb.stride(0), Xb.stride(1), _p(Q), m * r, m, r, b, _p(work), work.numel(),
                         _stream_ptr(X.device))
    check(rc, "sow_thin_qr")
    launch_counter["kernels"] += 1
    return Q[0] if squeeze else Q


def project(L: torch.Tensor, Q: torch.Tensor) -> torch.Tensor:
    """R (.., r, n) = Q^T (.., m, r) . L (.., m, n), fp32."""
    _require_cuda(L, Q)
    lib = _lib.load()
    squeeze = L.dim() == 2
    Lb = (L.unsqueeze(0) if squeeze else L).contiguous()
    Qb = (Q.unsqueeze(0) if squeeze else Q).contiguous()
    b, m, n = Lb.shape
    r = Qb.shape[2]
    R = torch.empty((b, r, n), dtype=torch.float32, device=L.device)
    ws_bytes = lib.tt_project_workspace_bytes(m, n, r, b)      # split partials, summed in split order (no atomics)
    ws = workspace(L.device, ws_bytes) if ws_bytes else None
    rc = lib.tt_project(_p(Lb), m * n, _p(Qb), m * r, _p(R), r * n, m, n, r, b, _p(ws) if ws is not None else None,
                        ws_bytes, _stream_ptr(L.device))
    check(rc, "tt_project")
    launch_counter["kernels"] += 2
    return R[0] if squeeze else R


def interleave(src: torch.Tensor, mm: int, nn: int, order: int) -> torch.Tensor:
    """(M,N) bf16/fp32 -> zero-padded, (i1,o1,...,id,od)-ordered fp32 flat tensor of (mm*nn)^order elements."""
    _require_cuda(src)
    lib = _lib.load()
    src = src.contiguous()
    M, N = src.shape
    out = torch.empty(((mm * nn) ** order,), dtype=torch.float32, device=src.device)
    rc = lib.tt_interleave(_p(src), M, N, mm, nn, order, _p(out), _tt_dtype_code(src.dtype), _stream_ptr(src.device))
    check(rc, "tt_interleave")
    launch_counter["kernels"] += 1
    return out


def deinterleave(src: torch.Tensor, M: int, N: int, mm: int, nn: int, order: int, dtype=torch.float32) -> torch.Tensor:
    _require_cuda(src)
    lib = _lib.load()
    src = src.contiguous()
    out = torch.empty((M, N), dtype=dtype, device=src.device)
    rc = lib.tt_deinterleave(_p(src), M, N, mm, nn, order, _p(out), _tt_dtype_code(dtype), _stream_ptr(src.device))
    check(rc, "tt_deinterleave")
    launch_counter["kernels"] += 1
    return out


def decompose2(src: torch.Tensor, mm: int, nn: int, r: int):
    """Order-2 TT of a (M,N) bf16/fp32 matrix without materialising the interleaved unfolding: returns
    (Q (P,r), R (r,P)) fp32 with P = mm*nn (include/sow_b200.h: tt_gather2 / sow_thin_qr / tt_project2)."""
    _require_cuda(src)
    lib = _lib.load()
    src = src.contiguous()
    M, N = src.shape
    P = mm * nn
    dt = _tt_dtype_code(src.dtype)
    st = _stream_ptr(src.device)
    ncols = min(P, (r + 7) // 8 * 8)
    X = torch.empty((P, ncols), dtype=torch.float32, device=src.device)
    check(lib.tt_gather2(_p(src), M, N, mm, nn, _p(X), ncols, dt, st), "tt_gather2")
    Q = thin_qr(X, r)
    R = torch.empty((r, P), dtype=torch.float32, device=src.device)
    ws_bytes = lib.tt_project2_workspace_bytes(mm, nn, r)
    ws = workspace(src.device, ws_bytes) if ws_bytes else None
    check(lib.tt_project2(_p(src), M, N, mm, nn, _p(Q), _p(R), r, dt, _p(ws) if ws is not None else None, ws_bytes, st),
          "tt_project2")
    launch_counter["kernels"] += 3
    return Q, R


def reconstruct2(G1: torch.Tensor, G2: torch.Tensor, M: int, N: int, mm: int, nn: int, dtype=torch.float32) -> torch.Tensor:
    """(M,N) window of the order-2 TT (G1 (P,r), G2 (r,P)), written de-interleaved in one pass."""
    _require_cuda(G1, G2)
    lib = _lib.load()
    G1 = G1.contiguous()
    G2 = G2.contiguous()
    r = G1.shape[1]
    out = torch.empty((M, N), dtype=dtype, device=G1.device)
    check(lib.tt_reconstruct2(_p(G1), _p(G2), r, _p(out), M, N, mm, nn, _tt_dtype_code(dtype), _stream_ptr(G1.device)),
          "tt_reconstruct2")
    launch_counter["kernels"] += 1
    return out


def matmul_rk(A: torch.Tensor, B: torch.Tensor) -> torch.Tensor:
    """fp32 C = A (m,r) . B (r,n) for small r."""
    _require_cuda(A, B)
    lib = _lib.load()
    A = A.contiguous()
    B = B.contiguous()
    m, r = A.shape
    n = B.shape[1]
    C = torch.empty((m, n), dtype=torch.float32, device=A.device)
    rc = lib.tt_matmul_rk(_p(A), _p(B), _p(C), m, n, r, _stream_ptr(A.device))
    check(rc, "tt_matmul_rk")
    launch_counter["kernels"] += 1
    return C


def tt_adam_fused2(p, g, cores_m, cores_v, mm, nn, beta1, beta2, eps, step_size, lr_wd, first_step):
    """Order-2 fused reconstruct + Adam.  Returns (m_new, v_new) as (P,P) fp32 interleaved matrices, P = mm*nn."""
    _require_cuda(p, g)
    lib = _lib.load()
    M, N = p.shape
    P = mm * nn
    m_out = torch.empty((P, P), dtype=torch.float32, device=p.device)
    v_out = torch.empty((P, P), dtype=torch.float32, device=p.device)
    if first_step:
        G1m = G2m = G1v = G2v = None
        r = 1
    else:
        G1m, G2m = cores_m
        G1v, G2v = cores_v
        r = G1m.shape[-1]
    g = g.contiguous()
    rc = lib.tt_adam_fused2(_p(p), _p(g), _p(G1m), _p(G2m), _p(G1v), _p(G2v), r, _p(m_out), _p(v_out), M, N, mm, nn,
                            float(beta1), float(beta2), float(eps), float(step_size), float(lr_wd),
                            1 if first_step else 0, _tt_dtype_code(p.dtype), _stream_ptr(p.device))
    check(rc, "tt_adam_fused2")
    launch_counter["kernels"] += 1
    return m_out, v_out


def tt_adam2_step(p, g, cores_m, cores_v, mm, nn, r, beta1, beta2, eps, step_size, lr_wd, first_step):
    """Order-2 TT-Adam with the re-compression fused in; the dense moments never reach HBM.  ONE C-ABI call
    (tt_adam2_step: head -> thin QR -> fused update + projection, on the tensor cores above rank 16).  Returns the new
    cores ((Qm (P,r), Rm (r,P)), (Qv, Rv))."""
    _require_cuda(p, g)
    lib = _lib.load()
    M, N = p.shape
    P = mm * nn
    dev = p.device
    if first_step:
        G1m = G2m = G1v = G2v = None
    else:
        G1m, G2m = cores_m
        G1v, G2v = cores_v
    g = g.contiguous()
    Q = torch.empty((2, P, r), dtype=torch.float32, device=dev)
    R = torch.empty((2, r, P), dtype=torch.float32, device=dev)
    ws = workspace(dev, lib.tt_adam2_workspace_bytes(mm, nn))
    rc = lib.tt_adam2_step(_p(p), _p(g), _p(G1m), _p(G2m), _p(G1v), _p(G2v), r, _p(Q[0]), _p(Q[1]), _p(R[0]), _p(R[1]),
                           M, N, mm, nn, float(beta1), float(beta2), float(eps), float(step_size), float(lr_wd),
                           1 if first_step else 0, _tt_dtype_code(p.dtype), _p(ws), ws.numel(), _stream_ptr(dev))
    check(rc, "tt_adam2_step")
    launch_counter["kernels"] += 8
    return (Q[0], R[0]), (Q[1], R[1])


class TTAdam2Plan:
    """Persistent state of the fused order-2 TT-Adam step of ONE parameter: two sets of cores (Q (2,P,r) | R (2,r,P), one
    for each moment) used ping-pong -- a step reads set ``cur`` and writes the other one -- with their C pointers built
    once.  A step is then one C-ABI call and no allocation; the host cost per parameter drops from ~100 us (tensor
    allocation, reshapes, TensorTrain construction, argument marshalling) to the ~30 us of the launches themselves,
    which is what keeps a many-parameter TTAdam.step GPU-bound.  ``cores(k)`` are views, so a TensorTrain built on a
    set is overwritten two steps later (the reference allocates new cores every step, ttadam.py:113-115)."""

    def __init__(self, device, mm: int, nn: int, r: int):
        lib = _lib.load()
        self.mm, self.nn, self.r, self.P = mm, nn, r, mm * nn
        P = self.P
        self.Q = [torch.empty((2, P, r), dtype=torch.float32, device=device) for _ in range(2)]
        self.R = [torch.empty((2, r, P), dtype=torch.float32, device=device) for _ in range(2)]
        self._ptr = [[_p(self.Q[k][0]), _p(self.R[k][0]), _p(self.Q[k][1]), _p(self.R[k][1])] for k in range(2)]
        self.ws_bytes = lib.tt_adam2_workspace_bytes(mm, nn)
        self.device = device
        self.cur = -1                      # set holding the current cores (-1: none yet)

    def cores(self, k: int):
        """((G1m (1,mm,nn,r), G2m (r,mm,nn,1)), (G1v, G2v)) of set k, as views."""
        mm, nn, r = self.mm, self.nn, self.r
        return tuple((self.Q[k][b].reshape(1, mm, nn, r), self.R[k][b].reshape(r, mm, nn, 1)) for b in range(2))

    def step(self, p, g, beta1, beta2, eps, step_size, lr_wd, stream=None) -> int:
        """One update of p from g (on ``stream`` when given, else on the current stream); returns the index of the core
        set that now holds the moments."""
        lib = _lib.load()
        first = self.cur < 0
        out = 0 if first else 1 - self.cur
        g1m, g2m, g1v, g2v = (None, None, None, None) if first else self._ptr[self.cur]
        qm, rm, qv, rv = self._ptr[out]
        M, N = p.shape
        ws = workspace(self.device, self.ws_bytes, stream)
        sp = ctypes.c_void_p(stream.cuda_stream) if stream is not None else _stream_ptr(self.device)
        rc = lib.tt_adam2_step(_p(p), _p(g), g1m, g2m, g1v, g2v, self.r, qm, qv, rm, rv, M, N, self.mm, self.nn,
                               float(beta1), float(beta2), float(eps), float(step_size), float(lr_wd), 1 if first else 0,
                               _tt_dtype_code(p.dtype), _p(ws), ws.numel(), sp)
        check(rc, "tt_adam2_step")
        launch_counter["kernels"] += 8
        self.cur = out
        return out


def decompose_nd(src: torch.Tensor, mm: int, nn: int, ranks):
    """Order >= 3 TT of a (M,N) bf16/fp32 matrix in one C-ABI call (tt_decompose_nd).  Returns the cores as
    (r_k, mm, nn, r_{k+1}) fp32 tensors, or None when the entry point does not take the ranks (caller: op-by-op sweep)."""
    _require_cuda(src)
    lib = _lib.load()
    ranks = [int(r) for r in ranks]
    order = len(ranks) - 1
    ranks_c = (ctypes.c_int * len(ranks))(*ranks)
    ws_bytes = lib.tt_nd_workspace_bytes(mm, nn, order, ranks_c)
    if ws_bytes == 0:
        return None
    src = src.contiguous()
    M, N = src.shape
    P = mm * nn
    cores = [torch.empty((ranks[k], mm, nn, ranks[k + 1]), dtype=torch.float32, device=src.device) for k in range(order)]
    tab = (ctypes.c_void_p * order)(*[c.data_ptr() for c in cores])
    ws = workspace(src.device, ws_bytes)
    rc = lib.tt_decompose_nd(_p(src), tab, ranks_c, M, N, mm, nn, order, _tt_dtype_code(src.dtype), _p(ws), ws.numel(),
                             _stream_ptr(src.device))
    check(rc, "tt_decompose_nd")
    launch_counter["kernels"] += 1 + 5 * (order - 1)
    return cores


def reconstruct_nd(cores, M: int, N: int, mm: int, nn: int, dtype=torch.float32):
    """(M,N) window of an order >= 3 TT in one C-ABI call (tt_reconstruct_nd); None when the ranks are not supported."""
    lib = _lib.load()
    order = len(cores)
    ranks = [int(c.shape[0]) for c in cores] + [int(cores[-1].shape[-1])]
    ranks_c = (ctypes.c_int * len(ranks))(*ranks)
    ws_bytes = lib.tt_nd_workspace_bytes(mm, nn, order, ranks_c)
    if ws_bytes == 0:
        return None
    cs = [c.detach().to(torch.float32).contiguous() for c in cores]
    _require_cuda(*cs)
    dev = cs[0].device
    out = torch.empty((M, N), dtype=dtype, device=dev)
    tab = (ctypes.c_void_p * order)(*[c.data_ptr() for c in cs])
    ws = workspace(dev, ws_bytes)
    rc = lib.tt_reconstruct_nd(tab, ranks_c, _p(out), M, N, mm, nn, order, _tt_dtype_code(dtype), _p(ws), ws.numel(), _stream_ptr(dev))
    check(rc, "tt_reconstruct_nd")
    launch_counter["kernels"] += order
    return out


class TTAdamNPlan:
    """Persistent state of the one-call TT-Adam step of ONE parameter with an order >= 3 tensor train (tt_adam_nd_step):
    two sets of cores used ping-pong, the k-th core of both moments in one (2, r_k * P * r_{k+1}) tensor, and the pointer
    tables of both sets.  ``supported`` is False when the C entry point does not take the shape (a rank above 64 or above
    an unfolding size): the caller then keeps the op-by-op path."""

    def __init__(self, device, mm: int, nn: int, ranks):
        lib = _lib.load()
        self.mm, self.nn, self.ranks, self.order = mm, nn, [int(r) for r in ranks], len(ranks) - 1
        self.P = mm * nn
        self._ranks_c = (ctypes.c_int * len(self.ranks))(*self.ranks)
        self.ws_bytes = lib.tt_adam_nd_workspace_bytes(mm, nn, self.order, self._ranks_c)
        self.supported = self.ws_bytes > 0
        self.device = device
        self.cur = -1
        if not self.supported:
            return
        P, rk = self.P, self.ranks
        self.bufs = [[torch.empty((2, rk[k] * P * rk[k + 1]), dtype=torch.float32, device=device) for k in range(self.order)]
                     for _ in range(2)]
        self._tab = [(ctypes.c_void_p * self.order)(*[t.data_ptr() for t in self.bufs[s]]) for s in range(2)]

    def cores(self, s: int, b: int):
        """Cores (r_k, mm, nn, r_{k+1}) of moment b (0: m, 1: v) in set s, as views."""
        rk = self.ranks
        return [self.bufs[s][k][b].reshape(rk[k], self.mm, self.nn, rk[k + 1]) for k in range(self.order)]

    def step(self, p, g, beta1, beta2, eps, step_size, lr_wd, stream=None) -> int:
        lib = _lib.load()
        first = self.cur < 0
        out = 0 if first else 1 - self.cur
        M, N = p.shape
        ws = workspace(self.device, self.ws_bytes, stream)
        sp = ctypes.c_void_p(stream.cuda_stream) if stream is not None else _stream_ptr(self.device)
        rc = lib.tt_adam_nd_step(_p(p), _p(g), None if first else self._tab[self.cur], self._tab[out], self._ranks_c, M, N,
                               self.mm, self.nn, self.order, float(beta1), float(beta2), float(eps), float(step_size),
                               float(lr_wd), 1 if first else 0, _tt_dtype_code(p.dtype), _p(ws), ws.numel(), sp)
        check(rc, "tt_adam_nd_step")
        launch_counter["kernels"] += 2 * (self.order - 1) + 1 + 8 * (self.order - 1)
        self.cur = out
        return out


def tt_adam_interleaved(p, g, m, v, mm, nn, order, beta1, beta2, eps, step_size, lr_wd):
    """In-place TT-Adam on interleaved fp32 moments m, v ((mm*nn)^order elements each); p, g are (M,N)."""
    _require_cuda(p, g, m, v)
    lib = _lib.load()
    g = g.contiguous()
    M, N = p.shape
    rc = lib.tt_adam_interleaved(_p(p), _p(g), _p(m), _p(v), M, N, mm, nn, order, float(beta1), float(beta2), float(eps),
                                 float(step_size), float(lr_wd), _tt_dtype_code(p.dtype), _stream_ptr(p.device))
    check(rc, "tt_adam_interleaved")
    launch_counter["kernels"] += 1


def tt_adam_dense(p, g, m, v, beta1, beta2, eps, step_size, lr_wd):
    _require_cuda(p, g, m, v)
    lib = _lib.load()
    g = g.contiguous()
    rc = lib.tt_adam_dense(_p(p), _p(g), _p(m), _p(v), p.numel(), float(beta1), float(beta2), float(eps),
                           float(step_size), float(lr_wd), _tt_dtype_code(p.dtype), _stream_ptr(p.device))
    check(rc, "tt_adam_dense")
    launch_counter["kernels"] += 1


# ---------------------------------------------------------------------------------------------------------
# multi-tensor Adam
# ---------------------------------------------------------------------------------------------------------

def build_adam_chunks(ps: List[torch.Tensor], gs: List[torch.Tensor], ms: List[torch.Tensor],
                      vs: List[torch.Tensor]) -> torch.Tensor:
    """Device table int64[n_chunks,5] = (p, g, m, v, n) per chunk of <= sow_adam_chunk_elems() elements."""
    lib = _lib.load()
    ce = lib.sow_adam_chunk_elems()
    rows = []
    for p, g, m, v in zip(ps, gs, ms, vs):
        _require_cuda(p, g, m, v)
        if not (p.is_contiguous() and g.is_contiguous() and m.is_contiguous() and v.is_contiguous()):
            raise SowB200Error("fused Adam needs contiguous p/g/m/v")
        n = p.numel()
        if not (g.numel() == m.numel() == v.numel() == n):
            raise SowB200Error("fused Adam needs p/g/m/v of the same size")
        ep, eg, em, ev = p.element_size(), g.element_size(), m.element_size(), v.element_size()
        for off in range(0, n, ce):
            rows.append((p.data_ptr() + off * ep, g.data_ptr() + off * eg, m.data_ptr() + off * em,
                         v.data_ptr() + off * ev, min(ce, n - off)))
    table = torch.from_numpy(np.asarray(rows, dtype=np.int64).reshape(-1, 5)).to(ps[0].device, non_blocking=False)
    table._sow_total_elems = int(sum(p.numel() for p in ps))
    return table


def adam_multi(chunks: torch.Tensor, dtype: torch.dtype, lr, beta1, beta2, eps, weight_decay, bc1, bc2, decoupled):
    lib = _lib.load()
    total = getattr(chunks, "_sow_total_elems", 0)
    rc = lib.sow_adam_multi_ex(_p(chunks), chunks.shape[0], total, float(lr), float(beta1), float(beta2), float(eps),
                               float(weight_decay), float(bc1), float(bc2), 1 if decoupled else 0, _dtype_code(dtype),
                               _stream_ptr(chunks.device))
    check(rc, "sow_adam_multi")
    launch_counter["kernels"] += 1


def adam_multi_dev(chunks: torch.Tensor, dtype: torch.dtype, lr, beta1, beta2, eps, weight_decay, step_dev: torch.Tensor,
                   decoupled):
    """Graph-capturable fused Adam: advances the device step counter and derives the bias corrections from it."""
    lib = _lib.load()
    if not (step_dev.is_cuda and step_dev.dtype == torch.float32 and step_dev.numel() == 1):
        raise SowB200Error("adam_multi_dev: step must be a single-element fp32 CUDA tensor")
    total = getattr(chunks, "_sow_total_elems", 0)
    rc = lib.sow_adam_multi_dev(_p(chunks), chunks.shape[0], total, float(lr), float(beta1), float(beta2), float(eps),
                                float(weight_decay), _p(step_dev), 1 if decoupled else 0, _dtype_code(dtype),
                                _stream_ptr(chunks.device))
    check(rc, "sow_adam_multi_dev")
    launch_counter["kernels"] += 2


def adam_multi_amp(chunks: torch.Tensor, dtype: torch.dtype, state_dtype: torch.dtype, lr, beta1, beta2, eps, weight_decay,
                   decoupled, bc1=1.0, bc2=1.0, step_dev: Optional[torch.Tensor] = None,
                   grad_scale: Optional[torch.Tensor] = None, found_inf: Optional[torch.Tensor] = None):
    """Fused Adam with moments of ``state_dtype`` (the parameter dtype or fp32) and torch.amp.GradScaler's device scalars:
    ``grad_scale`` unscales the gradients in the kernel (and writes them back unscaled), ``found_inf`` != 0 skips the step
    on the device.  ``step_dev`` given: device step counter as in adam_multi_dev (required with ``found_inf``); otherwise
    the host bias corrections ``bc1``, ``bc2``."""
    lib = _lib.load()
    for name, t in (("step", step_dev), ("grad_scale", grad_scale), ("found_inf", found_inf)):
        if t is not None and not (t.is_cuda and t.dtype == torch.float32 and t.numel() == 1 and t.device == chunks.device):
            raise SowB200Error(f"adam_multi_amp: {name} must be a single-element fp32 tensor on {chunks.device}")
    total = getattr(chunks, "_sow_total_elems", 0)
    rc = lib.sow_adam_multi_amp(_p(chunks), chunks.shape[0], total, float(lr), float(beta1), float(beta2), float(eps),
                                float(weight_decay), float(bc1), float(bc2), _p(step_dev), _p(grad_scale), _p(found_inf),
                                1 if decoupled else 0, _dtype_code(dtype), _dtype_code(state_dtype),
                                _stream_ptr(chunks.device))
    check(rc, "sow_adam_multi_amp")
    launch_counter["kernels"] += 1 if step_dev is None else 2


def _check_scalar(fn: str, name: str, t: Optional[torch.Tensor], device: torch.device):
    if t is not None and not (t.is_cuda and t.dtype == torch.float32 and t.numel() == 1 and t.device == device):
        raise SowB200Error(f"{fn}: {name} must be a single-element fp32 tensor on {device}")


def grad_norm(tables: Sequence[Tuple[torch.Tensor, torch.dtype]], partials: torch.Tensor, total_norm: torch.Tensor,
              clip_coef: torch.Tensor, max_norm: float, grad_scale: Optional[torch.Tensor] = None):
    """Global 2-norm of the gradients of several Adam chunk tables ``(chunks, gradient dtype)`` -- one partial per chunk
    row into consecutive ranges of ``partials`` (fp32, at least one element per row in total), then one finalize -- and
    the clip coefficient ``min(max_norm / (total_norm + 1e-6), 1)`` as torch computes it.  ``grad_scale``: the norm is
    that of the unscaled gradients.  Writes ``total_norm`` and ``clip_coef`` (single-element fp32 device tensors)."""
    lib = _lib.load()
    dev = partials.device
    _require_cuda(partials)
    if partials.dtype != torch.float32 or not partials.is_contiguous():
        raise SowB200Error("grad_norm: partials must be a contiguous fp32 tensor")
    for name, t in (("total_norm", total_norm), ("clip_coef", clip_coef), ("grad_scale", grad_scale)):
        _check_scalar("grad_norm", name, t, dev)
    rows = sum(chunks.shape[0] for chunks, _ in tables)
    if partials.numel() < max(rows, 1):
        raise SowB200Error(f"grad_norm: {partials.numel()} partials for {rows} chunk rows")
    off = 0
    for chunks, dtype in tables:
        if chunks.device != dev:
            raise SowB200Error(f"grad_norm: chunk table on {chunks.device}, partials on {dev}")
        n = chunks.shape[0]
        if n:
            rc = lib.sow_grad_norm_partials(_p(chunks), n, _dtype_code(dtype), _p(grad_scale),
                                            ctypes.c_void_p(partials.data_ptr() + 4 * off), _stream_ptr(dev))
            check(rc, "sow_grad_norm_partials")
            launch_counter["kernels"] += 1
        off += n
    rc = lib.sow_grad_norm_finalize(_p(partials), max(rows, 1), float(max_norm), _p(total_norm), _p(clip_coef),
                                    _stream_ptr(dev))
    check(rc, "sow_grad_norm_finalize")
    launch_counter["kernels"] += 1


def adam_multi_clip(chunks: torch.Tensor, dtype: torch.dtype, state_dtype: torch.dtype, lr, beta1, beta2, eps, weight_decay,
                    decoupled, clip_coef: torch.Tensor, bc1=1.0, bc2=1.0, step_dev: Optional[torch.Tensor] = None,
                    grad_scale: Optional[torch.Tensor] = None, found_inf: Optional[torch.Tensor] = None):
    """adam_multi_amp with the gradients multiplied by the device scalar ``clip_coef`` (after the unscale, each product
    rounded to the gradient dtype) and written back, as ``unscale_`` + ``clip_grad_norm_`` leave them."""
    lib = _lib.load()
    if clip_coef is None:
        raise SowB200Error("adam_multi_clip: clip_coef is required")
    for name, t in (("step", step_dev), ("grad_scale", grad_scale), ("found_inf", found_inf), ("clip_coef", clip_coef)):
        _check_scalar("adam_multi_clip", name, t, chunks.device)
    total = getattr(chunks, "_sow_total_elems", 0)
    rc = lib.sow_adam_multi_clip(_p(chunks), chunks.shape[0], total, float(lr), float(beta1), float(beta2), float(eps),
                                 float(weight_decay), float(bc1), float(bc2), _p(step_dev), _p(grad_scale), _p(found_inf),
                                 _p(clip_coef), 1 if decoupled else 0, _dtype_code(dtype), _dtype_code(state_dtype),
                                 _stream_ptr(chunks.device))
    check(rc, "sow_adam_multi_clip")
    launch_counter["kernels"] += 1 if step_dev is None else 2


# ---------------------------------------------------------------------------------------------------------
# Llama block glue: rotary embedding and SwiGLU (bit-identical to the eager HF chains; sow_b200/llama_glue.py)
# ---------------------------------------------------------------------------------------------------------

def _glue_dtype_code(dt: torch.dtype) -> int:
    if dt not in (torch.bfloat16, torch.float16):
        raise SowB200Error(f"the Llama glue kernels take bf16 / fp16 tensors, not {dt}")
    return _dtype_code(dt)


def _rope_strided(t: torch.Tensor) -> torch.Tensor:
    """(B, H, S, D) in any layout with a contiguous last dim, 16-byte aligned rows; anything else is made contiguous."""
    if t.stride(-1) == 1 and t.data_ptr() % 16 == 0 and all(s % 8 == 0 for s in t.stride()[:3]):
        return t
    return t.contiguous()


def _rope_call(fn: str, q: torch.Tensor, k: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor):
    _require_cuda(q, k, cos, sin)
    B, Hq, S, D = q.shape
    Hk = k.shape[1]
    if k.shape != (B, Hk, S, D) or cos.shape != sin.shape or cos.shape not in ((1, S, D), (B, S, D)):
        raise SowB200Error(f"{fn}: q {tuple(q.shape)}, k {tuple(k.shape)}, cos {tuple(cos.shape)} do not match")
    if not (q.dtype == k.dtype == cos.dtype == sin.dtype) or not (cos.is_contiguous() and sin.is_contiguous()):
        raise SowB200Error(f"{fn}: q, k, cos, sin must share one dtype and cos / sin be contiguous")
    q, k = _rope_strided(q), _rope_strided(k)
    # outputs (B, S, H, D) contiguous, returned as their (B, H, S, D) transpose: eager q_embed's strides
    q_out = torch.empty((B, S, Hq, D), dtype=q.dtype, device=q.device).transpose(1, 2)
    k_out = torch.empty((B, S, Hk, D), dtype=k.dtype, device=k.device).transpose(1, 2)
    cs_sb = 0 if cos.shape[0] == 1 else S * D
    rc = getattr(_lib.load(), fn)(_p(q), _p(k), _p(cos), _p(sin), _p(q_out), _p(k_out), B, S, Hq, Hk, D,
                                  q.stride(0), q.stride(1), q.stride(2), k.stride(0), k.stride(1), k.stride(2), cs_sb,
                                  _glue_dtype_code(q.dtype), _stream_ptr(q.device))
    check(rc, fn)
    launch_counter["kernels"] += 1
    return q_out, k_out


def rope_fwd(q: torch.Tensor, k: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor):
    """q * cos + rotate_half(q) * sin and the same for k, in one launch.  q, k: (B, H, S, D); cos, sin: (B or 1, S, D)."""
    return _rope_call("sow_rope_fwd", q, k, cos, sin)


def rope_bwd(gq: torch.Tensor, gk: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor):
    """Gradients of rope_fwd w.r.t. q and k from the upstream gradients gq, gk (either layout), in one launch."""
    return _rope_call("sow_rope_bwd", gq, gk, cos, sin)


def _glue_contig(t: torch.Tensor) -> torch.Tensor:
    return t if t.is_contiguous() and t.data_ptr() % 16 == 0 else t.contiguous()


def swiglu_fwd(gate: torch.Tensor, up: torch.Tensor) -> torch.Tensor:
    """silu(gate) * up."""
    _require_cuda(gate, up)
    if gate.shape != up.shape or gate.dtype != up.dtype:
        raise SowB200Error("swiglu: gate and up must have the same shape and dtype")
    gate, up = _glue_contig(gate), _glue_contig(up)
    h = torch.empty_like(gate, memory_format=torch.contiguous_format)
    rc = _lib.load().sow_swiglu_fwd(_p(gate), _p(up), _p(h), gate.numel(), _glue_dtype_code(gate.dtype),
                                    _stream_ptr(gate.device))
    check(rc, "sow_swiglu_fwd")
    launch_counter["kernels"] += 1
    return h


def swiglu_bwd(dh: torch.Tensor, gate: torch.Tensor, up: torch.Tensor):
    """(dgate, dup) of h = silu(gate) * up, in one pass over dh, gate and up."""
    _require_cuda(dh, gate, up)
    if not (dh.shape == gate.shape == up.shape) or not (dh.dtype == gate.dtype == up.dtype):
        raise SowB200Error("swiglu: dh, gate and up must have the same shape and dtype")
    dh, gate, up = _glue_contig(dh), _glue_contig(gate), _glue_contig(up)
    dgate = torch.empty_like(gate, memory_format=torch.contiguous_format)
    dup = torch.empty_like(up, memory_format=torch.contiguous_format)
    rc = _lib.load().sow_swiglu_bwd(_p(dh), _p(gate), _p(up), _p(dgate), _p(dup), gate.numel(),
                                    _glue_dtype_code(gate.dtype), _stream_ptr(gate.device))
    check(rc, "sow_swiglu_bwd")
    launch_counter["kernels"] += 1
    return dgate, dup


def _norm_args(fn: str, x: torch.Tensor, w: torch.Tensor, *others: torch.Tensor):
    _require_cuda(x, w, *others)
    if w.dim() != 1 or x.dim() < 1 or x.shape[-1] != w.shape[0] or any(t.shape != x.shape for t in others):
        raise SowB200Error(f"{fn}: x {tuple(x.shape)} and w {tuple(w.shape)} do not match")
    if any(t.dtype != x.dtype for t in (w, *others)):
        raise SowB200Error(f"{fn}: x, w and the gradients must share one dtype")
    return (_glue_contig(t) for t in (x, w, *others))


def rmsnorm_fwd(x: torch.Tensor, w: torch.Tensor, eps: float):
    """LlamaRMSNorm forward over the last dim: (y = w * (x * rs), rs = rsqrt(mean(x^2) + eps)), rs fp32 of shape
    x.shape[:-1]."""
    x, w = _norm_args("sow_rmsnorm_fwd", x, w)
    y = torch.empty_like(x)
    rs = torch.empty(x.shape[:-1], dtype=torch.float32, device=x.device)
    rc = _lib.load().sow_rmsnorm_fwd(_p(x), _p(w), _p(y), _p(rs), rs.numel(), x.shape[-1], eps,
                                     _glue_dtype_code(x.dtype), _stream_ptr(x.device))
    check(rc, "sow_rmsnorm_fwd")
    launch_counter["kernels"] += 1
    return y, rs


def rmsnorm_bwd(dy: torch.Tensor, x: torch.Tensor, w: torch.Tensor, rs: torch.Tensor, want_p: bool = True):
    """(dx, p) of rmsnorm_fwd from the upstream gradient dy and the saved rs; p = dy * (x * rs) is the per-element
    product whose sum over the rows is dw (None unless want_p)."""
    x, w, dy = _norm_args("sow_rmsnorm_bwd", x, w, dy)
    if rs.dtype != torch.float32 or rs.shape != x.shape[:-1] or not rs.is_contiguous():
        raise SowB200Error("sow_rmsnorm_bwd: rs must be contiguous fp32 of shape x.shape[:-1]")
    dx = torch.empty_like(x)
    p = torch.empty_like(x) if want_p else None
    rc = _lib.load().sow_rmsnorm_bwd(_p(dy), _p(x), _p(w), _p(rs), _p(dx), _p(p), rs.numel(), x.shape[-1],
                                     _glue_dtype_code(x.dtype), _stream_ptr(x.device))
    check(rc, "sow_rmsnorm_bwd")
    launch_counter["kernels"] += 1
    return dx, p


def _ce_args(fn: str, logits: torch.Tensor, target: torch.Tensor, *rows: torch.Tensor):
    _require_cuda(logits, target, *rows)
    if logits.dim() != 2 or target.shape != logits.shape[:1] or any(t.shape != target.shape for t in rows):
        raise SowB200Error(f"{fn}: logits {tuple(logits.shape)} and targets {tuple(target.shape)} do not match")
    if target.dtype != torch.int64 or any(t.dtype != torch.float32 for t in rows):
        raise SowB200Error(f"{fn}: targets must be int64 and the row values fp32")
    return _glue_contig(logits), target.contiguous(), *(t.contiguous() for t in rows)


def ce_fwd(logits: torch.Tensor, target: torch.Tensor):
    """Row statistics of log_softmax(logits.float()) for (N, V) logits and (N,) int64 targets: fp32 (row_max, row_logsum,
    logp_t), logp_t[i] = log_softmax(logits)[i, target[i]] (0 where the target is outside [0, V))."""
    logits, target = _ce_args("sow_ce_fwd", logits, target)
    N, V = logits.shape
    row_max, row_logsum, logp_t = (torch.empty(N, dtype=torch.float32, device=logits.device) for _ in range(3))
    rc = _lib.load().sow_ce_fwd(_p(logits), _p(target), _p(row_max), _p(row_logsum), _p(logp_t), N, V,
                                _glue_dtype_code(logits.dtype), _stream_ptr(logits.device))
    check(rc, "sow_ce_fwd")
    launch_counter["kernels"] += 1
    return row_max, row_logsum, logp_t


def ce_bwd(logits: torch.Tensor, row_max: torch.Tensor, row_logsum: torch.Tensor, target: torch.Tensor,
           dlogp_t: torch.Tensor) -> torch.Tensor:
    """Gradient w.r.t. the logits (their dtype, (N, V)) of sum_i dlogp_t[i] * logp_t[i], with ce_fwd's row statistics."""
    logits, target, row_max, row_logsum, dlogp_t = _ce_args("sow_ce_bwd", logits, target, row_max, row_logsum, dlogp_t)
    N, V = logits.shape
    grad = torch.empty_like(logits)
    rc = _lib.load().sow_ce_bwd(_p(logits), _p(row_max), _p(row_logsum), _p(target), _p(dlogp_t), _p(grad), N, V,
                                _glue_dtype_code(logits.dtype), _stream_ptr(logits.device))
    check(rc, "sow_ce_bwd")
    launch_counter["kernels"] += 1
    return grad


# ---------------------------------------------------------------------------------------------------------
# live profiling (bench.py)
# ---------------------------------------------------------------------------------------------------------
PROF_CLASSES = {"gemm_fwd": 0, "gemm_dx": 1, "gemm_skinny": 2, "gemm_splitk": 3, "merge": 4, "adam": 5, "gemm_k2": 6}


def profile_enable(on: bool) -> None:
    check(_lib.load().sow_profile_enable(1 if on else 0), "sow_profile_enable")


def profile_read(klass: str):
    """(total_ms, total_work, launches) of one kernel class since profiling was enabled; syncs on its events."""
    ms, work, n = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_int64(0)
    check(_lib.load().sow_profile_read(PROF_CLASSES[klass], ctypes.byref(ms), ctypes.byref(work), ctypes.byref(n)),
          "sow_profile_read")
    return ms.value, work.value, n.value
