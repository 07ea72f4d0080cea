"""GPU: gradient clipping inside FusedAdamW (max_grad_norm) -- the norm kernel against fp64, bit-exactness against
"native norm, torch's coefficient, the fp32 product, unclipped step", loss scaling, host syncs, determinism, CUDA-graph
replay, and SoWTrainer(fused_grad_clipping=True) against the torch.nn.utils.clip_grad_norm_ path."""
import math
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn

from test_amp_gpu import _bits, _golden_trainer, _sync_count
from test_trajectory_gpu import _golden

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _chunk_elems():
    from sow_b200 import _lib
    return _lib.load().sow_adam_chunk_elems()


def _same(a, b):
    """Bit-identical, NaN payloads aside (a NaN must be a NaN at the same position)."""
    a, b = a.detach(), b.detach()
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(_bits(a[~na]), _bits(b[~nb]))


# ---------------------------------------------------------------------------------------------------------
# the norm kernel
# ---------------------------------------------------------------------------------------------------------

def _native_norm(grads, max_norm=1.0, grad_scale=None):
    """ops.grad_norm over one chunk table per dtype, as FusedAdamW groups them."""
    from sow_b200 import ops
    by = {}
    for g in grads:
        by.setdefault(g.dtype, []).append(g)
    tables = [(ops.build_adam_chunks(gs, gs, gs, gs), dt) for dt, gs in by.items()]
    rows = sum(t.shape[0] for t, _ in tables)
    partials = torch.full((max(rows, 1),), float("nan"), device="cuda")
    total, coef = torch.empty((), device="cuda"), torch.empty((), device="cuda")
    ops.grad_norm(tables, partials, total, coef, max_norm, grad_scale)
    return total, coef


def _ref_sq(grads, scale=None):
    """fp64 sum of squares of the values the kernel squares: round_G(g / scale) (IEEE division on the device)."""
    acc = 0.0
    for g in grads:
        x = g if scale is None else (g.float() / scale).to(g.dtype)
        acc += float((x.double() ** 2).sum())
    return acc


def _bound(ref_sq):
    k = _chunk_elems() // 256
    return (k + math.ceil(math.log2(256)) + 2) * 2.0 ** -24 * ref_sq


def _sizes():
    ce = _chunk_elems()
    return [1, 7, 1000, ce - 3, ce, ce + 1, 3 * ce + 17]


def _make(dt, n, gen, offset=0, lo=-3.0, hi=1.0):
    """n values with log-uniform magnitudes 10^lo .. 10^hi and random signs; offset 1 = a view one element into its
    buffer (not 16-byte aligned: the element path)."""
    e = torch.rand(n + offset, generator=gen, device="cuda", dtype=torch.float64) * (hi - lo) + lo
    s = torch.randint(0, 2, (n + offset,), generator=gen, device="cuda").double() * 2 - 1
    return (s * 10.0 ** e).to(dt)[offset:]


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16, torch.float32])
@pytest.mark.parametrize("scale", [None, 2.0 ** 10, 3000.7])
def test_norm_against_fp64(dt, scale):
    gen = torch.Generator(device="cuda").manual_seed(0)
    grads = []
    for i, n in enumerate(_sizes()):
        grads.append(_make(dt, n, gen, offset=i % 2))
    assert any(g.data_ptr() % 16 for g in grads) and any(g.data_ptr() % 16 == 0 for g in grads)
    gs = None
    if scale is not None:
        grads = [(g.float() * scale).to(dt) for g in grads]
        gs = torch.full((), scale, device="cuda")
    total, coef = _native_norm(grads, 1.0, gs)
    ref_sq = _ref_sq(grads, None if scale is None else gs)
    n = float(total)
    print(f"{dt} scale {scale}: native {n!r}, fp64 {math.sqrt(ref_sq)!r}")
    assert abs(n * n - ref_sq) <= _bound(ref_sq)
    assert float(coef) == float(torch.clamp(1.0 / (total + 1e-6), max=1.0))


def test_norm_fp32_dynamic_range_and_mixed_group():
    gen = torch.Generator(device="cuda").manual_seed(1)
    wide = [_make(torch.float32, n, gen, offset=i % 2, lo=-20.0, hi=17.0) for i, n in enumerate([5000, 1, 33, 40000])]
    wide[1].fill_(1e18)
    wide[2][0] = -1e-20
    ref_sq = _ref_sq(wide)
    assert ref_sq < 3.0e38                                  # squares and partials stay below fp32's maximum
    total, _ = _native_norm(wide)
    assert abs(float(total) ** 2 - ref_sq) <= _bound(ref_sq)
    mixed = [_make(torch.bfloat16, 70001, gen), _make(torch.float16, 33, gen, offset=1), _make(torch.float32, 40000, gen),
             _make(torch.bfloat16, 1, gen)]
    for scale in (None, 777.3):
        grads = mixed if scale is None else [(g.float() * scale).to(g.dtype) for g in mixed]
        gs = None if scale is None else torch.full((), scale, device="cuda")
        total, _ = _native_norm(grads, 1.0, gs)
        ref_sq = _ref_sq(grads, gs)
        assert abs(float(total) ** 2 - ref_sq) <= _bound(ref_sq)


def test_zero_gradients_give_norm_zero_and_coefficient_one():
    grads = [torch.zeros(n, device="cuda", dtype=dt) for n, dt in ((70001, torch.bfloat16), (5, torch.float32))]
    total, coef = _native_norm(grads, 0.5)
    assert float(total) == 0.0 and float(coef) == 1.0


# ---------------------------------------------------------------------------------------------------------
# FusedAdamW(max_grad_norm) against the two-step recipe
# ---------------------------------------------------------------------------------------------------------

def _mul_coef_(grads, coef):
    """g <- round_G(float(g) * coef) with the fp32 coefficient, one rounding.  This is what torch._foreach_mul_ computes
    for bf16 and fp32 lists; for an fp16 list and an fp32 0-dim coefficient it rounds the coefficient to fp16 first
    (g * fp16(coef)), so the product is written out here."""
    for g in grads:
        g.copy_((g.float() * coef).to(g.dtype))


SHAPES = [(1024, 50), (50, 2736), (33,), (70001,)]


def _recipe_pair(pdt, sdt, capturable, max_norm, wd=0.1, decoupled=True):
    from sow_b200.optim import FusedAdamW
    gen = torch.Generator(device="cuda").manual_seed(3)
    init = [(torch.randn(s, generator=gen, device="cuda") * 0.1).to(pdt) for s in SHAPES]
    a = [nn.Parameter(t.clone()) for t in init]
    b = [nn.Parameter(t.clone()) for t in init]
    kw = dict(lr=1e-2, weight_decay=wd, decoupled=decoupled, capturable=capturable, state_dtype=sdt)
    return a, b, FusedAdamW(a, max_grad_norm=max_norm, **kw), FusedAdamW(b, **kw), gen


def _recipe_step(a, b, opt_a, opt_b, grads, max_norm):
    """opt_a clips natively; opt_b gets torch's coefficient from the native norm, the fp32 product, an unclipped step."""
    for p, q, g in zip(a, b, grads):
        p.grad, q.grad = g.clone(), g.clone()
    opt_a.step()
    total = opt_a.grad_norm(0)
    coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
    _mul_coef_([q.grad for q in b], coef)
    opt_b.step()
    return total, coef


@pytest.mark.parametrize("capturable", [False, True])
@pytest.mark.parametrize("pdt,sdt", [(torch.bfloat16, None), (torch.bfloat16, torch.float32), (torch.float16, None),
                                     (torch.float16, torch.float32), (torch.float32, None)])
def test_clipped_step_is_bit_exact_against_the_recipe(capturable, pdt, sdt):
    gen0 = torch.Generator(device="cuda").manual_seed(4)
    grads0 = [(torch.randn(s, generator=gen0, device="cuda") * 0.01).to(pdt) for s in SHAPES]
    ref = math.sqrt(_ref_sq(grads0))
    for factor, active in ((0.5, True), (2.0, False)):
        max_norm = factor * ref
        a, b, opt_a, opt_b, gen = _recipe_pair(pdt, sdt, capturable, max_norm, decoupled=not active)
        assert opt_a.grad_norm(0) is None
        for k in range(3):
            grads = [(torch.randn(s, generator=gen, device="cuda") * 0.01).to(pdt) for s in SHAPES] if k else grads0
            if k == 2:
                grads[3][5] = float("inf")                      # coefficient 0, as torch computes it
            total, coef = _recipe_step(a, b, opt_a, opt_b, grads, max_norm)
            torch.cuda.synchronize()
            native_coef = opt_a._clip[0]["clip_coef"]
            assert _same(native_coef, coef), (float(native_coef), float(coef))
            if k == 0:
                assert (float(coef) < 1.0) == active
            if k == 2:
                assert math.isinf(float(total)) and float(coef) == 0.0
            for p, q in zip(a, b):
                assert _same(p, q) and _same(p.grad, q.grad)
                for key in ("exp_avg", "exp_avg_sq"):
                    assert _same(opt_a.state[p][key], opt_b.state[q][key])
                assert float(opt_a.state[p]["step"]) == float(opt_b.state[q]["step"]) == k + 1
            if not active and k < 2:
                assert all(torch.equal(_bits(p.grad), _bits(g)) for p, g in zip(a, grads))     # left bit-identical


def test_clipped_steps_are_deterministic():
    runs = []
    for _ in range(2):
        a, b, opt_a, opt_b, gen = _recipe_pair(torch.bfloat16, torch.float32, True, 0.05)
        norms = []
        for k in range(3):
            grads = [(torch.randn(s, generator=gen, device="cuda") * 0.01).bfloat16() for s in SHAPES]
            for p, g in zip(a, grads):
                p.grad = g
            opt_a.step()
            norms.append(opt_a.grad_norm(0).clone().reshape(1))
        torch.cuda.synchronize()
        runs.append((norms, [_bits(p) for p in a], [_bits(opt_a.state[p]["exp_avg_sq"]) for p in a]))
    (n0, p0, v0), (n1, p1, v1) = runs
    assert all(torch.equal(_bits(x), _bits(y)) for x, y in zip(n0, n1))
    assert all(torch.equal(x, y) for x, y in zip(p0 + v0, p1 + v1))


# ---------------------------------------------------------------------------------------------------------
# loss scaling
# ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("capturable", [False, True])
def test_loss_scaled_fp16_clipping(capturable):
    """fp16 parameters, fp32 moments, GradScaler at 2^16, gradients whose scaled per-tensor norms overflow fp16 (torch's
    clip_grad_norm_ on them would zero every gradient): the native norm is that of the unscaled gradients, and the step
    equals "unscale, then the recipe" bit for bit.  A found_inf step changes no bit."""
    from sow_b200.optim import FusedAdamW
    scale = 2.0 ** 16
    gen = torch.Generator(device="cuda").manual_seed(5)
    init = [(torch.randn(s, generator=gen, device="cuda") * 0.1).half() for s in SHAPES]
    a = [nn.Parameter(t.clone()) for t in init]
    b = [nn.Parameter(t.clone()) for t in init]
    kw = dict(lr=1e-2, weight_decay=0.1, capturable=capturable, state_dtype=torch.float32)
    unscaled0 = [(torch.randn(s, generator=gen, device="cuda") * 0.1).half() for s in SHAPES]
    max_norm = 0.5 * math.sqrt(_ref_sq(unscaled0))
    opt_a, opt_b = FusedAdamW(a, max_grad_norm=max_norm, **kw), FusedAdamW(b, **kw)
    scaler = torch.amp.GradScaler("cuda", init_scale=scale, growth_interval=1000)
    for p in a:
        p.grad = torch.zeros_like(p)                         # stable addresses: the chunk tables are built once

    for k in range(4):
        unscaled = unscaled0 if k == 0 else [(torch.randn(s, generator=gen, device="cuda") * 0.1).half() for s in SHAPES]
        cur = scaler.get_scale()
        for p, u in zip(a, unscaled):
            p.grad.copy_(scaler.scale(u.float()).half())     # exact: a power-of-two scale, no overflow
        if k == 2:
            a[1].grad[3, 5] = float("inf")
        scaled = [p.grad.clone() for p in a]
        if k == 0:
            assert any(torch.isinf(torch.linalg.vector_norm(s_)) for s_ in scaled)   # fp16 norm of the scaled gradients
        snap = [(_bits(p), _bits(opt_a.state[p]["exp_avg"]) if p in opt_a.state else None) for p in a]
        n_sync = _sync_count(lambda: scaler.step(opt_a))
        scaler.update()
        torch.cuda.synchronize()
        if k > 0:
            assert n_sync == (0 if capturable else 1)
        if k == 2:                                           # skipped: nothing changed
            assert scaler.get_scale() == cur / 2
            for p, s_, (pb, mb) in zip(a, scaled, snap):
                assert torch.equal(_bits(p), pb) and torch.equal(_bits(p.grad), _bits(s_))
                assert torch.equal(_bits(opt_a.state[p]["exp_avg"]), mb)
            assert float(opt_a.state[a[0]]["step"]) == 2
            continue
        gs = torch.full((), cur, device="cuda")
        ref_sq = _ref_sq(scaled, gs)
        total = opt_a.grad_norm(0)
        assert abs(float(total) ** 2 - ref_sq) <= _bound(ref_sq), (float(total), math.sqrt(ref_sq))
        for q, s_ in zip(b, scaled):
            q.grad = (s_.float() / gs).half()                # what unscale_ writes
        coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
        _mul_coef_([q.grad for q in b], coef)
        opt_b.step()
        torch.cuda.synchronize()
        if k == 0:
            assert float(coef) < 1.0
        for p, q in zip(a, b):
            assert torch.equal(_bits(p), _bits(q)) and torch.equal(_bits(p.grad), _bits(q.grad))
            for key in ("exp_avg", "exp_avg_sq"):
                assert torch.equal(_bits(opt_a.state[p][key]), _bits(opt_b.state[q][key]))


# ---------------------------------------------------------------------------------------------------------
# CUDA graphs
# ---------------------------------------------------------------------------------------------------------

def test_captured_clipped_step_replays_bit_identical_to_eager():
    from sow_b200.optim import FusedAdamW
    gen = torch.Generator(device="cuda").manual_seed(6)
    init = [(torch.randn(s, generator=gen, device="cuda") * 0.1).bfloat16() for s in SHAPES]
    steps = [[(torch.randn(s, generator=gen, device="cuda") * (0.002 * (k % 4 + 1))).bfloat16() for s in SHAPES]
             for k in range(10)]
    max_norm = 0.6 * math.sqrt(_ref_sq(steps[1]))           # steps k % 4 == 0 have about half that norm: inactive
    results = []
    for graphed in (False, True):
        params = [nn.Parameter(t.clone()) for t in init]
        for p in params:
            p.grad = torch.zeros_like(p)
        opt = FusedAdamW(params, lr=1e-2, capturable=True, state_dtype=torch.float32, max_grad_norm=max_norm)
        norms, coefs, graph = [], [], None
        for k, grads in enumerate(steps):
            for p, g in zip(params, grads):
                p.grad.copy_(g)
            if not graphed or k < 2:
                opt.step()
            else:
                if graph is None:
                    torch.cuda.synchronize()
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph):            # records the step without running it
                        opt.step()
                graph.replay()
            norms.append(opt.grad_norm(0).clone().reshape(1))
            coefs.append(opt._clip[0]["clip_coef"].clone().reshape(1))
        torch.cuda.synchronize()
        results.append((norms, coefs, [_bits(p) for p in params], [_bits(p.grad) for p in params],
                        [_bits(opt.state[p]["exp_avg_sq"]) for p in params]))
    (ne, ce, pe, ge, ve), (ng, cg, pg, gg, vg) = results
    c = [float(x) for x in ce]
    print(f"coefficients {c}")
    assert any(x < 1.0 for x in c[2:]) and any(x == 1.0 for x in c[2:])
    assert all(torch.equal(_bits(x), _bits(y)) for x, y in zip(ne + ce, ng + cg))
    assert all(torch.equal(x, y) for x, y in zip(pe + ge + ve, pg + gg + vg))


# ---------------------------------------------------------------------------------------------------------
# SoWTrainer
# ---------------------------------------------------------------------------------------------------------

def _run_golden(g, dtype, fused, clip, record=None, **kw):
    tr, steps = _golden_trainer(g, dtype, grad_clipping=clip, fused_grad_clipping=fused, **kw)
    if record is not None:
        step = tr.optimizer.step

        def wrapped(*a, **k):
            grads = [p.grad for p in tr.trainable if p.grad is not None]
            sc = getattr(tr.optimizer, "grad_scale", None)
            ref = math.sqrt(_ref_sq(grads, sc))
            out = step(*a, **k)
            record.append((float(tr.optimizer.grad_norm(0)), ref))
            return out
        tr.optimizer.step = wrapped
    torch.manual_seed(1)
    losses = [float(tr.step(torch.from_numpy(g["batches"][s]).to("cuda"))) for s in range(steps)]
    assert tr.merges == 2
    return tr, losses


def _torch_norms(record):
    """Wrap torch.nn.utils.clip_grad_norm_ to record (returned norm, fp64 norm of its input gradients)."""
    orig = torch.nn.utils.clip_grad_norm_

    def wrapped(params, max_norm, *a, **k):
        params = list(params)
        ref = math.sqrt(_ref_sq([p.grad for p in params if p.grad is not None]))
        out = orig(params, max_norm, *a, **k)
        record.append((float(out), ref))
        return out
    return orig, wrapped


@pytest.mark.parametrize("dtype,clip,tol", [(torch.float32, 1e-3, 1e-5), (torch.bfloat16, 1e-3, 2e-2)])
def test_trainer_fused_clipping_matches_the_torch_path(dtype, clip, tol):
    g = _golden()
    torch_norms, native_norms = [], []
    orig, wrapped = _torch_norms(torch_norms)
    torch.nn.utils.clip_grad_norm_ = wrapped
    try:
        tr_t, l_t = _run_golden(g, dtype, False, clip)
    finally:
        torch.nn.utils.clip_grad_norm_ = orig
    tr_f, l_f = _run_golden(g, dtype, True, clip, record=native_norms)
    print(f"{dtype} losses torch {l_t} fused {l_f}")
    print(f"norms (value, fp64): torch {torch_norms}\n  native {native_norms}")
    assert len(torch_norms) == len(native_norms) == len(l_t)
    assert all(n > clip for n, _ in native_norms)              # clipping is active on every step
    for n, ref in native_norms:
        assert abs(n * n - ref * ref) <= _bound(ref * ref)
    for s, (a, b) in enumerate(zip(l_f, l_t)):
        assert abs(a - b) / abs(b) < tol, (s, a, b)
    if dtype == torch.float32:
        # the clipped (trainable) group to the loss tolerance.  The SoW factors restart Adam from zero moments after every
        # merge, where the update is lr * g / (|g| + eps): a last-bit difference of the clipped gradients, propagated into
        # a factor gradient element with |g| near eps, moves that element by O(lr), so they get a looser bound.
        clipped = {id(p) for p in tr_f.trainable}
        pt, pf = dict(tr_t.model.named_parameters()), dict(tr_f.model.named_parameters())
        errs = {n: float((pf[n].detach().double() - pt[n].detach().double()).norm() / (pt[n].detach().double().norm()
                                                                                      + 1e-30)) for n in pt}
        dense = {n: e for n, e in errs.items() if id(pf[n]) in clipped}
        factors = {n: e for n, e in errs.items() if id(pf[n]) not in clipped}
        print(f"parameter rel. error: clipped group max {max(dense.values()):.3e}, SoW factors max "
              f"{max(factors.values()):.3e}")
        assert dense and all(e < tol for e in dense.values()), dense
        assert all(e < 1e-3 for e in factors.values()), factors


def test_trainer_fp16_loss_scaling_with_fused_clipping_tracks_fp32():
    g = _golden()
    norms = []
    _, l_ref = _run_golden(g, torch.float32, False, 1e-3)
    tr, l16 = _run_golden(g, torch.float16, True, 1e-3, record=norms, optimizer_state_dtype=torch.float32,
                          loss_scaling=True, loss_scale_init=2.0 ** 12)
    print(f"fp16 + loss scaling + fused clipping {l16}\nfp32 torch-clipped {l_ref}\nnorms {norms}")
    assert tr.scaler.get_scale() == 2.0 ** 12                   # no step was skipped
    for s, (a, b) in enumerate(zip(l16, l_ref)):
        assert abs(a - b) / abs(b) < 2e-2, (s, a, b)


def test_fp16_loss_scaled_clipped_trainer_cuda_graph_replay_is_bit_identical_to_eager():
    from sow_b200.trainer import SoWTrainer, TrainConfig
    runs = []
    for graphed in (False, True):
        cfg = TrainConfig(model="llama_9m", rank=8, seq_len=64, batch_size=4, lr=1e-3, sow_lr=1e-3, sow_accumulation=100,
                          init_method="normal", cuda_graph=True, seed=1, dtype=torch.float16,
                          optimizer_state_dtype=torch.float32, loss_scaling=True, loss_scale_init=2.0 ** 30,
                          grad_clipping=0.05, fused_grad_clipping=True)
        torch.manual_seed(0)
        tr = SoWTrainer(cfg, torch.device("cuda", 0))
        tr.cfg.cuda_graph = graphed
        gen = torch.Generator().manual_seed(3)
        losses, scales, norms = [], [], []
        for _ in range(32):
            ids = torch.randint(1, 32000, (4, 64), generator=gen).cuda()
            losses.append(tr.step(ids).detach().clone())
            scales.append(tr.scaler.get_scale())
            norms.append(tr.optimizer.grad_norm(0).clone())
        torch.cuda.synchronize()
        assert (tr._graph is not None) == graphed
        moments = {n: (_bits(tr.optimizer.state[p]["exp_avg"]), _bits(tr.optimizer.state[p]["exp_avg_sq"]))
                   for n, p in tr.model.named_parameters() if p in tr.optimizer.state}
        runs.append((losses, scales, norms, {n: _bits(p) for n, p in tr.model.named_parameters()}, moments))
    (le, se, ne, pe, me), (lg, sg, ng, pg, mg) = runs
    print(f"scales {sg}\nnorms {[float(x) for x in ng]}")
    assert se == sg
    assert [k for k in range(2, 32) if sg[k] < sg[k - 1]] and [k for k in range(2, 32) if sg[k] >= sg[k - 1]], sg
    assert any(0.05 < float(x) < math.inf for x in ng)           # clipping active on taken steps
    assert all(torch.equal(a, b) for a, b in zip(le, lg))
    assert all(_same(a, b) for a, b in zip(ne, ng))
    for n in pe:
        assert torch.equal(pe[n], pg[n]), n
    for n in me:
        assert torch.equal(me[n][0], mg[n][0]) and torch.equal(me[n][1], mg[n][1]), n


# ---------------------------------------------------------------------------------------------------------
# two GPUs over NCCL
# ---------------------------------------------------------------------------------------------------------

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from sow_b200.parallel import assert_replicas_consistent
        from sow_b200.trainer import SoWTrainer, TrainConfig
        cfg = TrainConfig(model="llama_9m", rank=8, seq_len=64, batch_size=4, sow_accumulation=2, lr=1e-3, sow_lr=1e-3,
                          grad_clipping=0.05, fused_grad_clipping=True)
        tr = SoWTrainer(cfg, dev)
        gen = torch.Generator().manual_seed(99)
        batches = [torch.randint(1, 32000, (world * 4, 64), generator=gen) for _ in range(4)]
        norms = []
        for b in batches:
            tr.step(b[rank * 4:(rank + 1) * 4].to(dev))
            norms.append(tr.optimizer.grad_norm(0).clone().reshape(1))
        assert tr.merges >= 1
        assert_replicas_consistent([p for p in tr.model.parameters()], "parameter")
        assert_replicas_consistent(norms, "gradient norm")
        ret[rank] = [float(n) for n in norms]
    except Exception as e:  # pragma: no cover
        import traceback
        ret[rank] = "".join(traceback.format_exception(type(e), e, e.__traceback__))
    finally:
        dist.barrier()
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_fused_clipping_keeps_replicas_bit_identical():
    import torch.multiprocessing as mp
    mgr = mp.get_context("spawn").Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    for r in range(2):
        assert isinstance(ret.get(r), list), f"rank {r}: {ret.get(r)}"
    assert ret[0] == ret[1] and any(n > 0.05 for n in ret[0])
