"""GPU: fp32 optimizer moments (FusedAdamW state_dtype) and torch.amp.GradScaler loss scaling, from the kernel to SoWTrainer --
the oracle, parity with torch's fused AdamW, skipped steps, the exactness of power-of-two scales, the fp16 golden
trajectory, CUDA-graph replay and checkpoints."""
import copy
import warnings

import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import rel_err
from oracle import sow_oracle as O
from test_optim_loop_gpu import reset_optimizer
from test_trajectory_gpu import TARGETS, _golden, _prepared_from_golden

pytestmark = pytest.mark.gpu

SHAPES = [(1024, 50), (50, 2736), (33,), (70001,)]


def f16_round(a):
    return np.asarray(a, np.float64).astype(np.float16).astype(np.float64)


def _bits(t):
    return t.detach().contiguous().view(torch.uint8).clone()


# ---------------------------------------------------------------------------------------------------------
# FusedAdamW
# ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("pdt,rnd,tol", [(torch.float16, f16_round, 2e-3), (torch.bfloat16, O.bf16_round, 1e-2)])
def test_fp32_state_vs_oracle_with_reset(pdt, rnd, tol):
    from sow_b200.optim import FusedAdamW
    rng = np.random.default_rng(0)
    ps_np = [rnd(rng.standard_normal(s) * 0.1) for s in SHAPES]
    params = [nn.Parameter(torch.from_numpy(np.asarray(p, np.float32)).to("cuda", pdt)) for p in ps_np]
    opt = FusedAdamW([{"params": params[:2], "lr": 1e-2, "weight_decay": 0.1},
                      {"params": params[2:], "lr": 3e-3, "weight_decay": 0.0}], state_dtype=torch.float32)
    states = [dict() for _ in SHAPES]
    cur = [np.asarray(p, np.float64) for p in ps_np]
    for step in range(6):
        grads = [rnd(rng.standard_normal(s) * 1e-3) for s in SHAPES]     # small: (1 - b2) g^2 is below fp16's range
        for p, gr in zip(params, grads):
            p.grad = torch.from_numpy(np.asarray(gr, np.float32)).to("cuda", pdt)
        if step == 3:
            reset_optimizer(opt, 0)                     # rebinds 16-bit zeros: converted back to fp32 by the next step
            states[0], states[1] = {}, {}
            assert opt.state[params[0]]["exp_avg"].dtype == pdt
        opt.step()
        for i in range(len(SHAPES)):
            lr, wd = (1e-2, 0.1) if i < 2 else (3e-3, 0.0)
            cur[i] = rnd(O.adamw_step(cur[i], grads[i], states[i], lr, weight_decay=wd))
    torch.cuda.synchronize()
    for i, p in enumerate(params):
        st = opt.state[p]
        assert p.dtype == pdt
        assert st["exp_avg"].dtype == torch.float32 and st["exp_avg_sq"].dtype == torch.float32
        assert rel_err(p.detach().float().cpu().numpy(), cur[i]) < tol, i
        assert rel_err(st["exp_avg"].cpu().numpy(), states[i]["exp_avg"]) < 1e-6, i
        assert rel_err(st["exp_avg_sq"].cpu().numpy(), states[i]["exp_avg_sq"]) < 1e-6, i
    assert float(opt.state[params[0]]["step"]) == 3 and float(opt.state[params[2]]["step"]) == 6


def test_chunk_table_offsets_each_pointer_by_its_own_element_size():
    from sow_b200 import ops
    n = 70001
    ce = ops._lib.load().sow_adam_chunk_elems()
    p, g = torch.zeros(n, device="cuda", dtype=torch.float16), torch.zeros(n, device="cuda", dtype=torch.float16)
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    rows = ops.build_adam_chunks([p], [g], [m], [v]).cpu().numpy()
    assert rows.shape == (3, 5)
    for k in range(3):
        assert list(rows[k, :4]) == [p.data_ptr() + 2 * k * ce, g.data_ptr() + 2 * k * ce, m.data_ptr() + 4 * k * ce,
                                     v.data_ptr() + 4 * k * ce]
    assert list(rows[:, 4]) == [ce, ce, n - 2 * ce]


@pytest.mark.parametrize("capturable", [False, True])
def test_gradscaler_parity_with_torch_fused_adamw(capturable):
    """One GradScaler drives FusedAdamW and torch.optim.AdamW(fused=True) on fp32 parameters; step 4 has an inf."""
    from sow_b200.optim import FusedAdamW
    gen = torch.Generator(device="cuda").manual_seed(0)
    shapes = [(257, 33), (4096,), (7,)]
    init = [torch.randn(s, generator=gen, device="cuda") for s in shapes]
    ours = [nn.Parameter(t.clone()) for t in init]
    ref = [nn.Parameter(t.clone()) for t in init]
    opt_a = FusedAdamW(ours, lr=1e-2, weight_decay=0.1, capturable=capturable)
    opt_b = torch.optim.AdamW(ref, lr=1e-2, weight_decay=0.1, fused=True)
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 10, growth_interval=3)
    scales, skips_a, skips_b = [], [], []
    for k in range(8):
        grads = [torch.randn(s, generator=gen, device="cuda") for s in shapes]
        if k == 4:
            grads[1][17] = float("inf")
        for p, q, gr in zip(ours, ref, grads):
            p.grad, q.grad = scaler.scale(gr), scaler.scale(gr)   # as a loss scaled by scaler.scale would produce them
        scales.append(scaler.get_scale())
        before_a, before_b = [p.detach().clone() for p in ours], [q.detach().clone() for q in ref]
        scaled = [p.grad.clone() for p in ours]
        scaler.step(opt_a)
        scaler.step(opt_b)
        scaler.update()
        skips_a.append(all(torch.equal(p, b) for p, b in zip(ours, before_a)))
        skips_b.append(all(torch.equal(q, b) for q, b in zip(ref, before_b)))
        for p, q, gr, sc in zip(ours, ref, grads, scaled):
            if skips_a[-1]:
                assert torch.equal(p.grad, sc)                  # left scaled, inf included
            else:
                assert torch.equal(p.grad, gr) and torch.equal(p.grad, q.grad)      # unscaled in place, exactly
            assert float(opt_a.state[p]["step"]) == float(opt_b.state[q]["step"])
            assert rel_err(p.detach().cpu().numpy(), q.detach().cpu().numpy()) < 1e-6
    assert skips_a == skips_b == [False] * 4 + [True] + [False] * 3
    assert scales == [1024.0] * 3 + [2048.0] * 2 + [1024.0] * 3 and scaler.get_scale() == 2048.0
    assert float(opt_a.state[ours[0]]["step"]) == 7


class _DeviceScaler:
    """What torch.amp.GradScaler does around FusedAdamW -- scale the loss, set ``grad_scale`` / ``found_inf`` on the optimizer
    for its step, back off after an inf -- with the inf / nan check written in plain torch ops and no host sync.  GradScaler's
    own check (``_amp_foreach_non_finite_check_and_unscale_``) has no bf16 kernel, so bf16 gradients are driven with this."""

    def __init__(self, init_scale):
        self._scale = torch.full((), float(init_scale), device="cuda")
        self._found = None

    def scale(self, t):
        return t * self._scale

    def step(self, opt):
        grads = [p.grad for g in opt.param_groups for p in g["params"] if p.grad is not None]
        self._found = torch.stack([(~torch.isfinite(g)).any() for g in grads]).any().float()
        opt.grad_scale, opt.found_inf = self._scale.clone(), self._found
        try:
            opt.step()
        finally:
            del opt.grad_scale, opt.found_inf

    def update(self):
        self._scale.mul_(1.0 - 0.5 * self._found)

    def get_scale(self):
        return float(self._scale)


def _scaler(pdt, init_scale, **kw):
    return _DeviceScaler(init_scale) if pdt == torch.bfloat16 else torch.amp.GradScaler("cuda", init_scale=init_scale, **kw)


def _sync_count(fn):
    """Host synchronisations fn() performs, counted by torch's CUDA sync debug mode."""
    torch.cuda.set_sync_debug_mode("warn")
    try:
        with warnings.catch_warnings(record=True) as rec:
            warnings.simplefilter("always")
            fn()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    return sum("synchroniz" in str(w.message) for w in rec)


@pytest.mark.parametrize("capturable", [False, True])
@pytest.mark.parametrize("pdt,sdt", [(torch.float16, torch.float32), (torch.bfloat16, None), (torch.bfloat16, torch.float32),
                                     (torch.float32, None)])
def test_found_inf_step_changes_no_bit(capturable, pdt, sdt):
    """fp16 / fp32 gradients: torch.amp.GradScaler; bf16 gradients: _DeviceScaler (same attribute contract)."""
    from sow_b200.optim import FusedAdamW
    gen = torch.Generator(device="cuda").manual_seed(1)
    params = [nn.Parameter((torch.randn(s, generator=gen, device="cuda") * 0.1).to(pdt)) for s in SHAPES]
    opt = FusedAdamW([{"params": params[:2]}, {"params": params[2:], "lr": 3e-3}], lr=1e-2, capturable=capturable,
                     state_dtype=sdt)
    scaler = _scaler(pdt, 2.0 ** 8)

    for p in params:
        p.grad = torch.zeros_like(p)                    # stable addresses: no chunk-table upload after the first step

    def set_grads(inf):
        for p in params:
            p.grad.copy_(scaler.scale(torch.randn(p.shape, generator=gen, device="cuda")))
        if inf:
            params[1].grad[3, 5] = float("inf")

    set_grads(False)
    scaler.step(opt)                                    # first step: creates state, counters and chunk tables
    scaler.update()
    set_grads(True)
    snap = [(_bits(p), _bits(p.grad), _bits(opt.state[p]["exp_avg"]), _bits(opt.state[p]["exp_avg_sq"]),
             float(opt.state[p]["step"])) for p in params]
    n_sync = _sync_count(lambda: scaler.step(opt))
    torch.cuda.synchronize()
    for p, (pb, gb, mb, vb, step) in zip(params, snap):
        st = opt.state[p]
        assert torch.equal(_bits(p), pb) and torch.equal(_bits(p.grad), gb)
        assert torch.equal(_bits(st["exp_avg"]), mb) and torch.equal(_bits(st["exp_avg_sq"]), vb)
        assert float(st["step"]) == step == 1
    assert n_sync == (0 if capturable else 1)
    scaler.update()
    assert scaler.get_scale() == 2.0 ** 7
    set_grads(False)
    n_sync = _sync_count(lambda: scaler.step(opt))
    assert n_sync == (0 if capturable else 1)
    torch.cuda.synchronize()
    for p, (pb, _, _, _, _) in zip(params, snap):
        assert not torch.equal(_bits(p), pb)
        assert float(opt.state[p]["step"]) == 2
        assert opt.state[p]["exp_avg"].dtype == (sdt or pdt)


@pytest.mark.parametrize("capturable", [False, True])
def test_fp32_state_checkpoint_round_trip_is_bitwise(capturable):
    from sow_b200.optim import FusedAdamW
    gen = torch.Generator(device="cuda").manual_seed(2)
    init = [(torch.randn(s, generator=gen, device="cuda") * 0.1).half() for s in SHAPES]
    grads = [[torch.randn(s, generator=gen, device="cuda").half() * 1e-2 for s in SHAPES] for _ in range(4)]

    def run_steps(params, opt, ks):
        for k in ks:
            for p, gr in zip(params, grads[k]):
                p.grad = gr.clone()
            opt.step()

    params = [nn.Parameter(t.clone()) for t in init]
    opt = FusedAdamW(params, lr=1e-2, capturable=capturable, state_dtype=torch.float32)
    run_steps(params, opt, range(3))
    sd = copy.deepcopy(opt.state_dict())
    params2 = [nn.Parameter(p.detach().clone()) for p in params]
    opt2 = FusedAdamW(params2, lr=1e-2, capturable=capturable, state_dtype=torch.float32)
    opt2.load_state_dict(sd)
    for p, q in zip(params, params2):
        for k in ("exp_avg", "exp_avg_sq"):
            assert opt2.state[q][k].dtype == torch.float32
            assert torch.equal(_bits(opt2.state[q][k]), _bits(opt.state[p][k]))
    run_steps(params, opt, [3])
    run_steps(params2, opt2, [3])
    torch.cuda.synchronize()
    for p, q in zip(params, params2):
        assert torch.equal(_bits(p), _bits(q))
        for k in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(_bits(opt.state[p][k]), _bits(opt2.state[q][k]))
        assert float(opt2.state[q]["step"]) == 4


# ---------------------------------------------------------------------------------------------------------
# SoWTrainer
# ---------------------------------------------------------------------------------------------------------

def _golden_trainer(g, dtype, **kw):
    from sow_b200.trainer import SoWTrainer, TrainConfig
    vocab, seq, batch, rank, steps, sow_acc = [int(v) for v in g["meta"][:6]]
    model = _prepared_from_golden(g, dtype)
    cfg = TrainConfig(model="llama_tiny", rank=rank, seq_len=seq, batch_size=batch, lr=1e-3, sow_lr=1e-3, weight_decay=0.0,
                      sow_accumulation=sow_acc, init_method="normal", dtype=dtype, **kw)
    return SoWTrainer(cfg, torch.device("cuda", 0), model=model, targets=TARGETS), steps


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_power_of_two_loss_scale_is_exact(dtype):
    """Multiplying by 2^k commutes with round-to-nearest away from overflow and the subnormal range, and fp32 and bf16 share
    that exponent range: the scaled backward gives 2^8 times the gradients, bit for bit, and the kernel's division undoes it.
    fp32: SoWTrainer's loss scaling with torch.amp.GradScaler; bf16 (which GradScaler cannot check): the same trainer loop
    and optimizer path driven by _DeviceScaler."""
    g = _golden()
    runs = []
    for scaled in (False, True):
        torch.manual_seed(0)
        tr, steps = _golden_trainer(g, dtype, cuda_graph=True, loss_scaling=scaled and dtype == torch.float32,
                                    loss_scale_init=2.0 ** 8, loss_scale_growth_interval=1000)
        tr.cfg.cuda_graph = False                       # capturable optimizer in both arms, eager steps
        if scaled and dtype == torch.bfloat16:
            tr.scaler = _DeviceScaler(2.0 ** 8)
        torch.manual_seed(1)                            # the merges draw new factors
        losses = [tr.step(torch.from_numpy(g["batches"][s]).to("cuda")).clone() for s in range(steps)]
        torch.cuda.synchronize()
        assert tr.merges == 2
        if scaled:
            assert tr.scaler.get_scale() == 2.0 ** 8
        runs.append((losses, {n: _bits(p) for n, p in tr.model.named_parameters()}))
    (l0, p0), (l1, p1) = runs
    assert all(torch.equal(a, b) for a, b in zip(l0, l1)), ([float(v) for v in l0], [float(v) for v in l1])
    assert set(p0) == set(p1)
    for n in p0:
        assert torch.equal(p0[n], p1[n]), n


def test_fp16_trainer_with_fp32_state_and_loss_scaling_matches_reference():
    """The golden-trajectory protocol of test_trainer_loss_trajectory_matches_reference in fp16, with fp32 Adam moments and
    loss scaling (no step skipped at this scale), to the bf16 bounds: all losses through both merges, and the first merge."""
    from tn_gradient.layer.sow import SoWLinear
    g = _golden()
    want = [float(v) for v in g["losses"]]
    reports = {}
    for name, kw in (("fp32 state", dict(optimizer_state_dtype=torch.float32)),
                     ("fp32 state + loss scaling", dict(optimizer_state_dtype=torch.float32, loss_scaling=True,
                                                        loss_scale_init=2.0 ** 12))):
        tr, steps = _golden_trainer(g, torch.float16, **kw)
        losses, merge_err = [], None
        for step in range(1, steps + 1):
            merges_before = tr.merges
            losses.append(float(tr.step(torch.from_numpy(g["batches"][step - 1]).to("cuda"))))
            if tr.merges > merges_before and tr.merges == 1:
                merge_err = max(rel_err(m.acc_downweight.float().cpu().numpy(), g[f"merged{step}/{n}.acc_downweight"])
                                for n, m in tr.model.named_modules() if isinstance(m, SoWLinear))
        assert tr.merges == 2
        reports[name] = (losses, merge_err, tr)
        print(f"{name}: losses {losses} (reference {want}), first merge max rel. error {merge_err:.3e}")
    losses, merge_err, tr = reports["fp32 state + loss scaling"]
    assert tr.scaler.get_scale() == 2.0 ** 12                    # no step was skipped
    for s, (a, b) in enumerate(zip(losses, want)):
        assert abs(a - b) / abs(b) < 2e-2, (s, a, b)
    assert merge_err < 2e-2
    sp = tr.optimizer.state[tr.special[0]]
    assert sp["exp_avg"].dtype == torch.float32 and sp["exp_avg_sq"].dtype == torch.float32


def test_fp16_loss_scaled_trainer_cuda_graph_replay_is_bit_identical_to_eager():
    """fp16 trainer, fp32 moments, dynamic loss scaling from 2^30: the first steps overflow and back the scale off, inside
    the replays too.  Graph replay and eager steps agree bit for bit (losses, parameters, moments, scale)."""
    from sow_b200.trainer import SoWTrainer, TrainConfig
    runs = []
    for graphed in (False, True):
        cfg = TrainConfig(model="llama_9m", rank=8, seq_len=64, batch_size=4, lr=1e-3, sow_lr=1e-3, sow_accumulation=100,
                          init_method="normal", cuda_graph=True, seed=1, dtype=torch.float16,
                          optimizer_state_dtype=torch.float32, loss_scaling=True, loss_scale_init=2.0 ** 30)
        torch.manual_seed(0)
        tr = SoWTrainer(cfg, torch.device("cuda", 0))
        tr.cfg.cuda_graph = graphed
        gen = torch.Generator().manual_seed(3)
        losses, scales = [], []
        for _ in range(32):
            ids = torch.randint(1, 32000, (4, 64), generator=gen).cuda()
            losses.append(tr.step(ids).detach().clone())
            scales.append(tr.scaler.get_scale())
        torch.cuda.synchronize()
        assert (tr._graph is not None) == graphed
        moments = {n: (_bits(tr.optimizer.state[p]["exp_avg"]), _bits(tr.optimizer.state[p]["exp_avg_sq"]))
                   for n, p in tr.model.named_parameters() if p in tr.optimizer.state}
        runs.append((losses, scales, {n: _bits(p) for n, p in tr.model.named_parameters()}, moments))
    (le, se, pe, me), (lg, sg, pg, mg) = runs
    print(f"scales {sg}")
    assert se == sg
    skipped_in_replay = [k for k in range(2, 32) if sg[k] < sg[k - 1]]       # call k (a replay from k = 2) backed off
    taken_in_replay = [k for k in range(2, 32) if sg[k] >= sg[k - 1]]
    assert skipped_in_replay and taken_in_replay, sg
    assert all(torch.equal(a, b) for a, b in zip(le, lg)), ([float(v) for v in le], [float(v) for v in lg])
    assert set(pe) == set(pg) and set(me) == set(mg) and me
    for n in pe:
        assert torch.equal(pe[n], pg[n]), n
    for n in me:
        assert torch.equal(me[n][0], mg[n][0]) and torch.equal(me[n][1], mg[n][1]), n
