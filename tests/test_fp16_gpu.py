"""GPU: float16 modules end to end -- fused AdamW on fp16 parameters, the model-level trajectory against the reference,
checkpoints, torch.compile, memory (no bf16 shadow of W) and a CUDA-graph trainer step, all in fp16."""

import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import rel_err
from oracle import sow_oracle as O
from test_optim_loop_gpu import reset_optimizer
from test_trajectory_gpu import TARGETS, _golden, _prepared_from_golden

pytestmark = pytest.mark.gpu


def f16_round(a):
    return np.asarray(a, np.float64).astype(np.float16).astype(np.float64)


# ---------------------------------------------------------------------------------------------------------
# fused AdamW
# ---------------------------------------------------------------------------------------------------------

def test_fused_adamw_fp16_vs_oracle_with_reset():
    from sow_b200.optim import FusedAdamW
    rng = np.random.default_rng(0)
    shapes = [(1024, 50), (50, 2736), (33,), (70001,)]
    ps_np = [f16_round(rng.standard_normal(s) * 0.1) for s in shapes]
    params = [nn.Parameter(torch.from_numpy(p).to("cuda", torch.float16)) for p in ps_np]
    opt = FusedAdamW([{"params": params[:2], "lr": 1e-2, "weight_decay": 0.1},
                      {"params": params[2:], "lr": 3e-3, "weight_decay": 0.0}])
    states = [dict() for _ in shapes]
    cur = [p.copy() for p in ps_np]
    for step in range(6):
        grads = [f16_round(rng.standard_normal(s)) for s in shapes]
        for p, gr in zip(params, grads):
            p.grad = torch.from_numpy(gr).to("cuda", torch.float16)
        if step == 3:
            reset_optimizer(opt, 0)                     # merge step: moments of group 0 rebound to fresh zeros
            states[0], states[1] = {}, {}
        opt.step()
        for i in range(len(shapes)):
            lr, wd = (1e-2, 0.1) if i < 2 else (3e-3, 0.0)
            cur[i] = f16_round(O.adamw_step(cur[i], grads[i], states[i], lr, weight_decay=wd))   # fp16 between steps
    torch.cuda.synchronize()
    for p, c in zip(params, cur):
        assert p.dtype == torch.float16
        assert rel_err(p.detach().float().cpu().numpy(), c) < 2e-3
    st = opt.state[params[0]]
    assert st["exp_avg"].dtype == torch.float16 and st["exp_avg_sq"].dtype == torch.float16
    assert float(st["step"]) == 3 and float(opt.state[params[2]]["step"]) == 6


def test_fused_adamw_fp16_capturable_graph_replay_is_bit_identical_to_eager():
    from sow_b200.optim import FusedAdamW
    g = torch.Generator(device="cuda").manual_seed(0)
    shapes = [(1024, 50), (50, 2736), (33,), (70001,)]
    init = [(torch.randn(s, generator=g, device="cuda") * 0.1).half() for s in shapes]
    grads = [[torch.randn(s, generator=g, device="cuda").half() for s in shapes] for _ in range(5)]
    runs = []
    for graphed in (False, True):
        params = [nn.Parameter(t.clone()) for t in init]
        for p in params:
            p.grad = torch.zeros_like(p)
        opt = FusedAdamW([{"params": params[:2], "lr": 1e-2, "weight_decay": 0.1},
                          {"params": params[2:], "lr": 3e-3, "weight_decay": 0.0}], capturable=True)

        def load(k):
            for p, gr in zip(params, grads[k]):
                p.grad.copy_(gr)

        load(0)
        opt.step()                                      # first step eager: builds the device counters and chunk tables
        if graphed:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.stream(side), torch.cuda.graph(graph):
                opt.step()
            torch.cuda.current_stream().wait_stream(side)
        for k in range(1, 5):
            load(k)
            if graphed:
                graph.replay()
            else:
                opt.step()
        torch.cuda.synchronize()
        runs.append([(p.detach().clone(), opt.state[p]["exp_avg"].clone(), opt.state[p]["exp_avg_sq"].clone())
                     for p in params])
    for a, b in zip(*runs):
        for x, y in zip(a, b):
            assert torch.equal(x.view(torch.int16), y.view(torch.int16))


# ---------------------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------------------

def test_fp16_trainer_matches_reference_until_adam_state_underflows():
    """The golden-trajectory protocol in fp16.  The first two losses (forward and backward through every SoW kernel, one
    optimizer step) agree with the reference to 1e-2.  From the third step on the trajectory leaves the fp32 reference:
    AdamW keeps exp_avg_sq in fp16 (as torch.optim.AdamW does for fp16 parameters), (1 - beta2) * g^2 underflows to 0 for
    |g| below ~8e-3, and an element whose gradient then vanishes moves by lr * m / eps.  Training fp16 weights with Adam
    needs loss scaling or fp32 state, which this protocol (model.half(), no GradScaler) does not use."""
    from sow_b200.trainer import SoWTrainer, TrainConfig
    g = _golden()
    vocab, seq, batch, rank, steps, sow_acc = [int(v) for v in g["meta"][:6]]
    model = _prepared_from_golden(g, torch.float16)
    cfg = TrainConfig(model="llama_tiny", rank=rank, seq_len=seq, batch_size=batch, lr=1e-3, sow_lr=1e-3, weight_decay=0.0,
                      sow_accumulation=sow_acc, init_method="normal", dtype=torch.float16)
    tr = SoWTrainer(cfg, torch.device("cuda", 0), model=model, targets=TARGETS)
    losses = [float(tr.step(torch.from_numpy(g["batches"][s]).to("cuda"))) for s in range(2)]
    want = g["losses"]
    print(f"losses fp16 {losses} reference {[float(v) for v in want[:2]]}")
    for s, (a, b) in enumerate(zip(losses, want)):
        assert abs(a - b) / abs(b) < 1e-2, (s, a, b)


def test_fp16_model_merge_does_not_go_through_bf16():
    """First merge of every SoW layer of the golden model (W = s * A . B): the fp16 result is within 1e-2 of fp64 and more
    than twice as close as the bf16 model's -- the merge rounds once to fp16, not through bf16."""
    from tn_gradient.layer.sow import SoWLinear
    from tn_gradient.prepare import accumulate
    g = _golden()
    errs = {}
    for dt in (torch.float16, torch.bfloat16):
        model = _prepared_from_golden(g, dt)
        refs = {}
        for name, m in model.named_modules():
            if isinstance(m, SoWLinear):
                A = m.downscale_weights[0].detach().double()
                B = m.upscale_weights[0].detach().double()
                refs[name] = (m.scale * (A @ B)).cpu().numpy()
        accumulate(model)
        num = den = 0.0
        for name, m in model.named_modules():
            if isinstance(m, SoWLinear):
                assert m.acc_downweight.dtype == dt
                got = m.acc_downweight.double().cpu().numpy()
                num += float(((got - refs[name]) ** 2).sum())
                den += float((refs[name] ** 2).sum())
        errs[dt] = (num / den) ** 0.5
    print(f"first merge, relative error vs fp64: fp16 {errs[torch.float16]:.3e}, bf16 {errs[torch.bfloat16]:.3e}")
    assert errs[torch.float16] < 1e-2
    assert errs[torch.float16] < 0.5 * errs[torch.bfloat16]


def test_fp16_checkpoint_round_trip_is_bit_identical(tmp_path):
    from safetensors.torch import save_file
    from tn_gradient.prepare import accumulate, load_sow
    g = _golden()
    model = _prepared_from_golden(g, torch.float16)
    ids = torch.from_numpy(g["batches"][0]).to("cuda")
    accumulate(model)
    with torch.no_grad():
        for m in model.modules():
            if hasattr(m, "upscale_weights"):
                m.upscale_weights[0].normal_(0, 0.02)
    layers = {n: m for n, m in model.named_modules() if hasattr(m, "acc_downweight")}
    ptrs = {n: (m.acc_downweight.data_ptr(), id(m.acc_downweight)) for n, m in layers.items()}
    accumulate(model)                                   # second merge: in place, same storage and same Parameter
    assert all((m.acc_downweight.data_ptr(), id(m.acc_downweight)) == ptrs[n] for n, m in layers.items())
    assert all(m.acc_downweight.dtype == torch.float16 for m in layers.values())
    with torch.no_grad():
        ref_logits = model(input_ids=ids).logits.clone()
    path = str(tmp_path / "model.safetensors")
    save_file({k: v.detach().contiguous() for k, v in model.state_dict().items()}, path)
    fresh = _prepared_from_golden(g, torch.float16)
    with torch.no_grad():
        fresh(input_ids=ids)
    load_sow(fresh, path)
    with torch.no_grad():
        assert torch.equal(fresh(input_ids=ids).logits, ref_logits)


def test_fp16_model_under_torch_compile_is_bit_identical_to_eager():
    import torch._dynamo
    from tn_gradient.prepare import SoWConfig, prepare_sow
    torch.manual_seed(0)
    m = nn.Sequential(nn.Linear(256, 512), nn.GELU(), nn.Linear(512, 256))
    m = prepare_sow(m, SoWConfig(target_modules=["0", "2"], rank=8, device="cuda", init_method="normal",
                                 decompose="keep")).to("cuda", torch.float16)
    x = torch.randn(64, 256, device="cuda", dtype=torch.float16, requires_grad=True)
    y0 = m(x)
    y0.float().pow(2).mean().backward()
    g0 = x.grad.clone()
    gp0 = {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}
    assert y0.dtype == torch.float16 and all(v.dtype == torch.float16 for v in gp0.values())
    x.grad = None
    m.zero_grad()
    torch._dynamo.reset()
    ex = torch._dynamo.explain(m)(x)
    assert ex.graph_break_count == 0, ex.break_reasons
    y1 = torch.compile(m, fullgraph=True)(x)
    y1.float().pow(2).mean().backward()
    assert torch.equal(y0, y1) and torch.equal(g0, x.grad)
    for n, p in m.named_parameters():
        if n in gp0:
            assert torch.equal(gp0[n], p.grad), n


def test_fp16_forward_makes_no_copy_of_W():
    """First forward of a keep-mode fp16 module: the only new memory is the output and what autograd saves (A_cat, t_cat;
    x is saved as it is).  A compute copy of W would add in * out * 2 bytes."""
    from tn_gradient.prepare import SoWConfig, prepare_sow
    fin = fout = 4096
    torch.manual_seed(0)
    m = prepare_sow(nn.Sequential(nn.Linear(fin, fout, bias=False)),
                    SoWConfig(target_modules=["0"], rank=8, device="cuda", init_method="normal", decompose="keep"))
    m = m.to("cuda", torch.float16)
    layer = m[0]
    assert layer.acc_downweight.dtype == torch.float16 and layer.acc_downweight.numel() == fin * fout
    x = torch.randn(64, fin, device="cuda", dtype=torch.float16)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    y = m(x)
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    print(f"first fp16 forward: {extra} B beyond the inputs (W is {fin * fout * 2} B)")
    assert y.dtype == torch.float16
    assert extra < fin * fout * 2
    assert layer._w_shadow is None


def test_fp16_trainer_cuda_graph_replay_is_bit_identical_to_eager():
    """Two trainers built for CUDA graphs (capturable optimizer); one runs every step eagerly, the other captures step 3
    and replays it from there."""
    from sow_b200.trainer import SoWTrainer, TrainConfig
    runs = []
    for graphed in (False, True):
        cfg = TrainConfig(model="llama_9m", rank=8, seq_len=64, batch_size=4, lr=1e-3, sow_lr=1e-3, sow_accumulation=100,
                          init_method="normal", cuda_graph=True, seed=1, dtype=torch.float16)
        torch.manual_seed(0)
        tr = SoWTrainer(cfg, torch.device("cuda", 0))
        tr.cfg.cuda_graph = graphed
        g = torch.Generator().manual_seed(3)
        losses = []
        for _ in range(6):
            ids = torch.randint(1, 32000, (4, 64), generator=g).cuda()
            losses.append(tr.step(ids).detach().clone())
        torch.cuda.synchronize()
        assert (tr._graph is not None) == graphed
        runs.append((losses, {n: p.detach().clone() for n, p in tr.model.named_parameters()}))
    (le, pe), (lg, pg) = runs
    assert all(torch.equal(a, b) for a, b in zip(le, lg)), ([float(v) for v in le], [float(v) for v in lg])
    assert set(pe) == set(pg)
    for n in pe:
        assert pe[n].dtype == torch.float16 or pe[n].numel() == 0, n
        assert torch.equal(pe[n], pg[n]), n


# ---------------------------------------------------------------------------------------------------------
# tensor-train path: bf16 / fp32 only
# ---------------------------------------------------------------------------------------------------------

def test_ttadam_still_rejects_fp16_parameters():
    from sow_b200._lib import SowB200Error
    from tn_gradient.optimizer.ttadam import TTAdam
    p = nn.Parameter(torch.randn(64, 48, device="cuda").half())
    p.grad = torch.randn(64, 48, device="cuda").half()
    opt = TTAdam([{"params": [p], "ranks": [1, 8, 1]}], lr=1e-2)
    with pytest.raises(SowB200Error):
        opt.step()
