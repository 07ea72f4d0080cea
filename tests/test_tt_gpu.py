"""GPU parity: TensorTrain decompose / reconstruct and TTAdam / TTSGD through the public tn_gradient API against
the reference's golden outputs, its known-answer values (BASELINE.md section 2) and the CPU oracle.

Criterion (BASELINE.json north_star): TT reconstruction error within 1e-5 relative of the reference's; compare
reconstructions / errors, never cores (the decomposition is gauge-invariant)."""
import numpy as np
import pytest
import torch

from conftest import rel_err, tt_matrix
from oracle import sow_oracle as O

pytestmark = pytest.mark.gpu


def test_arange_known_answer(golden_tt):
    """tests/tt_test.py: from_tensor(arange(216).reshape(2,2,2,3,3,3), [1,4,4,1]) reconstructs to ~1.6e-07."""
    from tn_gradient.tt import TensorTrain
    g = golden_tt
    A = torch.from_numpy(g["tt/arange/tensor"]).cuda()
    tt = TensorTrain.from_tensor(A, [1, 4, 4, 1])
    assert [tuple(c.shape) for c in tt.cores] == [tuple(g[f"tt/arange/core{i}"].shape) for i in range(3)]
    rec = tt.reconstruct()
    assert rec.shape == A.shape
    err = float((rec - A).norm() / A.norm())
    assert err < 5e-7                                   # reference prints 1.59e-07
    assert rel_err(rec.cpu().numpy(), g["tt/arange/reconstruct"]) < 1e-6
    # compat algebra on GPU cores + kernel reconstruct
    assert rel_err((tt + tt).reconstruct().cpu().numpy(), g["tt/arange/add_rec"]) < 1e-6
    assert rel_err((tt * tt).reconstruct().cpu().numpy(), g["tt/arange/mul_rec"]) < 1e-6
    assert rel_err((2.5 * tt).reconstruct().cpu().numpy(), g["tt/arange/scaled_rec"]) < 1e-6


@pytest.mark.parametrize("case", ["m81_r4", "m81_r9", "m100x60", "m256_o3", "m300x200", "m256x192", "m130x70_pad"])
def test_from_matrix_to_matrix_vs_reference(golden_tt, case):
    from tn_gradient.tt import TensorTrain
    g = golden_tt
    mat_np = tt_matrix(g, case)
    ranks = [int(r) for r in g[f"tt/{case}/ranks"]]
    mat = torch.from_numpy(mat_np).cuda()
    tt = TensorTrain.from_matrix(mat, list(ranks))
    assert [list(c.shape) for c in tt.cores] == g[f"tt/{case}/core_shapes"].tolist()
    assert all(c.dtype == torch.float32 for c in tt.cores)
    back = tt.to_matrix(mat.shape)
    assert back.shape == mat.shape
    assert rel_err(back.cpu().numpy()[::int(g["tt/to_matrix_row_step"])], g[f"tt/{case}/to_matrix_rows"]) < 2e-5
    err = float((back - mat).norm() / mat.norm())
    ref_err = float(g[f"tt/{case}/rel_err"])
    assert abs(err - ref_err) <= 1e-5 * ref_err, (err, ref_err)      # the north-star criterion
    # left cores are orthonormal (left-unfolding has orthonormal columns)
    for k in range(len(ranks) - 2):
        L = tt.left_matrix(k)
        eye = torch.eye(L.shape[1], device="cuda")
        assert float((L.T @ L - eye).abs().max()) < 1e-5


def test_adam_update_script_known_answers(golden_tt):
    """tests/tt_adam_update.py: 81x81 gradient, order 4, ranks [1,4,4,4,1]: "TT decomposition error" ~8.6e-05."""
    from tn_gradient.tt import TensorTrain
    g = golden_tt
    grad = torch.from_numpy(g["tt/kat_adam_update/grad"]).cuda()
    tt = TensorTrain.from_matrix(grad, [1, 4, 4, 4, 1])
    back = tt.to_matrix(grad.shape)
    abs_err = float(torch.linalg.norm(back - grad))
    assert abs_err < 2e-4, abs_err                        # reference (fp32 LAPACK): 8.60e-05; exact arithmetic: 6.2e-05
    assert rel_err(back.cpu().numpy(), g["tt/kat_adam_update/reconstruct"]) < 1e-4


@pytest.mark.parametrize("case", ["o2", "o3", "o2_pad"])
def test_ttadam_trajectory_vs_reference(golden_tt, case):
    from tn_gradient.optimizer.ttadam import TTAdam
    from tn_gradient.tt import TensorTrain
    g = golden_tt
    ranks = [int(r) for r in g[f"ttadam/{case}/ranks"]]
    wd = float(g[f"ttadam/{case}/wd"])
    p = torch.nn.Parameter(torch.from_numpy(g[f"ttadam/{case}/p0"]).cuda())
    opt = TTAdam([{"params": [p], "ranks": list(ranks)}], lr=1e-2, weight_decay=wd)
    for step, grad in enumerate(g[f"ttadam/{case}/grads"]):
        p.grad = torch.from_numpy(grad).cuda()
        opt.step()
        torch.cuda.synchronize()
        assert rel_err(p.detach().cpu().numpy(), g[f"ttadam/{case}/p{step + 1}"]) < 2e-5, step
    st = opt.state[p]
    assert isinstance(st["exp_avg"], TensorTrain) and isinstance(st["exp_avg_sq"], TensorTrain) and st["step"] == 5
    assert all(c.dtype == torch.float32 for c in st["exp_avg"].cores)
    assert rel_err(st["exp_avg"].to_matrix(p.shape).cpu().numpy(), g[f"ttadam/{case}/m_final"]) < 1e-4
    assert rel_err(st["exp_avg_sq"].to_matrix(p.shape).cpu().numpy(), g[f"ttadam/{case}/v_final"]) < 1e-4


def test_ttadam_dense_branch_vs_reference(golden_tt):
    from tn_gradient.optimizer.ttadam import TTAdam
    g = golden_tt
    p = torch.nn.Parameter(torch.from_numpy(g["ttadam/dense/p0"]).cuda())
    opt = TTAdam([p], lr=1e-2)
    for grad in g["ttadam/dense/grads"]:
        p.grad = torch.from_numpy(grad).cuda()
        opt.step()
    assert rel_err(p.detach().cpu().numpy(), g["ttadam/dense/p3"]) < 2e-6


def test_ttadam_bf16_param_within_bf16_tolerance(golden_tt):
    from tn_gradient.optimizer.ttadam import TTAdam
    g = golden_tt
    p = torch.nn.Parameter(torch.from_numpy(g["ttadam/o2/p0"]).cuda().bfloat16())
    opt = TTAdam([{"params": [p], "ranks": [1, 8, 1]}], lr=1e-2)
    for step, grad in enumerate(g["ttadam/o2/grads"]):
        p.grad = torch.from_numpy(grad).cuda().bfloat16()
        opt.step()
    assert rel_err(p.detach().float().cpu().numpy(), g["ttadam/o2/p5"]) < 2e-2


def test_ttsgd_vs_reference(golden_tt):
    from tn_gradient.optimizer.ttsgd import TTSGD
    g = golden_tt
    p = torch.nn.Parameter(torch.from_numpy(g["ttsgd/p0"]).cuda())
    opt = TTSGD([{"params": [p], "ranks": [1, 12, 1]}], lr=1e-2, momentum=0.9, nesterov=True)
    for grad in g["ttsgd/grads"]:
        p.grad = torch.from_numpy(grad).cuda()
        opt.step()
    assert rel_err(p.detach().cpu().numpy(), g["ttsgd/p3"]) < 2e-5


@pytest.mark.parametrize("M,N,ranks", [(4096, 4096, [1, 8, 1]), (4096, 4096, [1, 64, 1]), (4096, 11008, [1, 16, 1]),
                                        (4096, 4096, [1, 16, 16, 1]), (1024, 2736, [1, 8, 8, 8, 1])])
def test_full_size_properties(M, N, ranks):
    """Llama-7B-shaped sweep (BASELINE.json configs[4]) through size-independent properties: projection
    idempotence (decompose(reconstruct(tt)) reconstructs to the same matrix), error monotone in rank, orthonormal
    left cores, zero padding preserved."""
    from tn_gradient.tt import TensorTrain
    torch.manual_seed(0)
    mat = torch.randn(M, N, device="cuda")
    tt = TensorTrain.from_matrix(mat, list(ranks))
    back = tt.to_matrix((M, N))
    err = float((back - mat).norm() / mat.norm())
    assert 0.0 < err < 1.0
    order = len(ranks) - 1
    mm, nn_ = tt.input_shape[0], tt.output_shape[0]
    if mm ** order == M and nn_ ** order == N:
        # no zero padding -> the truncated-QR sweep is a projection: decomposing its own output changes nothing
        back2 = TensorTrain.from_matrix(back, list(ranks)).to_matrix((M, N))
        assert float((back2 - back).norm() / back.norm()) < 2e-5
    else:
        # padded: the full padded reconstruction is what is idempotent
        full = tt.reconstruct().reshape(mm ** order, nn_ ** order)
        assert torch.equal(full[:M, :N], back)
        tt2 = TensorTrain.from_matrix(full, list(ranks))
        assert float((tt2.reconstruct().reshape(mm ** order, nn_ ** order) - full).norm() / full.norm()) < 2e-5
    big = [1] + [2 * r for r in ranks[1:-1]] + [1]
    err_big = float((TensorTrain.from_matrix(mat, big).to_matrix((M, N)) - mat).norm() / mat.norm())
    assert err_big < err
    for k in range(len(ranks) - 2):
        L = tt.left_matrix(k)
        assert float((L.T @ L - torch.eye(L.shape[1], device="cuda")).abs().max()) < 2e-5


def test_projection_matches_oracle_at_4096(golden_tt):
    """4096 x 4096, order 2, rank 16 against the oracle's complete-QR restatement on the same matrix."""
    from tn_gradient.tt import TensorTrain
    rng = np.random.default_rng(5)
    ema = np.zeros((1024, 1024), dtype=np.float32)
    for _ in range(4):                                   # Adam-moment-like input (SURVEY.md 8d)
        ema = 0.9 * ema + 0.1 * rng.standard_normal((1024, 1024), dtype=np.float32)
    tt = TensorTrain.from_matrix(torch.from_numpy(ema).cuda(), [1, 16, 1])
    back = tt.to_matrix(ema.shape).cpu().numpy()
    back_o = O.tt_to_matrix(O.tt_from_matrix(ema, [1, 16, 1]), ema.shape)
    assert rel_err(back, back_o) < 1e-5
    e, eo = rel_err(back, ema), rel_err(back_o, ema)
    assert abs(e - eo) <= 1e-5 * eo


@pytest.mark.parametrize("r,force_tc", [(8, "0"), (32, "1"), (64, "1"), (48, "0")])
def test_ttadam_step_is_bit_reproducible(r, force_tc, monkeypatch):
    """Every cross-CTA sum on the TT path is a fixed-order sum of split partials (Gram of the thin QR, the projections,
    the R' accumulation of both fused TT-Adam kernels): the same inputs give the same bits, run after run."""
    from sow_b200 import ops
    monkeypatch.setenv("SOWB_TT_TC", force_tc)
    M = N = 1024
    mm = nn_ = 32
    torch.manual_seed(3)
    p0 = torch.randn(M, N, device="cuda").to(torch.bfloat16)
    g = (0.01 * torch.randn(M, N, device="cuda")).to(torch.bfloat16)
    outs = []
    for _ in range(3):
        p = p0.clone()
        (Qm, Rm), (Qv, Rv) = ops.tt_adam2_step(p, g, None, None, mm, nn_, r, 0.9, 0.999, 1e-8, 1e-3, 0.0, True)
        cm, cv = (Qm.clone(), Rm.clone()), (Qv.clone(), Rv.clone())
        (Qm2, Rm2), (Qv2, Rv2) = ops.tt_adam2_step(p, g, cm, cv, mm, nn_, r, 0.9, 0.999, 1e-8, 1e-3, 0.0, False)
        outs.append([t.clone() for t in (p, Qm, Rm, Qv, Rv, Qm2, Rm2, Qv2, Rv2)])
    for other in outs[1:]:
        for a, b in zip(outs[0], other):
            assert torch.equal(a, b)


def test_decompose_is_bit_reproducible():
    from sow_b200 import ops
    torch.manual_seed(4)
    mat = torch.randn(4096, 4096, device="cuda")
    ref = None
    for _ in range(3):
        Q, R = ops.decompose2(mat, 64, 64, 16)
        L = torch.randn(2, 4096, 512, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
        Qb = ops.thin_qr(L, 24)
        Rb = ops.project(L, Qb)
        cur = [Q.clone(), R.clone(), Qb.clone(), Rb.clone()]
        if ref is None:
            ref = cur
        for a, b in zip(ref, cur):
            assert torch.equal(a, b)


@pytest.mark.parametrize("case", ["o2", "o3"])
def test_ttadam_plan_survives_replaced_and_reset_state(golden_tt, case):
    """The one-call paths (order 2 and order >= 3) keep persistent core buffers per parameter.  Moments that were replaced behind its back (a
    loaded checkpoint) must be picked up, and a cleared state must restart from zero moments: both runs reproduce the
    uninterrupted trajectory bit for bit."""
    from tn_gradient.optimizer.ttadam import TTAdam
    from tn_gradient.tt import TensorTrain
    g = golden_tt
    grads = [torch.from_numpy(x).cuda() for x in g[f"ttadam/{case}/grads"]]
    ranks = [int(r) for r in g[f"ttadam/{case}/ranks"]]
    wd = float(g[f"ttadam/{case}/wd"])

    def run(interfere):
        p = torch.nn.Parameter(torch.from_numpy(g[f"ttadam/{case}/p0"]).cuda())
        opt = TTAdam([{"params": [p], "ranks": list(ranks)}], lr=1e-2, weight_decay=wd)
        for step, grad in enumerate(grads):
            p.grad = grad
            opt.step()
            if interfere and step == 1:
                st = opt.state[p]
                for key in ("exp_avg", "exp_avg_sq"):                 # what load_state_dict leaves behind
                    st[key] = TensorTrain.from_cores([c.clone() for c in st[key].cores])
        return p.detach().clone(), [c.clone() for c in opt.state[p]["exp_avg"].cores]

    p_ref, cores_ref = run(False)
    p_int, cores_int = run(True)
    assert torch.equal(p_ref, p_int)
    for a, b in zip(cores_ref, cores_int):
        assert torch.equal(a, b)
    assert rel_err(p_ref.cpu().numpy(), g[f"ttadam/{case}/p5"]) < 2e-5

    # reset: clearing the state restarts from zero moments (the plan's stale cores must not leak in)
    p = torch.nn.Parameter(torch.from_numpy(g[f"ttadam/{case}/p0"]).cuda())
    opt = TTAdam([{"params": [p], "ranks": list(ranks)}], lr=1e-2, weight_decay=wd)
    p.grad = grads[0]
    opt.step()
    p1 = p.detach().clone()
    opt.state[p].clear()
    with torch.no_grad():
        p.copy_(torch.from_numpy(g[f"ttadam/{case}/p0"]).cuda())
    opt.step()
    assert torch.equal(p.detach(), p1)


def test_ttadam_side_streams_do_not_change_the_result(monkeypatch):
    """Several tensor-train parameters alternate between side streams inside TTAdam.step (the small QR chain of one overlaps the
    large kernel of another); the parameters are independent, so the result is bit-identical to the one-stream order."""
    from tn_gradient.optimizer.ttadam import TTAdam

    def run(streams):
        monkeypatch.setenv("SOWB_TT_STREAMS", str(streams))
        torch.manual_seed(11)
        ps = [torch.nn.Parameter(torch.randn(256, 320, device="cuda")) for _ in range(5)]
        ps.append(torch.nn.Parameter(torch.randn(64, device="cuda")))            # a dense one in the same optimizer
        opt = TTAdam([{"params": ps[:5], "ranks": [1, 8, 1]}, {"params": ps[5:]}], lr=1e-2)
        for step in range(4):
            gen = torch.Generator(device="cuda").manual_seed(100 + step)
            for p in ps:
                p.grad = torch.randn(p.shape, device="cuda", generator=gen)
            opt.step()
        torch.cuda.synchronize()
        return [p.detach().clone() for p in ps]

    ref = run(1)
    for streams in (2, 4):
        for a, b in zip(ref, run(streams)):
            assert torch.equal(a, b)
