"""Pin the CPU oracle (oracle/sow_oracle.py) against outputs of the unmodified reference (tests/golden/*.npz,
made by tests/golden/make_golden.py) and the known-answer values of the reference's own test scripts
(BASELINE.md section 2).  CPU only."""
import numpy as np
import pytest

from conftest import rel_err, tt_matrix
from oracle import sow_oracle as O

LINEAR_CASES = ["f32_w_bias", "f32_now", "f32_niter2", "bf16_w", "bf16_now_bias"]


@pytest.mark.parametrize("case", LINEAR_CASES)
def test_linear_forward_backward_matches_reference(golden_linear, case):
    g = golden_linear
    p = f"linear/{case}/"
    n_iter = int(g[p + "n_iter"])
    As = [g[p + f"A{i}"] for i in range(n_iter)]
    Bs = [g[p + f"B{i}"] for i in range(n_iter)]
    W = g[p + "W"] if (p + "W") in g else None
    bias = g[p + "bias"] if (p + "bias") in g else None
    scale = float(g[p + "scale"])
    # the reference's own bf16 run differs from exact math by ~3e-3 (SURVEY.md section 7); fp32 by ~1e-6
    tol = 2e-2 if case.startswith("bf16") else 2e-6
    y = O.sow_linear_forward(g[p + "x"], W, As, Bs, bias, scale)
    assert y.shape == g[p + "y"].shape
    assert rel_err(y, g[p + "y"]) < tol
    dx, dAs, dBs, dbias = O.sow_linear_backward(g[p + "dy"], g[p + "x"], W, As, Bs, scale)
    assert rel_err(dx, g[p + "dx"]) < tol
    for i in range(n_iter):
        assert rel_err(dAs[i], g[p + f"dA{i}"]) < tol
        assert rel_err(dBs[i], g[p + f"dB{i}"]) < tol
    if bias is not None:
        assert rel_err(dbias, g[p + "dbias"]) < tol


@pytest.mark.parametrize("case", ["dense_f32", "dense_bf16", "dense_niter2_f32", "factored_f32", "factored_bf16"])
def test_merge_matches_reference(golden_merge, case):
    g = golden_merge
    fin, fout, r, n_iter = [int(v) for v in g[f"merge/{case}/meta"]]
    scale = float(g[f"merge/{case}/scale"])
    tol = 1e-2 if "bf16" in case else 5e-6
    for step in range(3):
        p = f"merge/{case}/step{step}/"
        As = [g[p + f"A{i}"] for i in range(n_iter)]
        Bs = [g[p + f"B{i}"] for i in range(n_iter)]
        W_prev, Wup_prev = g[p + "W_prev"], g[p + "Wup_prev"]
        vr = int(g[p + "virtual_rank_prev"])
        W, Wup, vr_new = O.sow_merge(W_prev if W_prev.size else None, As, Bs, scale,
                                     W_up=Wup_prev if Wup_prev.size else None, virtual_rank=vr, rank=r)
        assert vr_new == int(g[p + "virtual_rank"])
        if Wup is None:
            assert g[p + "Wup"].size == 0
            assert rel_err(W, g[p + "W"]) < tol
        else:
            # factored branch: Q, R individually (same LAPACK Householder convention) and their product
            assert W.shape == g[p + "W"].shape and Wup.shape == g[p + "Wup"].shape
            # (bf16: the reference stores Q and R rounded to bf16, the oracle keeps them in fp64)
            assert rel_err(W @ Wup, g[p + "W"].astype(np.float64) @ g[p + "Wup"].astype(np.float64)) < (3e-2 if "bf16" in case else tol)
            assert rel_err(W, g[p + "W"]) < (3e-2 if "bf16" in case else 1e-4)


def test_reinit_normal_qr_matches_reference(golden_merge):
    g = golden_merge
    A_new, B_new = O.sow_reinit_from_gaussian(g["reinit/gauss"], g["reinit/A_new"].shape[1])
    assert rel_err(A_new, g["reinit/A_new"]) < 1e-5
    assert np.all(g["reinit/B_new"] == 0) and np.all(B_new == 0)
    # thin QR of the first r columns == Q[:, :r] of the full QR, including signs (SURVEY.md section 7)
    assert rel_err(O.thin_q(g["reinit/gauss"], A_new.shape[1]), g["reinit/A_new"]) < 1e-5


@pytest.mark.parametrize("case", ["tall", "wide", "square", "bf16"])
def test_qr_weight_matches_reference(golden_merge, case):
    g = golden_merge
    r = int(g[f"qr/{case}/rank"])
    Q, R = O.qr_weight(g[f"qr/{case}/w"], r)
    tol = 1e-2 if case == "bf16" else 2e-5
    assert rel_err(Q, g[f"qr/{case}/Q"]) < tol
    assert rel_err(R, g[f"qr/{case}/R"]) < tol


def test_tt_arange_known_answers(golden_tt):
    g = golden_tt
    A = g["tt/arange/tensor"]
    cores = O.tt_from_tensor(A, [1, 4, 4, 1])
    rec = O.tt_reconstruct(cores)
    assert rel_err(rec, A) < 1e-12                       # exact-rank case; reference fp32 prints 1.59e-07
    assert abs(float(g["tt/arange/rel_err"]) - 1.59e-07) < 0.05e-07   # BASELINE.md section 2
    assert rel_err(rec, g["tt/arange/reconstruct"]) < 1e-6
    for i, c in enumerate(cores):
        assert c.shape == g[f"tt/arange/core{i}"].shape
    s = O.tt_add(cores, cores)
    assert [c.shape[0] for c in s] + [1] == list(g["tt/arange/add_ranks"])
    assert rel_err(O.tt_reconstruct(s), g["tt/arange/add_rec"]) < 1e-6
    p = O.tt_mul(cores, cores)
    assert [c.shape[0] for c in p] + [1] == list(g["tt/arange/mul_ranks"])
    assert rel_err(O.tt_reconstruct(p), g["tt/arange/mul_rec"]) < 1e-6
    assert rel_err(O.tt_reconstruct(O.tt_round(p, [1, 4, 4, 1])), g["tt/arange/mul_round_rec"]) < 1e-5
    assert rel_err(O.tt_reconstruct(O.tt_scale(2.5, cores)), g["tt/arange/scaled_rec"]) < 1e-6
    assert abs(float(g["tt/arange/norm"]) - 3335941.0) <= 1.0


TT_MATRIX_CASES = ["m81_r4", "m81_r9", "m100x60", "m256_o3", "m300x200", "m256x192", "m130x70_pad"]


@pytest.mark.parametrize("case", TT_MATRIX_CASES)
def test_tt_from_matrix_matches_reference(golden_tt, case):
    g = golden_tt
    mat = tt_matrix(g, case)
    ranks = [int(r) for r in g[f"tt/{case}/ranks"]]
    cores = O.tt_from_matrix(mat, ranks)
    assert [list(c.shape) for c in cores] == g[f"tt/{case}/core_shapes"].tolist()
    back = O.tt_to_matrix(cores, mat.shape)
    # reconstruction is gauge invariant -> compare reconstructions and reconstruction ERRORS, never cores
    assert rel_err(back[::int(g["tt/to_matrix_row_step"])], g[f"tt/{case}/to_matrix_rows"]) < 5e-6
    err = rel_err(back, mat)
    assert abs(err - float(g[f"tt/{case}/rel_err"])) < 1e-5 * max(err, 1e-3)


def test_tt_lossy_probe_values(golden_tt):
    # BASELINE.md section 2: from_matrix(randn(81,81) seed 0): r=4 -> 0.98067, r=9 -> 0.89074
    assert abs(float(golden_tt["tt/m81_r4/rel_err"]) - 0.98067) < 1e-5
    assert abs(float(golden_tt["tt/m81_r9/rel_err"]) - 0.89074) < 1e-5


def test_tt_adam_update_script_known_answers(golden_tt):
    g = golden_tt
    grad = g["tt/kat_adam_update/grad"]
    cores = O.tt_from_matrix(grad, [1, 4, 4, 4, 1])
    back = O.tt_to_matrix(cores, grad.shape)
    # TT-rank <= 4 only up to the fp32 rounding of `grad`, and the first-4-columns basis is ill-conditioned:
    # the reference's fp32 run prints 8.60e-05 (BASELINE.md), exact arithmetic on the same input gives 6.2e-05.
    assert np.linalg.norm(back - grad) < 2e-4
    assert 8.0e-05 < float(g["tt/kat_adam_update/decomp_abs_err"]) < 9.2e-05
    assert rel_err(back, g["tt/kat_adam_update/reconstruct"]) < 1e-4
    # TT-SGD nesterov update (tests/tt_adam_update.py:28-51): buffer = 0.9*0 + grad ; upd = alpha*round(grad + .9*buf)
    zeros = [np.zeros_like(c) for c in cores]
    buf = O.tt_add(O.tt_scale(0.9, zeros), O.tt_scale(1.0, cores))
    upd = O.tt_scale(0.001, O.tt_round(O.tt_add(cores, O.tt_scale(0.9, buf))))
    upd_m = O.tt_to_matrix(upd, grad.shape)
    assert np.linalg.norm(upd_m - g["tt/kat_adam_update/update"]) < 5e-7
    assert 1.4e-07 < float(g["tt/kat_adam_update/l2"]) < 1.9e-07


@pytest.mark.parametrize("case", ["o2", "o3", "o2_pad"])
def test_ttadam_trajectory_matches_reference(golden_tt, case):
    g = golden_tt
    p = g[f"ttadam/{case}/p0"].astype(np.float64)
    ranks = [int(r) for r in g[f"ttadam/{case}/ranks"]]
    wd = float(g[f"ttadam/{case}/wd"])
    state = {}
    for step, grad in enumerate(g[f"ttadam/{case}/grads"]):
        p = O.ttadam_step(p, grad, state, lr=1e-2, weight_decay=wd, ranks=ranks)
        assert rel_err(p, g[f"ttadam/{case}/p{step + 1}"]) < 2e-5, step
    assert rel_err(O.tt_to_matrix(state["exp_avg"], p.shape), g[f"ttadam/{case}/m_final"]) < 1e-4
    assert rel_err(O.tt_to_matrix(state["exp_avg_sq"], p.shape), g[f"ttadam/{case}/v_final"]) < 1e-4


def test_ttadam_dense_branch(golden_tt):
    g = golden_tt
    p = g["ttadam/dense/p0"].astype(np.float64)
    state = {}
    for grad in g["ttadam/dense/grads"]:
        p = O.ttadam_step(p, grad, state, lr=1e-2)
    assert rel_err(p, g["ttadam/dense/p3"]) < 1e-6


def test_bf16_round_matches_torch():
    import torch
    x = np.random.default_rng(0).standard_normal(10000).astype(np.float32) * 37.0
    ref = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
    assert np.array_equal(O.bf16_round(x), ref)
