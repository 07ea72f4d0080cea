"""Generate golden fixtures by running the UNMODIFIED reference package (antoine311200/sow at /root/reference).

Run in the build container only (the reference does not exist on the GPU box):

    cd /root/repo/tests/golden && python make_golden.py

The reference imports four packages that are not installed here (peft, opt_einsum, termcolor, galore_torch); they
are shimmed below (SURVEY.md 8c).  Nothing from the reference is copied: only its *outputs* on seeded inputs are
stored, as small .npz files next to this script.
"""
import hashlib
import os
import sys
import types

import numpy as np
import torch

REF_ROOT = os.environ.get("SOW_REFERENCE_ROOT", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
TT_ROW_STEP = 4       # of each from_matrix / to_matrix reconstruction every 4th row is stored: keeps tt.npz under 1 MB


def install_shims():
    # --- peft: two empty base classes (prepare.py:13, sow.py:10)
    peft = types.ModuleType("peft")

    class PeftConfig:
        def __init__(self, **kwargs):
            for k, v in kwargs.items():
                setattr(self, k, v)

    class PeftModel(torch.nn.Module):
        pass

    peft.PeftConfig, peft.PeftModel = PeftConfig, PeftModel
    sys.modules["peft"] = peft

    # --- termcolor / galore_torch
    tc = types.ModuleType("termcolor")
    tc.colored = lambda s, *a, **k: s
    sys.modules["termcolor"] = tc
    gal = types.ModuleType("galore_torch")
    galp = types.ModuleType("galore_torch.galore_projector")
    galp.GaLoreProjector = object
    gal.galore_projector = galp
    sys.modules["galore_torch"] = gal
    sys.modules["galore_torch.galore_projector"] = galp

    # --- opt_einsum -> torch.einsum (interleaved operand/label-list form, string labels)
    oe = types.ModuleType("opt_einsum")
    oec = types.ModuleType("opt_einsum.contract")
    torch.backends.opt_einsum.enabled = False  # torch would otherwise pick up this fake module

    def _to_equation(struct):
        ops, label_lists = [], []
        i = 0
        out_labels = None
        while i < len(struct):
            if i + 1 < len(struct) and not isinstance(struct[i], (list, tuple)):
                ops.append(struct[i])
                label_lists.append(list(struct[i + 1]))
                i += 2
            else:
                out_labels = list(struct[i])
                i += 1
        names = {}
        letters = "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ"

        def sym(lbl):
            if lbl not in names:
                names[lbl] = letters[len(names)]
            return names[lbl]

        lhs = ",".join("".join(sym(l) for l in ll) for ll in label_lists)
        if out_labels is None:
            counts = {}
            for ll in label_lists:
                for l in ll:
                    counts[l] = counts.get(l, 0) + 1
            out_labels = sorted([l for l, c in counts.items() if c == 1], key=lambda l: names[l])
        rhs = "".join(sym(l) for l in out_labels)
        return lhs + "->" + rhs, ops

    def contract(*struct, **kw):
        eq, ops = _to_equation(struct)
        return torch.einsum(eq, *ops)

    class _PathInfo:
        def __init__(self, eq):
            self.eq = eq

    def contract_path(*struct, **kw):
        eq, _ = _to_equation(struct)
        return [], _PathInfo(eq)

    class ContractExpression:
        def __init__(self, eq):
            self.eq = eq

        def __call__(self, *ops):
            return torch.einsum(self.eq, *ops)

    def contract_expression(eq, *shapes, **kw):
        return ContractExpression(eq)

    oe.contract, oe.contract_path, oe.contract_expression = contract, contract_path, contract_expression
    oec.ContractExpression = ContractExpression
    oe.contract_module = oec
    sys.modules["opt_einsum"] = oe
    sys.modules["opt_einsum.contract"] = oec


def import_reference():
    repo_root = os.path.abspath(os.path.join(HERE, "..", ".."))
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or os.getcwd()) != repo_root]
    sys.path.insert(0, REF_ROOT)
    install_shims()
    import tn_gradient.layer.sow as ref_sow
    import tn_gradient.prepare as ref_prepare
    import tn_gradient.tt as ref_tt
    import tn_gradient.utils as ref_utils
    import tn_gradient.optimizer.ttadam as ref_ttadam
    import tn_gradient.optimizer.ttsgd as ref_ttsgd
    assert os.path.abspath(ref_sow.__file__).startswith(os.path.abspath(REF_ROOT)), ref_sow.__file__
    return ref_sow, ref_prepare, ref_tt, ref_utils, ref_ttadam, ref_ttsgd


def npy(t):
    return t.detach().to(torch.float32).cpu().numpy().copy()


def make_linear_cases(ref_sow, out):
    """SoWLinear fwd/bwd (sow.py:107-126 + autograd) in fp32 and bf16, with/without W, bias, 3-D input."""
    cases = [
        # name, lead shape, in, out, r, n_iter, scale, has_W, bias, dtype
        ("f32_w_bias", (2, 12), 40, 56, 6, 1, 0.125, True, True, torch.float32),
        ("f32_now", (3, 8), 40, 56, 6, 1, 1.0, False, False, torch.float32),
        ("f32_niter2", (24,), 32, 48, 4, 2, 0.5, True, False, torch.float32),
        ("bf16_w", (4, 32), 128, 192, 50, 1, 1.0, True, False, torch.bfloat16),
        ("bf16_now_bias", (4, 32), 128, 192, 8, 1, 0.125, False, True, torch.bfloat16),
    ]
    for name, lead, fin, fout, r, n_iter, scale, has_W, bias, dtype in cases:
        torch.manual_seed(1234)
        layer = ref_sow.SoWLinear(fin, fout, bias=bias, rank=r, n_iter=n_iter, scale=scale, init_method="normal",
                                  dtype=torch.float32)
        with torch.no_grad():
            for B in layer.upscale_weights:
                B.normal_(0, 0.05)
            for A in layer.downscale_weights:
                A.normal_(0, 0.05)
            if bias:
                layer.bias.normal_(0, 0.5)
            if has_W:
                layer.acc_downweight = torch.nn.Parameter(torch.randn(fin, fout) * 0.02, requires_grad=False)
        layer = layer.to(dtype)
        x = torch.randn(*lead, fin).to(dtype).requires_grad_(True)
        dy = torch.randn(*lead, fout).to(dtype)
        y = layer(x)
        y.backward(dy)
        d = {"x": npy(x), "dy": npy(dy), "y": npy(y), "dx": npy(x.grad), "scale": np.float32(scale),
             "n_iter": np.int32(n_iter)}
        if has_W:
            d["W"] = npy(layer.acc_downweight)
        if bias:
            d["bias"] = npy(layer.bias)
            d["dbias"] = npy(layer.bias.grad)
        for i in range(n_iter):
            d[f"A{i}"] = npy(layer.downscale_weights[i])
            d[f"B{i}"] = npy(layer.upscale_weights[i])
            d[f"dA{i}"] = npy(layer.downscale_weights[i].grad)
            d[f"dB{i}"] = npy(layer.upscale_weights[i].grad)
        for k, v in d.items():
            out[f"linear/{name}/{k}"] = v


def make_merge_cases(ref_sow, out):
    """SoWLinear.accumulate (sow.py:128-178): dense branch from empty and from dense W, factored (QR-growth)
    branch over two merges, in fp32 and bf16; re-init with init_method 'normal' and 'normal_QR'."""
    for name, fin, fout, r, n_iter, scale, dtype, dense in [
        ("dense_f32", 48, 80, 6, 1, 0.5, torch.float32, True),
        ("dense_bf16", 128, 192, 50, 1, 1.0, torch.bfloat16, True),
        ("dense_niter2_f32", 32, 40, 4, 2, 0.25, torch.float32, True),
        ("factored_f32", 64, 48, 10, 2, 1.0, torch.float32, False),
        ("factored_bf16", 64, 48, 10, 2, 1.0, torch.bfloat16, False),   # crosses the full-rank boundary in bf16
    ]:
        torch.manual_seed(77)
        layer = ref_sow.SoWLinear(fin, fout, bias=False, rank=r, n_iter=n_iter, scale=scale, init_method="normal",
                                  dtype=torch.float32)
        if dense:
            layer.virtual_rank = min(fin, fout)  # what prepare_sow does (prepare.py:120)
        with torch.no_grad():
            for A in layer.downscale_weights:
                A.normal_(0, 0.05)
            for B in layer.upscale_weights:
                B.normal_(0, 0.05)
        layer = layer.to(dtype)
        for step in range(3):
            pre = f"merge/{name}/step{step}"
            for i in range(n_iter):
                out[f"{pre}/A{i}"] = npy(layer.downscale_weights[i])
                out[f"{pre}/B{i}"] = npy(layer.upscale_weights[i])
            out[f"{pre}/W_prev"] = npy(layer.acc_downweight)
            out[f"{pre}/Wup_prev"] = npy(layer.acc_upweight)
            out[f"{pre}/virtual_rank_prev"] = np.int32(layer.virtual_rank)
            layer.accumulate()
            out[f"{pre}/W"] = npy(layer.acc_downweight)
            out[f"{pre}/Wup"] = npy(layer.acc_upweight)
            out[f"{pre}/virtual_rank"] = np.int32(layer.virtual_rank)
            # accumulate() re-initialised A (normal) and zeroed B: give B fresh values for the next round
            with torch.no_grad():
                for B in layer.upscale_weights:
                    assert float(B.abs().max()) == 0.0
                    B.copy_((torch.randn(B.shape) * 0.05).to(dtype))
        out[f"merge/{name}/meta"] = np.array([fin, fout, r, n_iter], dtype=np.int32)
        out[f"merge/{name}/scale"] = np.float32(scale)

    # normal_QR re-init (sow.py:162-172): A_new = Q[:, :r] of QR(N(0, .02) in x out)
    torch.manual_seed(5)
    fin, fout, r = 96, 160, 12
    layer = ref_sow.SoWLinear(fin, fout, bias=False, rank=r, n_iter=1, scale=1.0, init_method="normal",
                              dtype=torch.float32)
    layer.virtual_rank = min(fin, fout)
    layer.init_method = "normal_QR"  # ctor's normal_QR path hard-codes .to("cuda") (sow.py:91); accumulate()'s does not
    torch.manual_seed(99)
    layer.accumulate()
    torch.manual_seed(99)
    gauss = torch.zeros(fin, fout).normal_(mean=0.0, std=0.02)
    out["reinit/gauss"] = npy(gauss)
    out["reinit/A_new"] = npy(layer.downscale_weights[0])
    out["reinit/B_new"] = npy(layer.upscale_weights[0])


def make_qr_cases(ref_utils, out):
    torch.manual_seed(3)
    for name, m, n, r in [("tall", 200, 40, 16), ("wide", 64, 300, 20), ("square", 96, 96, 50)]:
        w = torch.randn(m, n)
        Q, R = ref_utils.qr_weight(w, r)
        out[f"qr/{name}/w"] = npy(w)
        out[f"qr/{name}/Q"] = npy(Q)
        out[f"qr/{name}/R"] = npy(R)
        out[f"qr/{name}/rank"] = np.int32(r)
    wb = torch.randn(128, 64).to(torch.bfloat16)
    Q, R = ref_utils.qr_weight(wb, 8)
    out["qr/bf16/w"], out["qr/bf16/Q"], out["qr/bf16/R"], out["qr/bf16/rank"] = npy(wb), npy(Q), npy(R), np.int32(8)


def store_tt_matrix_case(out, name, mat, ranks, back, rel_err, core_shapes):
    """One from_matrix / to_matrix case.  The input (torch.manual_seed(0); torch.randn(M, N)) is stored as its shape and
    SHA-256: the tests draw it again and check it bit for bit.  The reconstruction is stored as every TT_ROW_STEP-th
    row; ``rel_err`` is the reference's error over the full matrices."""
    out[f"tt/{name}/shape"] = np.array(mat.shape, dtype=np.int32)
    out[f"tt/{name}/matrix_sha256"] = np.array(hashlib.sha256(np.ascontiguousarray(mat).tobytes()).hexdigest())
    out[f"tt/{name}/ranks"] = np.array(ranks, dtype=np.int32)
    out[f"tt/{name}/to_matrix_rows"] = np.ascontiguousarray(back[::TT_ROW_STEP])
    out[f"tt/{name}/rel_err"] = np.float64(rel_err)
    out[f"tt/{name}/core_shapes"] = np.array(core_shapes, dtype=np.int32)


def make_tt_cases(ref_tt, ref_utils, ref_ttadam, ref_ttsgd, out):
    TT = ref_tt.TensorTrain
    # --- tests/tt_test.py KAT: arange tensor, ranks [1,4,4,1]
    A = torch.arange(2 * 2 * 2 * 3 * 3 * 3).reshape((2, 2, 2, 3, 3, 3)).float()
    ttA = TT.from_tensor(A, [1, 4, 4, 1])
    rec = ttA.reconstruct()
    out["tt/arange/tensor"] = npy(A)
    out["tt/arange/reconstruct"] = npy(rec)
    out["tt/arange/rel_err"] = np.float64((rec - A).norm() / A.norm())
    for i, c in enumerate(ttA.cores):
        out[f"tt/arange/core{i}"] = npy(c)
    s = ttA + ttA
    out["tt/arange/add_ranks"] = np.array(s.ranks, dtype=np.int32)
    out["tt/arange/add_rec"] = npy(s.reconstruct())
    p = ttA * ttA
    out["tt/arange/mul_ranks"] = np.array(p.ranks, dtype=np.int32)
    out["tt/arange/mul_rec"] = npy(p.reconstruct())
    rr = (ttA * ttA).round([1, 4, 4, 1])
    out["tt/arange/mul_round_rec"] = npy(rr.reconstruct())
    out["tt/arange/scaled_rec"] = npy((2.5 * ttA).reconstruct())
    out["tt/arange/addc_rec"] = npy(ttA.add_(-3).reconstruct())
    out["tt/arange/norm"] = np.float64(ttA.norm())

    # --- from_matrix / to_matrix, lossy and exact
    torch.manual_seed(0)
    cases = [("m81_r4", 81, 81, [1, 4, 4, 4, 1]), ("m81_r9", 81, 81, [1, 9, 9, 9, 1]), ("m100x60", 100, 60, [1, 16, 1]),
             ("m256_o3", 256, 256, [1, 8, 8, 1]), ("m300x200", 300, 200, [1, 12, 12, 1]),
             ("m256x192", 256, 192, [1, 32, 1]), ("m130x70_pad", 130, 70, [1, 10, 1])]
    out["tt/to_matrix_row_step"] = np.int32(TT_ROW_STEP)
    for name, M, N, ranks in cases:
        torch.manual_seed(0)
        mat = torch.randn(M, N)
        tt = TT.from_matrix(mat, list(ranks))
        back = tt.to_matrix((M, N))
        store_tt_matrix_case(out, name, npy(mat), ranks, npy(back), (back - mat).norm() / mat.norm(),
                             [list(c.shape) for c in tt.cores])

    # --- tests/tt_adam_update.py KATs (seed 0; "cuda" -> "cpu")
    from opt_einsum import contract
    torch.manual_seed(0)

    def generate_rank_k_tensor(shape, k, sumof=1):
        tensor = torch.zeros(shape)
        for _ in range(sumof):
            factors = [2 * torch.rand(dim, k) - 1 for dim in shape]
            struct = []
            for i, factor in enumerate(factors):
                struct.append(factor)
                struct.append([f"l_{i}", "k"])
            tensor += contract(*struct)
        return tensor

    M = N = 81
    order, rank = 4, 4
    ranks = [1] + [rank] * (order - 1) + [1]
    input_shape = ref_utils.closest_factorization(M, order)[0]
    output_shape = ref_utils.closest_factorization(N, order)[0]
    rank_grad = generate_rank_k_tensor(input_shape + output_shape, 2, sumof=2)
    grad = rank_grad.reshape(M, N).float()
    mm = nn = 3
    padded = ref_utils.pad_matrix(grad, (mm ** order, nn ** order))
    tt_grad = TT.from_tensor(padded.reshape((mm,) * order + (nn,) * order), ranks=list(ranks))
    tt2t = ref_utils.unpad_matrix(tt_grad.reconstruct().reshape(81, 81), (M, N))
    out["tt/kat_adam_update/grad"] = npy(grad)
    out["tt/kat_adam_update/decomp_abs_err"] = np.float64(torch.linalg.norm(tt2t - grad))
    out["tt/kat_adam_update/reconstruct"] = npy(tt2t)
    # TT-SGD nesterov update vs dense (tests/tt_adam_update.py:28-51,182-216)
    momentum, alpha, dampening = 0.9, 0.001, 0.0
    tt_m = TT.zeros(list(ranks), (mm,) * order, (nn,) * order)
    buf = momentum * tt_m + (1 - dampening) * tt_grad
    upd = (tt_grad + momentum * buf).round()
    upd = alpha * upd
    tt_update = ref_utils.unpad_matrix(upd.reconstruct().reshape(81, 81), (M, N))
    m_dense = torch.zeros(M, N)
    buf_d = momentum * m_dense + (1 - dampening) * grad
    update = alpha * (grad + momentum * buf_d)
    out["tt/kat_adam_update/tt_update"] = npy(tt_update)
    out["tt/kat_adam_update/update"] = npy(update)
    out["tt/kat_adam_update/l2"] = np.float64(torch.linalg.norm(tt_update - update))

    # --- TTAdam trajectories (ttadam.py:32-117)
    for name, M, N, ranks, wd in [("o2", 64, 48, [1, 8, 1], 0.0), ("o3", 64, 27, [1, 4, 4, 1], 0.01),
                                  ("o2_pad", 50, 30, [1, 6, 1], 0.0)]:
        torch.manual_seed(11)
        p = torch.nn.Parameter(torch.randn(M, N) * 0.1)
        opt = ref_ttadam.TTAdam([{"params": [p], "ranks": list(ranks)}], lr=1e-2, weight_decay=wd)
        out[f"ttadam/{name}/p0"] = npy(p)
        out[f"ttadam/{name}/ranks"] = np.array(ranks, dtype=np.int32)
        out[f"ttadam/{name}/wd"] = np.float32(wd)
        grads = []
        for step in range(5):
            g = torch.randn(M, N) * (1.0 + 0.3 * step)
            grads.append(npy(g))
            p.grad = g.clone()
            opt.step()
            out[f"ttadam/{name}/p{step + 1}"] = npy(p)
        out[f"ttadam/{name}/grads"] = np.stack(grads)
        st = opt.state[p]
        out[f"ttadam/{name}/m_final"] = npy(st["exp_avg"].to_matrix((M, N)))
        out[f"ttadam/{name}/v_final"] = npy(st["exp_avg_sq"].to_matrix((M, N)))
    # dense (no "ranks") branch
    torch.manual_seed(12)
    p = torch.nn.Parameter(torch.randn(20, 12) * 0.1)
    opt = ref_ttadam.TTAdam([p], lr=1e-2)
    out["ttadam/dense/p0"] = npy(p)
    grads = []
    for step in range(3):
        g = torch.randn(20, 12)
        grads.append(npy(g))
        p.grad = g.clone()
        opt.step()
    out["ttadam/dense/grads"] = np.stack(grads)
    out["ttadam/dense/p3"] = npy(p)

    # --- TTSGD (ttsgd.py:28-86), nesterov + momentum, TT-compressed gradient
    torch.manual_seed(13)
    p = torch.nn.Parameter(torch.randn(36, 25) * 0.1)
    opt = ref_ttsgd.TTSGD([{"params": [p], "ranks": [1, 12, 1]}], lr=1e-2, momentum=0.9, nesterov=True)
    out["ttsgd/p0"] = npy(p)
    grads = []
    for step in range(3):
        g = torch.randn(36, 25)
        grads.append(npy(g))
        p.grad = g.clone()
        opt.step()
    out["ttsgd/grads"] = np.stack(grads)
    out["ttsgd/p3"] = npy(p)


def make_loop_case(ref_sow, ref_prepare, out):
    """Replay of the training-loop contract (scripts/simple_train.py:611-650) on a tiny 2-layer MLP through
    prepare_sow: backward -> [accumulate + reset_optimizer at the merge step] -> optimizer.step."""
    import torch.nn as nn

    class MLP(nn.Module):
        def __init__(self):
            super().__init__()
            self.fc1 = nn.Linear(24, 40, bias=True)
            self.fc2 = nn.Linear(40, 16, bias=False)

        def forward(self, x):
            return self.fc2(torch.tanh(self.fc1(x)))

    def reset_optimizer(optimizer, group_id):  # scripts/utils/training_utils.py:257-277 (behaviour)
        group = optimizer.param_groups[group_id]
        for param in group["params"]:
            state = optimizer.state[param]
            state["exp_avg"] = torch.zeros_like(param)
            state["exp_avg_sq"] = torch.zeros_like(param)
            if "step" in state:
                state["step"] = torch.zeros_like(state["step"])

    for mode in ["keep", None]:
        torch.manual_seed(21)
        model = MLP()
        w1, w2 = npy(model.fc1.weight), npy(model.fc2.weight)
        b1 = npy(model.fc1.bias)
        cfg = ref_prepare.SoWConfig(target_modules=["fc1", "fc2"], rank=4, scale=0.5, device="cpu",
                                    init_method="normal", decompose=mode)
        model = ref_prepare.prepare_sow(model, cfg)
        tag = f"loop/{mode}"
        out[f"{tag}/fc1_weight"], out[f"{tag}/fc2_weight"], out[f"{tag}/fc1_bias"] = w1, w2, b1
        factors = []
        for mod in [model.fc1, model.fc2]:
            factors += list(mod.downscale_weights) + list(mod.upscale_weights)
        for i, f in enumerate(factors):
            out[f"{tag}/factor{i}_init"] = npy(f)
        others = [p for p in model.parameters() if p.requires_grad and all(p is not f for f in factors)]
        opt = torch.optim.AdamW([{"params": others, "lr": 1e-2, "weight_decay": 0.0},
                                 {"params": factors, "lr": 1e-2, "weight_decay": 0.0}])
        g = torch.Generator().manual_seed(5)
        losses, xs, ys = [], [], []
        reinit_A = []
        for step in range(1, 7):
            x = torch.randn(32, 24, generator=g)
            y = torch.randn(32, 16, generator=g)
            xs.append(npy(x))
            ys.append(npy(y))
            loss = ((model(x) - y) ** 2).mean()
            loss.backward()
            if step == 3:
                ref_prepare.accumulate(model)
                reset_optimizer(opt, 1)
                reinit_A.append([npy(model.fc1.downscale_weights[0]), npy(model.fc2.downscale_weights[0])])
            opt.step()
            opt.zero_grad()
            losses.append(float(loss))
        out[f"{tag}/x"] = np.stack(xs)
        out[f"{tag}/y"] = np.stack(ys)
        out[f"{tag}/losses"] = np.array(losses, dtype=np.float64)
        out[f"{tag}/reinit_A_fc1"] = reinit_A[0][0]
        out[f"{tag}/reinit_A_fc2"] = reinit_A[0][1]
        out[f"{tag}/final_W_fc1"] = npy(model.fc1.acc_downweight)
        out[f"{tag}/final_W_fc2"] = npy(model.fc2.acc_downweight)
        for i, f in enumerate(factors):
            out[f"{tag}/factor{i}_final"] = npy(f)
        out[f"{tag}/state_dict_keys"] = np.array(sorted(model.state_dict().keys()))


def main():
    ref_sow, ref_prepare, ref_tt, ref_utils, ref_ttadam, ref_ttsgd = import_reference()
    torch.set_num_threads(1)  # deterministic reductions
    groups = {
        "linear": lambda o: make_linear_cases(ref_sow, o),
        "merge": lambda o: (make_merge_cases(ref_sow, o), make_qr_cases(ref_utils, o)),
        "tt": lambda o: make_tt_cases(ref_tt, ref_utils, ref_ttadam, ref_ttsgd, o),
        "loop": lambda o: make_loop_case(ref_sow, ref_prepare, o),
    }
    for name, fn in groups.items():
        out = {}
        fn(out)
        path = os.path.join(HERE, f"{name}.npz")
        np.savez_compressed(path, **out)
        print(f"wrote {path}: {len(out)} arrays, {os.path.getsize(path) / 1024:.1f} KiB")


if __name__ == "__main__":
    main()
