"""GPU: the SOWB_F16 mode of the group kernels and of the grouped merge, element by element against fp64, with the case
table, the guarded NaN slabs and the checkers of test_linear_edges_gpu / test_merge_edges_gpu.

fp16 runs the same component-wise bound as bf16 with u = u_out = 2^-11 (fp16 unit roundoff).  The inputs are drawn with
full 11-bit mantissas, so a bf16 rounding anywhere inside the path (2^-9 relative) breaks the bound.
"""
import os
import subprocess
import sys

import pytest
import torch

import test_linear_edges_gpu as LE
import test_merge_edges_gpu as ME
from conftest import ROOT
from sow_b200 import _lib, ops

pytestmark = pytest.mark.gpu

U16 = 2.0 ** -11     # fp16 unit roundoff
F16_CASES = [c for c in LE.CASES if not c.f32]


def make_inputs(case, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)

    def rn(*shape, s=1.0):
        return (torch.randn(*shape, generator=g, device="cuda") * s).to(torch.float16).contiguous()

    inp = {"x": rn(case.T, case.fin), "m": []}
    for m in case.members:
        d = {
            "W": rn(case.fin, m.out, s=case.fin ** -0.5) if m.W else None,
            "A": rn(case.fin, m.r, s=case.fin ** -0.5),
            "B": rn(m.r, m.out, s=0.1),
            "bias": rn(m.out, s=0.1) if m.bias else None,
            "dy": rn(case.T, m.out),
        }
        d["W_hi"], d["W_lo"], d["dy_hi"], d["dy_lo"] = d["W"], None, d["dy"], None
        inp["m"].append(d)
    torch.cuda.synchronize()
    return inp


def make_slab(case):
    R = LE.plan(case)["R"]
    h = torch.float16
    specs = [(f"y{i}", (case.T, m.out), h) for i, m in enumerate(case.members)]
    specs += [("A_cat", (case.fin, R), h), ("t_cat", (case.T, R), h), ("dt_cat", (case.T, R), h), ("dx", (case.T, case.fin), h)]
    for i, m in enumerate(case.members):
        specs += [(f"dA{i}", (case.fin, m.r), h), (f"dB{i}", (m.r, m.out), h)]
        if m.bias:
            specs.append((f"dbias{i}", (m.out,), h))
    specs.append(("ws", (LE.cdiv(LE.workspace_bytes(case), 2),), torch.int16))
    return LE.Slab(specs, "cuda")


def group_fwd(case, inp, slab):
    lib, arr = LE._member_array(case, inp, slab, True)
    rc = lib.sow_group_fwd(LE._p(inp["x"]), None, arr, len(case.members), LE._p(slab["A_cat"]), LE._p(slab["t_cat"]),
                           case.T, case.fin, _lib.SOWB_F16, LE._stream())
    _lib.check(rc, "sow_group_fwd")


def group_bwd(case, inp, slab):
    lib, arr = LE._member_array(case, inp, slab, False)
    ws = slab["ws"]
    rc = lib.sow_group_bwd(LE._p(inp["x"]), LE._p(slab["A_cat"]), LE._p(slab["t_cat"]), arr, len(case.members),
                           LE._p(slab["dt_cat"]), LE._p(slab["dx"]), case.T, case.fin, _lib.SOWB_F16, LE._p(ws),
                           ws.numel() * 2, LE._stream())
    _lib.check(rc, "sow_group_bwd")


def use_fp16(mod):
    """Points the checker of test_linear_edges_gpu (run_case / check_case / reference) at the SOWB_F16 mode: fp16 inputs,
    slab and calls, and u = u_out = 2^-11 in its bound.  Returns the previous attributes."""
    new = {"U": U16, "make_inputs": make_inputs, "make_slab": make_slab, "group_fwd": group_fwd, "group_bwd": group_bwd}
    old = {k: getattr(mod, k) for k in new}
    for k, v in new.items():
        setattr(mod, k, v)
    return old


@pytest.fixture
def fp16_checker():
    old = use_fp16(LE)
    yield LE
    for k, v in old.items():
        setattr(LE, k, v)


@pytest.mark.parametrize("case", F16_CASES, ids=repr)
def test_fp16_group_kernels_within_componentwise_bounds(case, fp16_checker):
    fp16_checker.check_case(case)


def test_fp16_big_tiles_within_componentwise_bounds():
    """SOWB_BIG_TILES is read once per process: the 256 x 256 tile GEMMs run in a child interpreter."""
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import test_linear_edges_gpu as t, test_fp16_edges_gpu as h\n"
            "h.use_fp16(t)\n"
            "for c in t.BIG_TILE_CASES: t.check_case(c)\n") % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ, SOWB_BIG_TILES="1")
    p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    print(p.stdout)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    assert p.stdout.count("EDGE big_tiles") == len(LE.BIG_TILE_CASES)


def test_fp16_checker_rejects_unwritten_and_stray_elements(fp16_checker):
    """In fp16 mode the checker still sees a NaN left in an output, a stray write into a guard band and a 2-ulp error."""
    case = F16_CASES[0]
    got, ref, problems = LE.run_case(case)
    assert not problems and max(LE.ratios(got, ref).values()) < 1.0
    y = got["y0"].clone()
    y.view(-1)[7] = float("nan")                             # an element the kernels did not write
    assert LE.ratios(dict(got, y0=y), ref)["y0"] == float("inf")
    y = got["y0"].clone()
    i = int(ref["y0"][0].abs().argmax())
    y.view(-1).view(torch.int16)[i] += 2                     # 2 fp16 ulps further from zero
    assert LE.ratios(dict(got, y0=y), ref)["y0"] > 1.0
    slab = make_slab(case)
    assert slab.guards_intact()
    slab.raw[0] = 0                                          # a write in front of the first view
    assert not slab.guards_intact()


@pytest.mark.parametrize("name", ["G8_out4096_in4096_r65", "K2_two_launches_out14336_r128_T4113", "qkv_uniform_R192"])
def test_fp16_two_runs_bit_identical(name, fp16_checker):
    case = next(c for c in F16_CASES if c.name == name)
    got1, _, p1 = LE.run_case(case)
    got2, _, p2 = LE.run_case(case)
    assert not p1 and not p2
    for k in got1:
        assert torch.equal(got1[k].view(torch.int16), got2[k].view(torch.int16)), k


def test_fp16_overflow_is_inf_in_exactly_that_position():
    """y[i, j] = 60000 * 2 + ... > 65504 becomes +inf (IEEE fp16, no saturation); every other element stays finite."""
    g = torch.Generator(device="cuda").manual_seed(3)
    T, fin, fout, r, i, j = 300, 264, 1000, 50, 131, 517
    h = torch.float16
    x = torch.randn(T, fin, generator=g, device="cuda").to(h)
    W = (torch.randn(fin, fout, generator=g, device="cuda") * fin ** -0.5).to(h)
    A = (torch.randn(fin, r, generator=g, device="cuda") * fin ** -0.5).to(h)
    B = (torch.randn(r, fout, generator=g, device="cuda") * 0.1).to(h)
    x[:, 0] = 0
    x[i, 0] = 60000.0
    W[0, :] = 0
    W[0, j] = 2.0
    A[0, :] = 0
    (y,), _, _ = ops.group_fwd(x, [(W, A, B, None, 1.0)])
    torch.cuda.synchronize()
    assert y.dtype == h
    bad = (~torch.isfinite(y)).nonzero().tolist()
    assert bad == [[i, j]], bad
    assert float(y[i, j]) == float("inf")


# ---------------------------------------------------------------------------------------------------------
# grouped merge
# ---------------------------------------------------------------------------------------------------------

def check_merge16(items, meta, slab):
    """ME.check with u = 2^-11, plus the absolute error of rounding into the fp16 subnormal range (half the subnormal
    spacing, 2^-25, per rounding): the product of a rank-1 term can be far below the smallest normal fp16 number."""
    ME.check(items, meta, slab, True)                   # asserts the guard bands and the separate W_prev unchanged
    out = []
    for (W, _, A, B, s), (init, _) in zip(items, meta):
        A64, B64 = A.to(torch.float64), B.to(torch.float64)
        ref = s * (A64 @ B64) + (0 if init is None else init.to(torch.float64))
        mag = abs(s) * (A64.abs() @ B64.abs()) + (0 if init is None else init.to(torch.float64).abs())
        nch = -(-A.shape[1] // 64)
        per = U16 + 2 * LE.U32
        bound = nch * per * (1 + per) ** nch * mag + LE.gamma(64) * (abs(s) * (A64.abs() @ B64.abs())) + nch * 2.0 ** -25
        got = W.to(torch.float64)
        q = torch.where(torch.isfinite(got), (got - ref).abs() / bound, torch.inf)
        out.append(float(q.max()))
    return out


def test_fp16_merge_mixed_list_elementwise():
    """Each element within ceil(r/64) fp16 roundings of |W_prev| + |s| |A| |B|; in place: W keeps its storage."""
    specs = [
        (200, 136, 1, "none", 0.5, False),
        (201, 1000, 7, "same", 1.0, False),
        (300, 2736, 50, "separate", 2.0, False),
        (136, 1000, 64, "same", -1.5, False),
        (264, 136, 65, "none", 1.0, False),
        (72, 2736, 128, "separate", 0.25, False),
        (330, 1000, 200, "same", 1.0, False),
        (200, 2736, 7, "separate", 1.0, True),
        (129, 136, 50, "same", 3.0, True),
        (1000, 1000, 64, "none", 1.0, False),
    ]
    slab, items, meta = ME.build(specs, torch.float16, 0)
    ptrs = [it[0].data_ptr() for it in items]
    ops.merge_grouped(items)
    torch.cuda.synchronize()
    assert [it[0].data_ptr() for it in items] == ptrs
    ME.report("merge_fp16_mixed", specs, check_merge16(items, meta, slab))


def test_fp16_merge_with_zero_B_keeps_every_bit():
    """B = 0: W_prev + s * A . 0 rounds back to W_prev exactly, including the 3 mantissa bits bf16 does not have."""
    g = torch.Generator(device="cuda").manual_seed(5)
    W = (torch.randn(300, 1000, generator=g, device="cuda") * 0.05).to(torch.float16)
    before = W.clone()
    A = (torch.randn(300, 50, generator=g, device="cuda") * 0.05).to(torch.float16)
    B = torch.zeros(50, 1000, dtype=torch.float16, device="cuda")
    assert not torch.equal(before.to(torch.bfloat16).to(torch.float16), before)   # the data has sub-bf16 bits
    ops.merge_grouped([(W, W, A, B, 1.0)])
    torch.cuda.synchronize()
    assert torch.equal(W.view(torch.int16), before.view(torch.int16))
