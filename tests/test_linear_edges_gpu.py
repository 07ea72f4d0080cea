"""GPU: the SoW group kernels (sow_group_fwd / sow_group_bwd) element by element against an fp64 restatement of the same
operation, on every dispatch branch of linear.cu / k2.cuh, with every output in caller-owned buffers surrounded by guard
bands.

Each output element must satisfy a component-wise bound

    |got - ref| <= C * (u_out * |ref| + u * P_round) + gamma_K * P_acc  (+ SPLIT * P_split in fp32 mode)

with u = 2^-8 (bf16 unit roundoff), u_out the unit roundoff of the output type, gamma_K = K * 2^-24 for a K-term fp32
accumulation, P_round the absolute product through which a bf16 rounding inside the kernel propagates and P_acc the
absolute product of the fp32 accumulation.  Every output is a contiguous view into a slab that is filled with a NaN bit
pattern before the call: an element the kernels never write stays NaN, a write outside the views changes a guard element.
"""
import ctypes
import json
import math
import os
import re
import subprocess
import sys

import pytest
import torch

from conftest import ROOT

from sow_b200 import _lib, ops
from sow_b200._lib import SowB200Error

pytestmark = pytest.mark.gpu

CSRC = os.path.join(ROOT, "sow_b200", "csrc")


def _const(fname, name):
    with open(os.path.join(CSRC, fname)) as f:
        m = re.search(r"constexpr int %s = (\d+);" % name, f.read())
    assert m, (fname, name)
    return int(m.group(1))


# dispatch constants, read from the kernel sources so that the case table follows them
K2_MAX_G = _const("k2.cuh", "kK2MaxG")
K2_MAX_BPG = _const("k2.cuh", "kK2MaxBpg")
MAX_GROUP = _const("linear.cu", "kMaxGroup")
MAX_SEG = _const("gemm.cuh", "kMaxSeg")
MAX_ALPHA = _const("gemm.cuh", "kMaxAlphaBlocks")
BM = _const("gemm.cuh", "kBM")
BK = _const("gemm.cuh", "kBK")

U = 2.0 ** -8        # bf16 unit roundoff
U32 = 2.0 ** -24     # fp32 unit roundoff
# Roundings per output: one of the output itself and at most two on the P_round path (fp32 mode: the bf16 high piece of x
# or dY that the rank-r products read, plus the bf16 t / dt the kernels store).
C = 3.0
# bf16x3 products of fp32 operands: hi = bf16(v), lo = bf16(v - hi) leave |v - hi - lo| <= 2^-16 |v| for each operand,
# and the dropped lo * lo term is <= 2^-16 |x| |W|: 3 * 2^-16 per term of |x| . |W|.
SPLIT = 3 * 2.0 ** -16
SENTINEL = 0x7FA5    # bf16 NaN with a payload (and, as a pair, an fp32 NaN) that no kernel produces


def cdiv(a, b):
    return -(-a // b)


def gamma(K):
    return K * U32


# ---------------------------------------------------------------------------------------------------------
# case table
# ---------------------------------------------------------------------------------------------------------

class M:
    """One member: out features, rank, dense W or not, bias or not, scale."""

    def __init__(self, out, r, W=True, bias=True, scale=1.0):
        self.out, self.r, self.W, self.bias, self.scale = out, r, W, bias, scale


class Case:
    def __init__(self, name, T, fin, members, expect, f32=False, repro=False):
        self.name, self.T, self.fin, self.members, self.expect, self.f32, self.repro = \
            name, T, fin, members, expect, f32, repro

    def __repr__(self):
        return self.name


def k2_plan(out):
    """(G, n_launch, blocks per launch) of k2_plan (linear.cu)."""
    nblk = cdiv(out, 128)
    n_launch = cdiv(nblk, K2_MAX_G * K2_MAX_BPG)
    bpl = cdiv(nblk, n_launch)
    G = 1
    while G * K2_MAX_BPG < bpl:
        G *= 2
    return G, n_launch, bpl


def plan(case):
    """Which branches of sow_group_fwd / sow_group_bwd a case takes, derived from the dispatch code."""
    rpad = [ops.rank_pad(m.r) for m in case.members]
    R = sum(rpad)
    k2 = [k2_plan(m.out) for m in case.members]
    batched = len({(g, nl, rp) for (g, nl, _), rp in zip(k2, rpad)}) == 1
    nW = sum(m.W for m in case.members)
    return {
        "G": tuple(p[0] for p in k2),
        "launches": tuple(p[1] for p in k2),
        "batched": batched,
        "R": R,
        "bn": 256 if R >= 256 else R,
        "dx_segs": nW * (3 if case.f32 else 1) + 1,
        "chunks": tuple(rp // 64 for rp in rpad),
        "alpha_blocks": R // 64,
    }


CASES = [
    Case("G1_out136_r8", 300, 264, [M(136, 8, scale=0.5)], {"G": (1,), "bn": 64}),
    Case("G2_out1000_T1_in72", 1, 72, [M(1000, 50, bias=False)], {"G": (2,)}),
    Case("G4_out2736_T127", 127, 264, [M(2736, 64, scale=2.0)], {"G": (4,), "chunks": (1,)}),
    Case("G8_out4096_in4096_r65", 128, 4096, [M(4096, 65, bias=False)], {"G": (8,), "chunks": (2,), "bn": 128},
         repro=True),
    Case("G16_out11008_r127", 129, 72, [M(11008, 127, scale=0.5)], {"G": (16,), "launches": (1,)}, repro=True),
    Case("K2_two_launches_out12296_r1", 300, 264, [M(12296, 1, bias=False)], {"G": (16,), "launches": (2,)}, repro=True),
    Case("K2_two_launches_out14336_r128_T4113", 4113, 264, [M(14336, 128, scale=0.25)], {"G": (16,), "launches": (2,)},
         repro=True),
    Case("out1016_r200_in8", 300, 8, [M(1016, 200, bias=False)], {"chunks": (4,), "bn": 256}),
    Case("out1088_long_T16384", 16384, 72, [M(1088, 50)], {"G": (2,)}),
    Case("qkv_uniform_R192", 300, 264, [M(1000, 50), M(1000, 50, scale=0.5), M(1000, 50, scale=2.0)],
         {"batched": True, "bn": 192, "dx_segs": 4}),
    Case("gqa_q4096_kv1024", 129, 4096, [M(4096, 64, bias=False), M(1024, 64, bias=False), M(1024, 64, bias=False)],
         {"G": (8, 2, 2), "batched": False}),
    Case("ranks_8_100", 127, 264, [M(1000, 8), M(1000, 100)], {"batched": False, "R": 192}),
    Case("four_members_mixed_W_bias", 300, 264,
         [M(136, 1, W=True, bias=True, scale=0.5), M(1000, 64, W=False, bias=True),
          M(2736, 65, W=True, bias=False, scale=2.0), M(1016, 128, W=False, bias=False, scale=1.5)],
         {"R": 384, "bn": 256, "dx_segs": 3, "batched": False}),
    Case("scales_ranks_above_64", 129, 72, [M(1000, 100, bias=False, scale=0.25), M(1000, 200, scale=2.0)],
         {"R": 384, "alpha_blocks": 6}),
    Case("R1024_four_members", 128, 264,
         [M(136, 256, scale=0.5), M(1000, 256), M(1016, 256, bias=False, scale=1.5), M(264, 256, scale=2.0)],
         {"R": 64 * MAX_ALPHA, "bn": 256}),
    Case("fp32_three_members_10_segments", 129, 264,
         [M(1000, 8), M(136, 50, scale=0.5), M(2736, 65, bias=False, scale=2.0)], {"dx_segs": MAX_SEG}, f32=True),
]

# run with SOWB_BIG_TILES=1 (256 x 256 CTA tiles in the forward and dX GEMMs): ragged T, in and out
BIG_TILE_CASES = [
    Case("big_tiles_qkv_T385", 385, 264, [M(1000, 50), M(136, 8, scale=0.5), M(1016, 64, bias=False)],
         {"dx_segs": 4}),
    Case("big_tiles_single_T129", 129, 72, [M(2736, 65, scale=2.0)], {"G": (4,)}),
]


# ---------------------------------------------------------------------------------------------------------
# caller-owned output slab with guard bands
# ---------------------------------------------------------------------------------------------------------

class Slab:
    """Contiguous views into one int16 buffer, each with guard elements before and after it.  The whole buffer starts as
    the SENTINEL pattern; ``guards_intact`` checks that nothing outside the views changed."""

    def __init__(self, specs, device):
        off = 0
        layout = []
        for name, shape, dt in specs:
            itemsize = torch.empty((), dtype=dt).element_size()
            n16 = math.prod(shape) * itemsize // 2
            # room for a stray 128-row tile of this view's width, at least 32 KB
            guard = max(16384, min(128 * shape[-1] * itemsize // 2, 4 << 20))
            off = (off + guard + 127) // 128 * 128
            layout.append((name, shape, dt, off, n16, guard))
            off += n16
        off += layout[-1][5] if layout else 16384
        self.raw = torch.full((off,), SENTINEL, dtype=torch.int16, device=device)
        self.views = {}
        self.spans = []
        for name, shape, dt, o, n, _ in layout:
            self.views[name] = self.raw[o:o + n].view(dt).view(shape)
            self.spans.append((o, n))

    def __getitem__(self, name):
        return self.views[name]

    def refill(self, names):
        for n in names:
            self.views[n].view(torch.int16).fill_(SENTINEL)

    def guards_intact(self):
        keep = torch.ones(self.raw.numel(), dtype=torch.bool, device=self.raw.device)
        for o, n in self.spans:
            keep[o:o + n] = False
        return bool((self.raw[keep] == SENTINEL).all())

    def untouched(self):
        return bool((self.raw == SENTINEL).all())


# ---------------------------------------------------------------------------------------------------------
# inputs, ctypes calls
# ---------------------------------------------------------------------------------------------------------

def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def make_inputs(case, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    dev = "cuda"
    wdt = torch.float32 if case.f32 else torch.bfloat16

    def rn(*shape, s=1.0, dt=torch.bfloat16):
        return (torch.randn(*shape, generator=g, device=dev) * s).to(dt).contiguous()

    inp = {"x": rn(case.T, case.fin, dt=wdt), "m": []}
    if case.f32:
        inp["x_hi"], inp["x_lo"] = ops.split_f32(inp["x"])
    for m in case.members:
        d = {
            "W": rn(case.fin, m.out, s=case.fin ** -0.5, dt=wdt) if m.W else None,
            "A": rn(case.fin, m.r, s=case.fin ** -0.5),
            "B": rn(m.r, m.out, s=0.1),
            "bias": rn(m.out, s=0.1, dt=wdt) if m.bias else None,
            "dy": rn(case.T, m.out, dt=wdt),
        }
        if case.f32:
            d["W_hi"], d["W_lo"] = ops.split_f32(d["W"]) if m.W else (None, None)
            d["dy_hi"], d["dy_lo"] = ops.split_f32(d["dy"])
        else:
            d["W_hi"], d["W_lo"], d["dy_hi"], d["dy_lo"] = d["W"], None, d["dy"], None
        inp["m"].append(d)
    torch.cuda.synchronize()
    return inp


def _member_array(case, inp, slab, fwd):
    lib = _lib.load()
    arr = (_lib.GroupMember * len(case.members))()
    for i, (m, d) in enumerate(zip(case.members, inp["m"])):
        a = arr[i]
        a.W, a.W_lo, a.B = _p(d["W_hi"]), _p(d["W_lo"]), _p(d["B"])
        a.out_features, a.r, a.scale = m.out, m.r, float(m.scale)
        if fwd:
            a.A, a.bias, a.y = _p(d["A"]), _p(d["bias"]), _p(slab[f"y{i}"])
        else:
            a.A = _p(slab["A_cat"])
            a.dy, a.dy_lo = _p(d["dy_hi"]), _p(d["dy_lo"] if m.W else None)
            a.dA, a.dB = _p(slab[f"dA{i}"]), _p(slab[f"dB{i}"])
            a.dbias = _p(slab[f"dbias{i}"]) if m.bias else None
    return lib, arr


def workspace_bytes(case):
    lib = _lib.load()
    arr = (_lib.GroupMember * len(case.members))()
    for i, m in enumerate(case.members):
        arr[i].out_features, arr[i].r = m.out, m.r
    return lib.sow_group_workspace_bytes(_lib.OP_LINEAR_BWD, case.T, case.fin, arr, len(case.members))


def make_slab(case):
    R = plan(case)["R"]
    odt = torch.float32 if case.f32 else torch.bfloat16
    specs = [(f"y{i}", (case.T, m.out), odt) for i, m in enumerate(case.members)]
    specs += [("A_cat", (case.fin, R), torch.bfloat16), ("t_cat", (case.T, R), torch.bfloat16),
              ("dt_cat", (case.T, R), torch.bfloat16), ("dx", (case.T, case.fin), odt)]
    for i, m in enumerate(case.members):
        specs += [(f"dA{i}", (case.fin, m.r), torch.bfloat16), (f"dB{i}", (m.r, m.out), torch.bfloat16)]
        if m.bias:
            specs.append((f"dbias{i}", (m.out,), torch.bfloat16))
    specs.append(("ws", (cdiv(workspace_bytes(case), 2),), torch.int16))
    return Slab(specs, "cuda")


def group_fwd(case, inp, slab):
    lib, arr = _member_array(case, inp, slab, True)
    x = inp["x_hi"] if case.f32 else inp["x"]
    rc = lib.sow_group_fwd(_p(x), _p(inp.get("x_lo")), arr, len(case.members), _p(slab["A_cat"]), _p(slab["t_cat"]),
                           case.T, case.fin, _lib.SOWB_F32 if case.f32 else _lib.SOWB_BF16, _stream())
    _lib.check(rc, "sow_group_fwd")


def group_bwd(case, inp, slab):
    lib, arr = _member_array(case, inp, slab, False)
    x = inp["x_hi"] if case.f32 else inp["x"]
    ws = slab["ws"]
    rc = lib.sow_group_bwd(_p(x), _p(slab["A_cat"]), _p(slab["t_cat"]), arr, len(case.members), _p(slab["dt_cat"]),
                           _p(slab["dx"]), case.T, case.fin, _lib.SOWB_F32 if case.f32 else _lib.SOWB_BF16, _p(ws),
                           ws.numel() * 2, _stream())
    _lib.check(rc, "sow_group_bwd")


BWD_OUTPUTS = ("dt_cat", "dx", "dA", "dB", "dbias")


# ---------------------------------------------------------------------------------------------------------
# fp64 reference and component-wise bounds
# ---------------------------------------------------------------------------------------------------------

def reference(case, inp):
    """{output name: (ref, bound)} in fp64; names match the slab views (t{i} / dt{i} are column ranges of t_cat / dt_cat)."""
    f64 = torch.float64
    x = inp["x"].to(f64)
    ax = x.abs()
    u_out = U32 if case.f32 else U
    nseg = 3 if case.f32 else 1
    res = {}
    dX = torch.zeros_like(x)
    dX_round = torch.zeros_like(x)
    dX_acc = torch.zeros_like(x)
    dX_split = torch.zeros_like(x)
    kX = plan(case)["R"]
    for i, (m, d) in enumerate(zip(case.members, inp["m"])):
        A, B, dy = d["A"].to(f64), d["B"].to(f64), d["dy"].to(f64)
        aA, aB, ady = A.abs(), B.abs(), dy.abs()
        s = float(m.scale)
        t = s * (x @ A)
        at_acc = abs(s) * (ax @ aA)
        res[f"t{i}"] = (t, C * U * t.abs() + (gamma(case.fin * (2 if case.f32 else 1)) + (SPLIT if case.f32 else 0)) * at_acc)
        tB = t.abs() @ aB
        y = t @ B
        acc = tB.clone()
        split = torch.zeros_like(y)
        K = ops.rank_pad(m.r)
        if m.W:
            W = d["W"].to(f64)
            y += x @ W
            xW = ax @ W.abs()
            acc += xW
            K += nseg * case.fin
            if case.f32:
                split = SPLIT * xW
        if m.bias:
            y += d["bias"].to(f64)
        res[f"y{i}"] = (y, C * (u_out * y.abs() + U * tB) + gamma(K) * acc + split)

        # dt = s dY B^T; a second K2 launch adds onto the bf16 dt of the first one (a second rounding, of the partial p1)
        dt = s * (dy @ B.T)
        dt_acc = abs(s) * (ady @ aB.T)
        dt_round = torch.zeros_like(dt)
        G, n_launch, bpl = k2_plan(m.out)
        if n_launch > 1:
            c1 = min(m.out, bpl * 128)
            dt_round += (s * (dy[:, :c1] @ B[:, :c1].T)).abs()
        if case.f32:
            dt_round += dt_acc              # dY enters K2 as its bf16 high piece
        res[f"dt{i}"] = (dt, C * U * (dt.abs() + dt_round) + gamma(m.out) * dt_acc)
        dt_mag = dt.abs() + dt_round        # bounds |error of the stored dt| / u

        dA = x.T @ dt
        xdt = ax.T @ dt_mag
        res[f"dA{i}"] = (dA, C * U * (dA.abs() + xdt) + gamma(case.T) * xdt)
        dB = t.T @ dy
        tdy = t.abs().T @ ady
        res[f"dB{i}"] = (dB, C * U * (dB.abs() + tdy) + gamma(case.T) * tdy)
        if m.bias:
            db = dy.sum(0)
            sdy = ady.sum(0)
            res[f"dbias{i}"] = (db, C * U * (db.abs() + (sdy if case.f32 else 0)) + gamma(case.T) * sdy)

        dX += dt @ A.T
        dtA = dt_mag @ aA.T
        dX_round += dtA
        dX_acc += dtA
        if m.W:
            W = d["W"].to(f64)
            dX += dy @ W.T
            dyW = ady @ W.abs().T
            dX_acc += dyW
            kX += nseg * m.out
            if case.f32:
                dX_split += SPLIT * dyW
    res["dx"] = (dX, C * (u_out * dX.abs() + U * dX_round) + gamma(kX) * dX_acc + dX_split)
    return res


def gather(case, slab):
    """{output name: kernel result} for the names of ``reference``."""
    L = plan(case)
    got = {"dx": slab["dx"]}
    off = 0
    for i, m in enumerate(case.members):
        got[f"y{i}"] = slab[f"y{i}"]
        got[f"t{i}"] = slab["t_cat"][:, off:off + m.r]
        got[f"dt{i}"] = slab["dt_cat"][:, off:off + m.r]
        got[f"dA{i}"] = slab[f"dA{i}"]
        got[f"dB{i}"] = slab[f"dB{i}"]
        if m.bias:
            got[f"dbias{i}"] = slab[f"dbias{i}"]
        off += ops.rank_pad(m.r)
    assert off == L["R"]
    return got


def ratios(got, ref):
    """{name: max |got - ref| / bound}; inf where an element is not finite or exceeds a zero bound."""
    out = {}
    for k, (r, b) in ref.items():
        g = got[k].to(torch.float64)
        err = (g - r).abs()
        q = torch.where(b > 0, err / b, torch.where(err > 0, torch.inf, 0.0))
        q = torch.where(torch.isfinite(g), q, torch.inf)
        out[k] = float(q.max()) if q.numel() else 0.0
    return out


def padding_checks(case, inp, slab):
    """A_cat is the members' A packed bit for bit with zero padding; the padding columns of t_cat and dt_cat are 0."""
    A_cat, t_cat, dt_cat = slab["A_cat"], slab["t_cat"], slab["dt_cat"]
    exp = torch.zeros_like(A_cat)
    off = 0
    pad_cols = []
    for m, d in zip(case.members, inp["m"]):
        exp[:, off:off + m.r] = d["A"]
        pad_cols += list(range(off + m.r, off + ops.rank_pad(m.r)))
        off += ops.rank_pad(m.r)
    problems = []
    if not torch.equal(A_cat.view(torch.int16), exp.view(torch.int16)):
        problems.append("A_cat differs from the packed factors")
    if pad_cols:
        idx = torch.tensor(pad_cols, device=A_cat.device)
        if not bool((t_cat.index_select(1, idx) == 0).all()):
            problems.append("t_cat padding columns are not 0")
        if not bool((dt_cat.index_select(1, idx) == 0).all()):
            problems.append("dt_cat padding columns are not 0")
    return problems


def run_case(case, seed=0):
    """Runs forward and backward into guarded buffers.  Returns (got, ref, problems)."""
    inp = make_inputs(case, seed)
    slab = make_slab(case)
    problems = []
    group_fwd(case, inp, slab)
    saved = (slab["A_cat"].clone(), slab["t_cat"].clone())
    group_bwd(case, inp, slab)
    torch.cuda.synchronize()
    if not (torch.equal(saved[0].view(torch.int16), slab["A_cat"].view(torch.int16))
            and torch.equal(saved[1].view(torch.int16), slab["t_cat"].view(torch.int16))):
        problems.append("the backward changed A_cat / t_cat")
    problems += padding_checks(case, inp, slab)
    if case.repro:
        names = [n for n in slab.views if n.startswith(BWD_OUTPUTS)]
        first = {n: slab[n].clone() for n in names}
        slab.refill(names)
        group_bwd(case, inp, slab)
        torch.cuda.synchronize()
        for n in names:
            if not torch.equal(first[n].view(torch.int16), slab[n].view(torch.int16)):
                problems.append(f"second backward differs in {n}")
    if not slab.guards_intact():
        problems.append("a guard element was overwritten")
    ref = reference(case, inp)
    return gather(case, slab), ref, problems


def check_case(case):
    """Asserts the case reaches its branches, stays inside its bounds and its buffers; returns the worst ratio."""
    L = plan(case)
    assert {k: L[k] for k in case.expect} == case.expect, (case.name, L)
    got, ref, problems = run_case(case)
    q = ratios(got, ref)
    worst = max(q, key=q.get)
    print(f"EDGE {case.name}: G={L['G']} launches={L['launches']} batched={L['batched']} R={L['R']} bn={L['bn']} "
          f"dx_segs={L['dx_segs']} worst={q[worst]:.3f} ({worst}) " + json.dumps({k: round(v, 4) for k, v in q.items()}))
    assert not problems, (case.name, problems)
    bad = {k: v for k, v in q.items() if not v < 1.0}
    assert not bad, (case.name, bad)
    return q[worst]


# ---------------------------------------------------------------------------------------------------------
# tests
# ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", CASES, ids=repr)
def test_group_kernels_within_componentwise_bounds(case):
    check_case(case)


def test_big_tiles_within_componentwise_bounds():
    """SOWB_BIG_TILES is read once per process: the 256 x 256 tile GEMMs run in a child interpreter."""
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import test_linear_edges_gpu as t\n"
            "for c in t.BIG_TILE_CASES: t.check_case(c)\n") % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ, SOWB_BIG_TILES="1")
    p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    print(p.stdout)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    assert p.stdout.count("EDGE big_tiles") == len(BIG_TILE_CASES)


@pytest.mark.parametrize("kind", ["in_not_multiple_of_8", "out_not_multiple_of_8", "rank_above_limit"])
def test_limit_errors_raise_and_write_nothing(kind):
    if kind == "in_not_multiple_of_8":
        case = Case(kind, 64, 12, [M(136, 8)], {})
    elif kind == "out_not_multiple_of_8":
        case = Case(kind, 64, 72, [M(100, 8)], {})
    else:
        case = Case(kind, 64, 72, [M(136, 256), M(136, 256), M(136, 256), M(136, 257)], {})
        assert plan(case)["R"] > 64 * MAX_ALPHA
    inp = make_inputs(case)
    slab = make_slab(case)
    with pytest.raises(SowB200Error):
        group_fwd(case, inp, slab)
    with pytest.raises(SowB200Error):
        group_bwd(case, inp, slab)
    torch.cuda.synchronize()
    assert slab.untouched()


def test_checker_rejects_a_single_bad_element():
    """The bounds are tight enough to catch one output element off by 4 bf16 ulps, and two swapped rows of a tail tile."""
    case = CASES[0]
    assert case.T % BM != 0
    got, ref, problems = run_case(case)
    assert not problems
    assert max(ratios(got, ref).values()) < 1.0
    y = got["y0"].clone()
    i = int(ref["y0"][0].abs().argmax())
    bits = y.view(-1).view(torch.int16)
    bits[i] += 4                                           # 4 ulps further from zero
    q = ratios(dict(got, y0=y), ref)
    print(f"EDGE mutation: 4-ulp change of y0[{i}] -> ratio {q['y0']:.2f}")
    assert q["y0"] > 1.0
    y = got["y0"].clone()
    T = case.T
    y[[T - 2, T - 1]] = y[[T - 1, T - 2]]
    q = ratios(dict(got, y0=y), ref)
    print(f"EDGE mutation: rows {T - 2} / {T - 1} swapped -> ratio {q['y0']:.2f}")
    assert q["y0"] > 1.0


# ---------------------------------------------------------------------------------------------------------
# concatenated-rank limit at the module level
# ---------------------------------------------------------------------------------------------------------

class _QKV(torch.nn.Module):
    def __init__(self, h, r, n_iter):
        super().__init__()
        from sow_b200.layer import SoWLinear
        kw = dict(rank=r, n_iter=n_iter, init_method="normal", device="cuda", dtype=torch.bfloat16, bias=True)
        self.q_proj = SoWLinear(h, h, **kw)
        self.k_proj = SoWLinear(h, h // 2, **kw)
        self.v_proj = SoWLinear(h, h // 2, **kw)
        with torch.no_grad():
            for m in (self.q_proj, self.k_proj, self.v_proj):
                m.acc_downweight = torch.nn.Parameter(torch.randn(h, m.out_features, device="cuda").mul_(h ** -0.5)
                                                      .to(torch.bfloat16), requires_grad=False)
                for b in m.upscale_weights:
                    b.normal_(0, 0.05)
                m.bias.normal_(0, 0.1)

    def forward(self, x):
        return torch.cat([self.q_proj(x), self.k_proj(x), self.v_proj(x)], dim=-1)


def test_group_wider_than_the_rank_limit_runs_its_members_one_by_one():
    """q/k/v with rank=128, n_iter=4: each member has r = 512, the three together R = 1536 > 1024.  The group falls back to
    one call per member and computes what the ungrouped block computes."""
    import copy
    from sow_b200.surgery import group_shared_inputs
    torch.manual_seed(0)
    plain = _QKV(512, 128, 4)
    fused = copy.deepcopy(plain)
    assert group_shared_inputs(fused) == 1 and plain.q_proj._group is None
    x = torch.randn(2, 100, 512, device="cuda", dtype=torch.bfloat16)
    res = []
    for blk in (fused, plain):
        xi = x.clone().requires_grad_(True)
        y = blk(xi)
        y.float().pow(2).mean().backward()
        res.append((y, xi.grad, {n: p.grad for n, p in blk.named_parameters() if p.grad is not None}))
    (y0, gx0, g0), (y1, gx1, g1) = res
    assert torch.equal(y0, y1) and torch.equal(gx0, gx1)
    assert set(g0) == set(g1) and len(g0) == 3 * (2 * 4 + 1)
    for k in g0:
        assert torch.equal(g0[k], g1[k]), k


def test_single_module_wider_than_the_rank_limit_raises():
    from sow_b200.layer import SoWLinear
    m = SoWLinear(256, 256, rank=1088, init_method="normal", device="cuda", dtype=torch.bfloat16)
    with pytest.raises(SowB200Error, match="concatenated rank"):
        m(torch.randn(8, 256, device="cuda", dtype=torch.bfloat16))
