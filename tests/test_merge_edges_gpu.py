"""GPU: the grouped merge W <- W_prev + s * A . B (ops.merge_grouped) element by element against fp64, with every W a view
into a slab filled with a NaN bit pattern and separated from its neighbours by guard bands.

bf16: the kernel adds the rank in 64-wide chunks, one launch per chunk, and rounds W to bf16 after each, so the bound is
ceil(r / 64) bf16 roundings (plus the two fp32 roundings of the epilogue) of |W_prev| + |s| |A| |B|, plus the fp32
accumulation of a chunk.  fp32: the same with one fp32 rounding per chunk.
"""
import math

import pytest
import torch

from sow_b200 import ops
from test_linear_edges_gpu import U, U32, Slab, _const, gamma

pytestmark = pytest.mark.gpu

MG_MAX_ENTRIES = _const("merge.cu", "kMgMaxEntries")   # longer tables are split over several launches per rank chunk


def a_bulk(fin, r, A):
    """Whether merge.cu stages the [128 x r] blocks of A with one bulk copy (MergeDevEntry::a_bulk)."""
    return r <= 64 and A.data_ptr() % 16 == 0 and ((fin % 128) * r) % 8 == 0


def build(specs, dtype, seed):
    """specs: (in, out, r, prev kind, scale, misaligned A).  Returns (slab, items, expected state per entry)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    slab = Slab([(f"W{i}", (s[0], s[1]), dtype) for i, s in enumerate(specs)], "cuda")
    items, meta = [], []
    for i, (fin, fout, r, prev, scale, misaligned) in enumerate(specs):
        W = slab[f"W{i}"]
        if misaligned:           # A one element into its buffer: not 16-byte aligned
            A = (torch.randn(fin * r + 1, generator=g, device="cuda") * fin ** -0.5).to(dtype)[1:].view(fin, r)
        else:
            A = (torch.randn(fin, r, generator=g, device="cuda") * fin ** -0.5).to(dtype)
        B = (torch.randn(r, fout, generator=g, device="cuda") * 0.1).to(dtype)
        init = (torch.randn(fin, fout, generator=g, device="cuda") * 0.05).to(dtype)
        if prev == "same":
            W.copy_(init)
            Wp = W
        elif prev == "separate":
            Wp = init.clone()
        else:
            Wp = None
        items.append((W, Wp, A, B, scale))
        meta.append((None if prev == "none" else init, Wp if prev == "separate" else None))
    torch.cuda.synchronize()
    return slab, items, meta


def check(items, meta, slab, bf16):
    """Largest |W - ref| / bound of each entry; asserts separate W_prev are unchanged and the guards intact."""
    out = []
    for (W, _, A, B, s), (init, sep) in zip(items, meta):
        A64, B64 = A.to(torch.float64), B.to(torch.float64)
        prod = s * (A64 @ B64)
        aprod = abs(s) * (A64.abs() @ B64.abs())
        ref = prod if init is None else prod + init.to(torch.float64)
        mag = aprod if init is None else aprod + init.to(torch.float64).abs()
        nch = math.ceil(A.shape[1] / 64)
        per = (U + 2 * U32) if bf16 else U32
        bound = nch * per * (1 + per) ** nch * mag + gamma(64) * aprod
        got = W.to(torch.float64)
        q = torch.where(torch.isfinite(got), (got - ref).abs() / bound, torch.inf)
        out.append(float(q.max()))
        if sep is not None:
            assert torch.equal(sep, init), "merge changed a separate W_prev"
    assert slab.guards_intact(), "a guard element was overwritten"
    return out


def report(name, specs, q):
    worst = max(range(len(q)), key=q.__getitem__)
    print(f"EDGE {name}: {len(q)} matrices, worst {q[worst]:.3f} at {specs[worst][:4]}")
    assert max(q) < 1.0, [(s[:4], round(v, 3)) for s, v in zip(specs, q) if not v < 1.0]


def test_bf16_mixed_list_elementwise():
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
        (77, 136, 128, "same", -0.5, False),
        (300, 1000, 1, "separate", 1.0, False),
    ]
    slab, items, meta = build(specs, torch.bfloat16, 0)
    bulk = [a_bulk(s[0], s[2], it[2]) for s, it in zip(specs, items)]
    assert any(bulk) and not all(bulk)
    ops.merge_grouped(items)
    torch.cuda.synchronize()
    report("merge_bf16_mixed", specs, check(items, meta, slab, True))


def test_bf16_list_longer_than_one_device_table():
    """440 matrices, most of rank > 192: every 64-wide rank chunk splits into two launches, eight table uploads cycle the
    four-slot pinned ring twice within the call."""
    ranks = [1, 7, 200, 256, 230, 250, 210, 193, 256, 240, 220, 256, 199, 256, 250, 256, 245, 256, 200, 256]
    specs = [((64, 72, 136, 200)[i % 4], (8, 136, 264)[i % 3], ranks[i % len(ranks)],
              ("none", "same", "separate")[i % 3], (0.5, 1.0, -2.0)[i // 3 % 3], False) for i in range(440)]
    for c in range(4):
        assert sum(s[2] > 64 * c for s in specs) > MG_MAX_ENTRIES
    slab, items, meta = build(specs, torch.bfloat16, 1)
    ops.merge_grouped(items)
    torch.cuda.synchronize()
    report("merge_bf16_440_entries", specs, check(items, meta, slab, True))


def test_fp32_mixed_list_elementwise():
    specs = [
        (200, 1002, 130, "none", 0.5, False),
        (72, 136, 65, "same", 1.0, False),
        (300, 1000, 8, "separate", 2.0, False),
        (129, 2738, 200, "same", -1.0, False),
        (64, 6, 1, "separate", 1.0, False),
        (33, 1001, 64, "none", 1.0, False),
        (100, 500, 150, "separate", 0.25, False),
    ]
    assert any(s[1] % 4 for s in specs) and any(s[2] > 64 for s in specs)
    slab, items, meta = build(specs, torch.float32, 2)
    ops.merge_grouped(items)
    torch.cuda.synchronize()
    report("merge_fp32_mixed", specs, check(items, meta, slab, False))
