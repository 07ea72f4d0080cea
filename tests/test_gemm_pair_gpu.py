"""GPU: the CTA-pair GEMM (sow_gemm_pair_kernel, 256 x 256 tiles over clusters of two CTAs) that runs the 16-bit forward y_i
and group dX.

* every output of sow_group_fwd / sow_group_bwd within the component-wise bounds of test_linear_edges_gpu, in guarded slabs,
  bf16 and fp16, over the tails of the pair tile: T < 256 (the odd CTA's rows all out of bounds), T not a multiple of 256,
  an N tail whose odd-CTA half of B is entirely out of bounds, K segments that are not a multiple of 64;
* y and dX bit for bit equal to the 128 x 256 single-CTA kernel (SOWB_GEMM_PAIR=0) at the Llama-350M shapes;
* capture and replay in a CUDA graph;
* at the shape bench.py measures, every forward and dX GEMM of a training step takes the pair kernel.

SOWB_GEMM_PAIR is read once per process, so the runs that set it go to child interpreters.
"""
import json
import os
import re
import subprocess
import sys

import pytest
import torch

import test_linear_edges_gpu as LE
from conftest import ROOT
from test_linear_edges_gpu import Case, M

pytestmark = pytest.mark.gpu

TESTS = os.path.join(ROOT, "tests")

PAIR_CASES = [
    Case("pair_T1_out2624_in72", 1, 72, [M(2624, 8)], {}),
    Case("pair_T129_out136_in264", 129, 264, [M(136, 50, scale=0.5)], {}),
    Case("pair_T255_out2736_in2736", 255, 2736, [M(2736, 64, bias=False)], {}),
    Case("pair_T256_out1000_in264", 256, 264, [M(1000, 8, scale=2.0)], {}),
    Case("pair_qkv_T385", 385, 264, [M(1000, 50), M(1000, 50, scale=0.5, bias=False), M(1000, 50, scale=2.0)],
         {"dx_segs": 4}),
    Case("pair_T4113_out2624_in2736", 4113, 2736, [M(2624, 65, scale=0.5)], {}),
]


def _child(code, env_extra, timeout=900):
    env = dict(os.environ, **env_extra)
    p = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n" % (ROOT, TESTS)
                        + code], env=env, capture_output=True, text=True, timeout=timeout)
    print(p.stdout)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    return p.stdout


# At T = 1 every element of dB is the single product t * dy, and a few of them fall into fp16's subnormal range, where the
# checker's relative bound does not hold (dB comes from K2, the same with either GEMM tile).  fp16 starts at T = 129.
FP16_PAIR_CASES = [c for c in PAIR_CASES if c.T > 1]


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_pair_tiles_within_componentwise_bounds(dtype):
    cases = "FP16_PAIR_CASES" if dtype == "fp16" else "PAIR_CASES"
    code = ("import test_linear_edges_gpu as t, test_fp16_edges_gpu as h, test_gemm_pair_gpu as g\n"
            + ("h.use_fp16(t)\n" if dtype == "fp16" else "")
            + "for c in g.%s: t.check_case(c)\n" % cases)
    out = _child(code, {"SOWB_GEMM_PAIR": "1"})
    assert out.count("EDGE pair_") == len(FP16_PAIR_CASES if dtype == "fp16" else PAIR_CASES)


# the four Llama-350M groups (in, [out_i]) at r = 50, and one ragged group
LLAMA_GROUPS = [("qkv", 32768, 1024, [1024] * 3), ("o", 32768, 1024, [1024]), ("gate_up", 32768, 1024, [2736] * 2),
                ("down", 32768, 2736, [1024]), ("ragged", 385, 264, [1000, 136, 1016])]

_HASH_CODE = """
import hashlib, json, torch
from sow_b200 import ops
import test_gemm_pair_gpu as g
res = {}
for name, T, fin, outs in g.LLAMA_GROUPS:
    gen = torch.Generator(device="cuda").manual_seed(1)
    rn = lambda *s, sc=1.0: (torch.randn(*s, generator=gen, device="cuda") * sc).bfloat16()
    x = rn(T, fin)
    mem = [(rn(fin, o, sc=fin ** -0.5), rn(fin, 50, sc=fin ** -0.5), rn(50, o, sc=0.1), rn(o, sc=0.1), rn(T, o)) for o in outs]
    ys, A_cat, t_cat = ops.group_fwd(x, [(W, A, B, b, 0.5) for W, A, B, b, dy in mem])
    dx = ops.group_bwd(x, A_cat, t_cat, [(W, B, dy, 0.5, None, None, False) for W, A, B, b, dy in mem], True)[0]
    torch.cuda.synchronize()
    for i, y in enumerate(ys + [dx]):
        res[f"{name}/{'dx' if i == len(ys) else 'y%d' % i}"] = hashlib.sha256(y.view(torch.int16).cpu().numpy().tobytes()).hexdigest()
print("HASHES " + json.dumps(res))
"""


def test_pair_bit_identical_to_single_cta_tiles():
    runs = {}
    for knob in ("0", "1"):
        out = _child(_HASH_CODE, {"SOWB_GEMM_PAIR": knob})
        runs[knob] = json.loads(re.search(r"^HASHES (.*)$", out, re.M).group(1))
    assert len(runs["1"]) == sum(len(o) + 1 for _, _, _, o in LLAMA_GROUPS)
    diff = [k for k in runs["0"] if runs["0"][k] != runs["1"][k]]
    assert not diff, diff


def test_pair_gemm_in_cuda_graph_replays_eager_bits():
    from sow_b200 import ops
    torch.manual_seed(3)
    T, fin, outs = 1000, 1024, [1024, 520]
    x = torch.randn(T, fin, device="cuda").bfloat16()
    mem = [((torch.randn(fin, o, device="cuda") * fin ** -0.5).bfloat16(), (torch.randn(fin, 50, device="cuda") * 0.05).bfloat16(),
            (torch.randn(50, o, device="cuda") * 0.1).bfloat16(), torch.randn(T, o, device="cuda").bfloat16()) for o in outs]

    def run():
        ys, A_cat, t_cat = ops.group_fwd(x, [(W, A, B, None, 1.0) for W, A, B, dy in mem])
        dx = ops.group_bwd(x, A_cat, t_cat, [(W, B, dy, 1.0, None, None, False) for W, A, B, dy in mem], True)[0]
        return ys + [dx]

    eager = [t.clone() for t in run()]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        run()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs_g = run()
    for t in outs_g:
        t.fill_(0)
    graph.replay()
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, outs_g):
        assert torch.equal(a.view(torch.int16), b.view(torch.int16))


def test_every_forward_and_dx_gemm_of_the_bench_step_is_a_pair_launch():
    """bench.py's workload (Llama-350M, batch 128 x 256 tokens): 24 layers x 7 projections forward, 24 x 4 group dX."""
    if os.environ.get("SOWB_GEMM_PAIR", "1") == "0":
        pytest.skip("SOWB_GEMM_PAIR=0 selects the single-CTA tiles")
    from torch.profiler import ProfilerActivity, profile
    from sow_b200.trainer import SoWTrainer, TrainConfig
    tr = SoWTrainer(TrainConfig(batch_size=128), torch.device("cuda", 0))
    ids = torch.randint(1, 32000, (128, 256), device="cuda")
    for _ in range(2):
        tr.step(ids)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        tr.step(ids)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    fwd = sum("sow_gemm_pair_kernel<true," in n for n in names)
    dx = sum("sow_gemm_pair_kernel<false," in n for n in names)
    single = [n for n in names if re.search(r"sow_gemm_kernel<256, false, (true|false), 0, 1,", n)]
    assert (fwd, dx, len(single)) == (168, 96, 0), (fwd, dx, single[:3])
    del tr
    torch.cuda.empty_cache()
