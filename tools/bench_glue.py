#!/usr/bin/env python
"""Stock HF vs native (csrc/glue.cu) rotary embedding, SwiGLU and RMSNorm of one Llama layer, forward and backward, at the
bench shape (Llama-350M: batch 128 x seq 256, hidden 1024 = 16 heads of 64, intermediate 2736, bf16).

    python tools/bench_glue.py [--batch 128] [--seq 256] [--iters 20] [--dtype bf16] [--out FILE]

Each pass is timed with CUDA events over --iters repetitions after a warm-up.  The working set of every pass (>= 268 MB)
is larger than the 126 MB L2, so each repetition reads from HBM.  Achieved bandwidth = the bytes the pass must move at
least (every input read once, every output written once; cos / sin and the norm weight counted once; the RMSNorm
backward's bf16 product for the weight gradient, and torch's reduction of it, are not counted) over its time, set against the HBM
peak: MEASURED_PEAKS.json when present, otherwise the rate of a 2 GiB device-to-device copy measured here.
Prints one JSON line per pass plus one with the card, its power limit and the peak used.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # pragma: no cover
        return {"name": None, "error": str(e)}


def time_ms(fn, iters, warmup=3):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def hbm_peak_gbs(iters):
    import torch
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json"
    src = torch.empty(1 << 30, dtype=torch.int16, device="cuda")
    dst = torch.empty_like(src)
    ms = time_ms(lambda: dst.copy_(src), iters)
    return 2 * src.numel() * 2 / (ms / 1e3) / 1e9, "device-to-device copy of 2 GiB, measured here"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--seq", type=int, default=256)
    ap.add_argument("--heads", type=int, default=16)
    ap.add_argument("--head-dim", type=int, default=64)
    ap.add_argument("--intermediate", type=int, default=2736)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()

    import torch
    import torch.nn.functional as F
    from transformers.models.llama import modeling_llama as ml
    from sow_b200.llama_glue import _RMSNorm, _RoPE, _SwiGLU

    assert torch.cuda.is_available(), "bench_glue.py measures on the GPU"
    dt = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    B, S, H, D, I = args.batch, args.seq, args.heads, args.head_dim, args.intermediate
    stock_rope = getattr(ml.apply_rotary_pos_emb, "stock", ml.apply_rotary_pos_emb)
    g = torch.Generator(device="cuda").manual_seed(0)
    lines = []
    peak, peak_src = hbm_peak_gbs(args.iters)

    # ---- rotary embedding of q and k, laid out as HF's attention passes them ----
    q = torch.randn(B, S, H * D, device="cuda", generator=g).to(dt).view(B, S, H, D).transpose(1, 2).requires_grad_(True)
    k = torch.randn(B, S, H * D, device="cuda", generator=g).to(dt).view(B, S, H, D).transpose(1, 2).requires_grad_(True)
    inv = 1.0 / (10000.0 ** (torch.arange(0, D, 2, device="cuda").float() / D))
    fr = torch.arange(S, device="cuda").float()[:, None] * inv
    emb = torch.cat((fr, fr), -1)[None]
    cos, sin = emb.cos().to(dt), emb.sin().to(dt)
    gq = torch.randn(B, H, S, D, device="cuda", generator=g).to(dt)
    gk = torch.randn(B, H, S, D, device="cuda", generator=g).to(dt)
    n_qk = 2 * B * H * S * D
    rope_bytes = 2 * n_qk * 2 + 2 * S * D * 2        # q, k read + written; cos, sin read once
    swi_n = B * S * I
    gate = torch.randn(B, S, I, device="cuda", generator=g).to(dt).requires_grad_(True)
    up = torch.randn(B, S, I, device="cuda", generator=g).to(dt).requires_grad_(True)
    dh = torch.randn(B, S, I, device="cuda", generator=g).to(dt)
    norm = ml.LlamaRMSNorm(H * D, eps=1e-6).to("cuda", dt)
    xn = torch.randn(B, S, H * D, device="cuda", generator=g).to(dt).requires_grad_(True)
    dyn = torch.randn(B, S, H * D, device="cuda", generator=g).to(dt)
    norm_n = B * S * H * D
    ops = {
        "rope": {
            "stock": lambda: stock_rope(q, k, cos, sin),
            "native": lambda: _RoPE.apply(q, k, cos, sin),
            "bwd": lambda out: torch.autograd.grad(out, (q, k), (gq, gk)),
            "bytes": (rope_bytes, rope_bytes),
        },
        "swiglu": {
            "stock": lambda: F.silu(gate) * up,
            "native": lambda: _SwiGLU.apply(gate, up),
            "bwd": lambda out: torch.autograd.grad(out, (gate, up), dh),
            "bytes": (3 * swi_n * 2, 5 * swi_n * 2),     # fwd: gate, up -> h; bwd: dh, gate, up -> dgate, dup
        },
        "rmsnorm": {
            "stock": lambda: ml.LlamaRMSNorm.forward(norm, xn),
            "native": lambda: _RMSNorm.apply(xn, norm.weight, norm.variance_epsilon),
            "bwd": lambda out: torch.autograd.grad(out, (xn, norm.weight), dyn),
            "bytes": (2 * norm_n * 2, 3 * norm_n * 2),   # fwd: x -> y; bwd: dy, x -> dx
            "per_step": 2 * 24 + 1,
        },
    }
    for name, o in ops.items():
        fwd_b, bwd_b = o["bytes"]
        for impl in ("stock", "native"):
            f = o[impl]
            t_f = time_ms(f, args.iters)
            # a backward needs its own forward graph: time forward + backward together and subtract the forward
            t_fb = time_ms(lambda: o["bwd"](f()), args.iters)
            t_b = t_fb - t_f
            row = {"op": name, "impl": impl, "dtype": args.dtype, "shape": {"B": B, "S": S, "H": H, "D": D, "I": I},
                   "fwd_ms": t_f, "bwd_ms": t_b, "fwd_bwd_ms": t_fb,
                   "algorithmic_bytes_fwd": fwd_b, "algorithmic_bytes_bwd": bwd_b,
                   "gbs_fwd_bwd": (fwd_b + bwd_b) / (t_fb / 1e3) / 1e9,
                   "frac_of_hbm_peak": (fwd_b + bwd_b) / (t_fb / 1e3) / 1e9 / peak}
            lines.append(row)
        st, nat = lines[-2], lines[-1]
        nat["speedup_fwd_bwd"] = st["fwd_bwd_ms"] / nat["fwd_bwd_ms"]
    # per step of Llama-350M: 24 layers, one rotary and one SwiGLU call each, two norms each plus the final norm
    per_step = [o.get("per_step", 24) for o in ops.values()]
    lines.append({"card": card(), "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "iters": args.iters,
                  "per_step_calls": dict(zip(ops, per_step)),
                  "per_step_saving_ms": sum(n * (lines[2 * i]["fwd_bwd_ms"] - lines[2 * i + 1]["fwd_bwd_ms"])
                                            for i, n in enumerate(per_step))})
    for ln in lines:
        s = json.dumps(ln)
        print(s, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(s + "\n")


if __name__ == "__main__":
    main()
