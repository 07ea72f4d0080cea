#!/usr/bin/env python
"""Stock HF ForCausalLMLoss vs the native causal-LM loss (csrc/glue.cu ce_fwd_kernel / ce_bwd_kernel behind
llama_glue.CausalLMLoss), forward + backward, at the bench shape (batch 128 x seq 256, vocabulary 32000, bf16 logits).

    python tools/bench_loss.py [--batch 128] [--seq 256] [--vocab 32000] [--iters 20] [--dtype bf16] [--out FILE]

Each arm is timed with CUDA events over --iters repetitions after a warm-up; the logits (2.1 GB at the bench shape) are far
larger than the 126 MB L2, so every pass reads them from HBM.  Algorithmic bytes = what a native loss must move at least:
the logits read by the forward, read again by the backward, and the 16-bit gradient written (6.3 GB at the bench shape).
Peak memory = the largest allocation over the logits themselves during one forward + backward.  The native kernels are
also timed alone (ops.ce_fwd, ops.ce_bwd).  Prints one JSON line per measurement plus one with the card, its power
limit and the copy bandwidth measured in the same process.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.bench_glue import card, hbm_peak_gbs, time_ms  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--seq", type=int, default=256)
    ap.add_argument("--vocab", type=int, default=32000)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--dtype", choices=["bf16", "fp16"], default="bf16")
    ap.add_argument("--out")
    args = ap.parse_args()

    import torch
    from transformers.loss.loss_utils import ForCausalLMLoss
    from sow_b200 import ops
    from sow_b200.llama_glue import CausalLMLoss, loss_native_ok

    dt = {"bf16": torch.bfloat16, "fp16": torch.float16}[args.dtype]
    B, S, V = args.batch, args.seq, args.vocab
    gen = torch.Generator(device="cuda").manual_seed(0)
    logits = (torch.randn(B, S, V, device="cuda", generator=gen) * 3).to(dt).requires_grad_(True)
    labels = torch.randint(0, V, (B, S), device="cuda", generator=gen)
    assert loss_native_ok(logits, labels, V)
    N = B * S
    elem = logits.element_size()
    alg_bytes = 3 * N * V * elem
    lines = [dict(card(), what="card")]
    peak, peak_src = hbm_peak_gbs(args.iters)
    lines[0].update(copy_gbs=round(peak, 1), copy_source=peak_src)

    def arm(fn):
        def step():
            loss = fn(logits=logits, labels=labels, vocab_size=V)
            torch.autograd.grad(loss, logits)
        return step

    for name, fn in (("stock", ForCausalLMLoss), ("native", CausalLMLoss(ForCausalLMLoss))):
        step = arm(fn)
        ms = time_ms(step, args.iters)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        step()
        torch.cuda.synchronize()
        extra = torch.cuda.max_memory_allocated() - base
        gbs = alg_bytes / (ms / 1e3) / 1e9
        lines.append({"what": f"loss fwd+bwd {name}", "ms": round(ms, 4), "alg_GB": round(alg_bytes / 1e9, 3),
                      "GBps_vs_alg_bytes": round(gbs, 1), "of_copy_bw": round(gbs / peak, 3),
                      "peak_mem_GB_over_logits": round(extra / 1e9, 2)})

    x = logits.detach().view(N, V)
    t = labels.view(N)
    mx, ls, lpt = ops.ce_fwd(x, t)
    v = torch.full((N,), -1.0 / N, device="cuda")
    for name, fn, nbytes in (("ce_fwd kernel", lambda: ops.ce_fwd(x, t), N * V * elem),
                             ("ce_bwd kernel", lambda: ops.ce_bwd(x, mx, ls, t, v), 2 * N * V * elem)):
        ms = time_ms(fn, args.iters)
        gbs = nbytes / (ms / 1e3) / 1e9
        lines.append({"what": name, "ms": round(ms, 4), "GB": round(nbytes / 1e9, 3), "GBps": round(gbs, 1),
                      "of_copy_bw": round(gbs / peak, 3)})

    for ln in lines:
        print(json.dumps(ln), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(ln) + "\n" for ln in lines))


if __name__ == "__main__":
    main()
