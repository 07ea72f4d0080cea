"""Gradient clipping inside FusedAdamW (max_grad_norm) against torch.nn.utils.clip_grad_norm_ + FusedAdamW, alternating the
variants in one process (CUDA events):  python tools/bench_clip.py [--out FILE]

  norm      : the norm pass alone (partials + finalize) over the trainable (non-SoW) group of Llama-350M r = 50 in bf16:
              embedding, lm_head and the 49 norms, 65.6 M elements = 131 MB, more than L2.  Algorithmic bytes are the 2 B
              per element read; the rate is given as a fraction of the copy bandwidth measured in the same process.
  opt_step  : one optimizer step of that model's two groups (trainable + SoW factors, 89 M elements), median over the
              alternated steps: clip_grad_norm_(trainable) + FusedAdamW against FusedAdamW(max_grad_norm) on the
              trainable group.
  trainer   : SoWTrainer bf16 at batch 128 x 256, grad_clipping = 1.0, torch path against fused_grad_clipping, alternated
              rounds (tokens/s).
  graph     : batch 16 x 256 with cuda_graph = True and grad_clipping = 1.0: the torch path (the graph is refused, so it
              runs eagerly) against the fused path (graphed).
  fp16      : fp16, fp32 moments, dynamic loss scaling and fused clipping at batch 128 (rejected before fused clipping).
Prints one JSON line per row and the GPU name and power limit."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sow_b200 import ops  # noqa: E402
from sow_b200.optim import FusedAdamW  # noqa: E402
from tools.bench_amp import copy_gbps, llama350m_trainable_shapes, median, timed  # noqa: E402

DEV = torch.device("cuda", 0)
N_DENSE = 51                 # the last shapes of llama350m_trainable_shapes: embedding, lm_head, 49 norms


def _params(shapes, gen, dt=torch.bfloat16):
    ps = [torch.nn.Parameter((torch.randn(s, generator=gen, device=DEV) * 0.02).to(dt)) for s in shapes]
    for p in ps:
        p.grad = (torch.randn(p.shape, generator=gen, device=DEV) * 1e-3).to(dt)
    return ps


def bench_norm(rounds, copy_bw):
    shapes = llama350m_trainable_shapes()[-N_DENSE:]
    gen = torch.Generator(device=DEV).manual_seed(0)
    gs = [(torch.randn(s, generator=gen, device=DEV) * 1e-3).bfloat16() for s in shapes]
    n = sum(g.numel() for g in gs)
    table = ops.build_adam_chunks(gs, gs, gs, gs)
    partials = torch.zeros(table.shape[0], device=DEV)
    total, coef = torch.zeros((), device=DEV), torch.zeros((), device=DEV)
    fn = lambda: ops.grad_norm([(table, torch.bfloat16)], partials, total, coef, 1.0)   # noqa: E731
    ms = median([timed(fn, 200) for _ in range(rounds)])
    gbps = 2 * n / (ms * 1e-3) / 1e9
    return [{"row": "norm", "elements": n, "bytes": 2 * n, "chunk_rows": table.shape[0], "ms_median": round(ms, 4),
             "GBps": round(gbps, 0), "of_copy_bw": round(gbps / copy_bw, 3)}]


def bench_opt_step(steps=60):
    shapes = llama350m_trainable_shapes()
    arms = {}
    for label in ("torch clip + FusedAdamW", "FusedAdamW(max_grad_norm)"):
        gen = torch.Generator(device=DEV).manual_seed(0)
        ps = _params(shapes, gen)
        dense, factors = ps[-N_DENSE:], ps[:-N_DENSE]
        fused = label.startswith("FusedAdamW(")
        opt = FusedAdamW([{"params": dense, "lr": 1e-2, "max_grad_norm": 1.0 if fused else None},
                          {"params": factors, "lr": 1e-3}], weight_decay=0.0)

        def step(dense=dense, opt=opt, fused=fused):
            if not fused:
                torch.nn.utils.clip_grad_norm_(dense, 1.0)
            opt.step()
        arms[label] = step
    for fn in arms.values():
        for _ in range(3):
            fn()
    times = {k: [] for k in arms}
    for _ in range(steps):
        for k, fn in arms.items():
            times[k].append(timed(fn, 1, warmup=0))
    row = {"row": "opt_step", "elements": sum(torch.Size(s).numel() for s in shapes), "steps": steps}
    for k, v in times.items():
        row[k] = {"ms_median": round(median(v), 4), "ms_min": round(min(v), 4)}
    return [row]


def _trainers(arms, batch, seq, warm=3, **common):
    from sow_b200.trainer import SoWTrainer, TrainConfig
    out = {}
    g = torch.Generator().manual_seed(0)
    ids = [torch.randint(1, 32000, (batch, seq), generator=g).to(DEV) for _ in range(6)]
    for label, kw in arms.items():
        cfg = TrainConfig(model="llama_350m", rank=50, seq_len=seq, batch_size=batch, init_method="normal",
                          grad_clipping=1.0, **{**common, **kw})
        tr = SoWTrainer(cfg, DEV)
        for i in range(warm):
            tr.step(ids[i % len(ids)])
        out[label] = tr
    return out, ids


def _run_rounds(trainers, ids, rounds, steps):
    res = {k: [] for k in trainers}
    for _ in range(rounds):
        for label, tr in trainers.items():
            ms = timed(lambda it=iter(ids * 4): tr.step(next(it)), steps, warmup=0)
            res[label].append(ids[0].numel() / (ms * 1e-3))
    return res


def _row(name, trainers, res, batch, seq, rounds, steps, **extra):
    row = {"row": name, "model": "llama_350m", "r": 50, "batch": batch, "seq": seq, "steps_per_round": steps,
           "rounds": rounds, **extra}
    for label, v in res.items():
        tr = trainers[label]
        row[label] = {"tokens_per_s_median": round(median(v), 0), "tokens_per_s_min": round(min(v), 0),
                      "graphed": tr._graph is not None}
        if tr.scaler is not None:
            row[label]["final_loss_scale"] = tr.scaler.get_scale()
    return row


def bench_trainer(rounds, steps=6):
    arms = {"torch clip_grad_norm_": {}, "fused_grad_clipping": dict(fused_grad_clipping=True)}
    trainers, ids = _trainers(arms, 128, 256)
    res = _run_rounds(trainers, ids, rounds, steps)
    row = _row("trainer", trainers, res, 128, 256, rounds, steps, dtype="bf16")
    del trainers
    torch.cuda.empty_cache()
    return [row]


def bench_graph(rounds, steps=20):
    arms = {"torch clip_grad_norm_ (eager)": {}, "fused_grad_clipping (graphed)": dict(fused_grad_clipping=True)}
    trainers, ids = _trainers(arms, 16, 256, warm=4, cuda_graph=True)
    res = _run_rounds(trainers, ids, rounds, steps)
    row = _row("graph", trainers, res, 16, 256, rounds, steps, dtype="bf16")
    del trainers
    torch.cuda.empty_cache()
    return [row]


def bench_fp16(rounds, steps=6):
    arms = {"fp16 fp32-state + loss scaling + fused clipping": dict(fused_grad_clipping=True)}
    trainers, ids = _trainers(arms, 128, 256, dtype=torch.float16, optimizer_state_dtype=torch.float32,
                              loss_scaling=True)
    tr = trainers[next(iter(arms))]
    st = tr.optimizer.state[tr.special[0]]["step"]
    before = float(st)
    res = _run_rounds(trainers, ids, rounds, steps)
    skipped = rounds * steps - int(float(tr.optimizer.state[tr.special[0]]["step"]) - before)
    row = _row("fp16", trainers, res, 128, 256, rounds, steps, dtype="fp16", skipped_steps=skipped)
    del trainers, tr
    torch.cuda.empty_cache()
    return [row]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the rows to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_clip needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    rows = [{"row": "gpu", "nvidia_smi": q[0] if q else "?"}]
    print(json.dumps(rows[0]), flush=True)
    bw = copy_gbps(a.rounds)
    rows.append({"row": "copy", "GBps": round(bw, 0), "bytes": 2 << 30})
    print(json.dumps(rows[-1]), flush=True)
    for bench in (lambda: bench_norm(a.rounds, bw), bench_opt_step, lambda: bench_trainer(a.rounds),
                  lambda: bench_graph(a.rounds), lambda: bench_fp16(a.rounds)):
        for row in bench():
            print(json.dumps(row), flush=True)
            rows.append(row)
    if a.out:
        with open(a.out, "w") as f:
            for row in rows:
                f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
