"""fp32 optimizer moments and loss scaling: cost of the mixed-precision Adam kernel and of a loss-scaled fp16 trainer step,
alternating the variants in one process (CUDA events):  python tools/bench_amp.py [--out FILE]

  adam    : one fused Adam launch over the trainable parameters of Llama-350M, r = 50 (SoW factors of the 168 matrices,
            embeddings, lm_head and norms: 89 M elements), for bf16 and fp16 parameters: moments of the parameter dtype
            (the plain kernel, and the mixed-precision kernel with a loss scale) against fp32 moments (without and with a
            scale).  Algorithmic bytes are 2 e_p + e_g + 4 e_state per element, plus e_g when the gradient is unscaled and
            written back; the rate is given as a fraction of the copy bandwidth measured in the same process.  The working
            set (1.2-2 GB) is far larger than L2.
  trainer : SoWTrainer tokens/s, Llama-350M in fp16, batch 128 x 256: plain fp16 (fp16 moments), fp32 moments, and fp32
            moments with dynamic loss scaling, with the number of skipped steps.
Prints one JSON line per row and the GPU name and power limit."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sow_b200 import ops  # noqa: E402

DEV = torch.device("cuda", 0)
DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}


def timed(fn, iters, warmup=3):
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


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def llama350m_trainable_shapes(r=50):
    h, ff = 1024, 2736
    per = [(h, h)] * 4 + [(h, ff)] * 2 + [(ff, h)]
    shapes = []
    for fin, fout in per * 24:
        shapes += [(fin, r), (r, fout)]
    return shapes + [(32000, h)] * 2 + [(h,)] * 49


def copy_gbps(rounds):
    src = torch.empty(2 << 30, dtype=torch.uint8, device=DEV)
    dst = torch.empty_like(src)
    ms = median([timed(lambda: dst.copy_(src), 10) for _ in range(rounds)])
    del src, dst
    torch.cuda.empty_cache()
    return 2 * (2 << 30) / (ms * 1e-3) / 1e9


def bench_adam(rounds, copy_bw):
    rows = []
    shapes = llama350m_trainable_shapes()
    n = sum(torch.Size(s).numel() for s in shapes)
    scale = torch.ones((), dtype=torch.float32, device=DEV)        # 1.0: the gradients keep their values across calls
    for label, dt in DTYPES.items():
        g = torch.Generator(device=DEV).manual_seed(0)
        ps = [(torch.randn(s, generator=g, device=DEV) * 0.02).to(dt) for s in shapes]
        gs = [torch.randn(s, generator=g, device=DEV).to(dt) * 1e-3 for s in shapes]
        tables = {}
        for sname, sdt in (("state=param", dt), ("state=fp32", torch.float32)):
            ms_ = [torch.zeros(s, dtype=sdt, device=DEV) for s in shapes]
            vs_ = [torch.zeros(s, dtype=sdt, device=DEV) for s in shapes]
            tables[sname] = (sdt, ops.build_adam_chunks(ps, gs, ms_, vs_), ms_, vs_)
        ep, p16 = 2, tables["state=param"][1]
        variants = {
            "state=param": (lambda: ops.adam_multi(p16, dt, 1e-3, 0.9, 0.999, 1e-8, 0.0, 0.1, 0.001, True), 2, False),
        }
        for sname, (sdt, tab, _, _) in tables.items():
            es = sdt.itemsize
            if sname == "state=fp32":
                variants[sname] = (lambda tab=tab, sdt=sdt: ops.adam_multi_amp(tab, dt, sdt, 1e-3, 0.9, 0.999, 1e-8, 0.0,
                                                                                True, 0.1, 0.001), es, False)
            variants[sname + "+scale"] = (lambda tab=tab, sdt=sdt: ops.adam_multi_amp(
                tab, dt, sdt, 1e-3, 0.9, 0.999, 1e-8, 0.0, True, 0.1, 0.001, grad_scale=scale), es, True)
        times = {k: [] for k in variants}
        for _ in range(rounds):
            for k, (fn, _, _) in variants.items():
                times[k].append(timed(fn, 20))
        row = {"row": "adam", "param_dtype": label, "elements": n}
        for k, (_, es, scaled) in variants.items():
            ms = median(times[k])
            nbytes = n * (2 * ep + ep + 4 * es + (ep if scaled else 0))
            gbps = nbytes / (ms * 1e-3) / 1e9
            row[k] = {"ms_median": round(ms, 4), "ms_min": round(min(times[k]), 4), "bytes_per_elem": nbytes // n,
                      "GBps": round(gbps, 0), "of_copy_bw": round(gbps / copy_bw, 3)}
        rows.append(row)
        del ps, gs, tables, variants
        torch.cuda.empty_cache()
    return rows


def bench_trainer(rounds, steps=6):
    from sow_b200.trainer import SoWTrainer, TrainConfig
    batch, seq = 128, 256
    arms = {"fp16": {}, "fp16 fp32-state": dict(optimizer_state_dtype=torch.float32),
            "fp16 fp32-state + loss scaling": dict(optimizer_state_dtype=torch.float32, loss_scaling=True)}
    g = torch.Generator().manual_seed(0)
    ids = [torch.randint(1, 32000, (batch, seq), generator=g).to(DEV) for _ in range(steps)]
    trainers, res, skipped = {}, {k: [] for k in arms}, {k: 0 for k in arms}
    for label, kw in arms.items():
        cfg = TrainConfig(model="llama_350m", rank=50, seq_len=seq, batch_size=batch, dtype=torch.float16,
                          init_method="normal", **kw)
        tr = SoWTrainer(cfg, DEV)
        for i in range(2):
            tr.step(ids[i])
        trainers[label] = tr
    for _ in range(rounds):
        for label, tr in trainers.items():
            st = tr.optimizer.state[tr.special[0]]["step"]
            before = float(st)
            ms = timed(lambda it=iter(ids): tr.step(next(it)), steps, warmup=0)
            skipped[label] += steps - int(float(tr.optimizer.state[tr.special[0]]["step"]) - before)
            res[label].append(batch * seq / (ms * 1e-3))
    row = {"row": "trainer", "model": "llama_350m", "r": 50, "batch": batch, "seq": seq, "steps_per_round": steps,
           "rounds": rounds}
    for label, v in res.items():
        row[label] = {"tokens_per_s_median": round(median(v), 0), "tokens_per_s_min": round(min(v), 0),
                      "skipped_steps": skipped[label]}
        if trainers[label].scaler is not None:
            row[label]["final_loss_scale"] = trainers[label].scaler.get_scale()
    return [row]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the rows to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_amp needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    rows = [{"row": "gpu", "nvidia_smi": q[0] if q else "?"}]
    print(json.dumps(rows[0]), flush=True)
    bw = copy_gbps(a.rounds)
    rows.append({"row": "copy", "GBps": round(bw, 0), "bytes": 2 << 30})
    print(json.dumps(rows[-1]), flush=True)
    for row in bench_adam(a.rounds, bw) + bench_trainer(a.rounds):
        print(json.dumps(row), flush=True)
        rows.append(row)
    if a.out:
        with open(a.out, "w") as f:
            for row in rows:
                f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
