"""fp16 against bf16 on the hot paths, alternating the two dtypes in one process (CUDA events; sow_profile_* for the
merge and Adam kernels):  python tools/bench_fp16.py [--out FILE]

  layer   : Llama-350M q/k/v and gate/up group forward + backward at T = 32768, r = 50, through the public SoWLinear API.
            "fp16 cast" replays what an fp16 module cost before the native fp16 path: x / dY / factors cast to bf16, the
            bf16 kernels, outputs cast back.
  merge   : grouped merge of the 168 Llama-350M matrices (r = 50), in place.
  adam    : FusedAdamW over the Llama-350M factor + dense parameter groups.
  trainer : SoWTrainer tokens/s, Llama-350M, batch 128 x 256.
Prints one JSON line per row and the GPU name and power limit."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sow_b200 import ops  # noqa: E402
from sow_b200.layer import SoWLinear, sow_linear_group  # noqa: E402

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


def bench_layer(rounds):
    T, fin, r = 32768, 1024, 50
    rows = []
    for gname, outs in (("q/k/v", [1024] * 3), ("gate/up", [2736] * 2)):
        setups = {}
        for label, dt in DTYPES.items():
            torch.manual_seed(0)
            mods = [SoWLinear(fin, o, bias=False, rank=r, init_method="normal", device=DEV, dtype=dt) for o in outs]
            for m in mods:
                m.acc_downweight = torch.nn.Parameter((torch.randn(fin, m.out_features, device=DEV) * 0.02).to(dt),
                                                      requires_grad=False)
            x = torch.randn(T, fin, device=DEV).to(dt).requires_grad_(True)
            dys = [torch.randn(T, o, device=DEV).to(dt) for o in outs]
            setups[label] = (mods, x, dys)
        mods16, x16, dys16 = setups["fp16"]

        def native(label):
            mods, x, dys = setups[label]

            def run():
                params = []
                for m in mods:
                    params += [m.acc_downweight, m.downscale_weights[0], m.upscale_weights[0], None, None]
                ys = sow_linear_group(x, [1.0] * len(mods), params)
                torch.autograd.backward(ys, dys)
            return run

        def cast_path():
            # the parent commit's fp16 policy: every operand rounded to bf16, bf16 kernels, results cast back
            xb = x16.detach().to(torch.bfloat16).requires_grad_(True)
            params = []
            for m in mods16:
                params += [m.acc_downweight.to(torch.bfloat16),
                           m.downscale_weights[0].detach().to(torch.bfloat16).requires_grad_(True),
                           m.upscale_weights[0].detach().to(torch.bfloat16).requires_grad_(True), None, None]
            ys = [y.to(torch.float16) for y in sow_linear_group(xb, [1.0] * len(mods16), params)]
            torch.autograd.backward(ys, dys16)
            xb.grad.to(torch.float16)
            for p in params[1::5] + params[2::5]:
                p.grad.to(torch.float16)

        times = {"bf16": [], "fp16": [], "fp16 cast": []}
        for _ in range(rounds):
            times["bf16"].append(timed(native("bf16"), 10))
            times["fp16"].append(timed(native("fp16"), 10))
            times["fp16 cast"].append(timed(cast_path, 10))
        fl = sum(2 * T * fin * o * 3 + 2 * T * r * (2 * fin + 3 * o) for o in outs)   # fwd + dX + factor products
        row = {"row": "layer", "group": gname, "T": T, "in": fin, "outs": outs, "r": r}
        for k, v in times.items():
            v = sorted(v)
            row[k] = {"ms_median": round(v[len(v) // 2], 3), "ms_min": round(v[0], 3),
                      "tflops": round(fl / (v[len(v) // 2] * 1e-3) / 1e12, 1)}
        rows.append(row)
        del setups
        torch.cuda.empty_cache()
    return rows


def llama350m_shapes():
    """(in, out) of the 168 SoW matrices of Llama-350M (24 layers x q, k, v, o, gate, up, down)."""
    h, ff = 1024, 2736
    per = [(h, h)] * 4 + [(h, ff)] * 2 + [(ff, h)]
    return per * 24


def bench_merge(rounds):
    r = 50
    items = {}
    for label, dt in DTYPES.items():
        g = torch.Generator(device=DEV).manual_seed(0)
        lst = []
        for fin, fout in llama350m_shapes():
            W = (torch.randn(fin, fout, generator=g, device=DEV) * 0.02).to(dt)
            A = (torch.randn(fin, r, generator=g, device=DEV) * 0.05).to(dt)
            B = (torch.randn(r, fout, generator=g, device=DEV) * 1e-4).to(dt)
            lst.append((W, W, A, B, 1.0))
        items[label] = lst
    row = {"row": "merge", "matrices": len(items["bf16"]), "r": r}
    res = {k: [] for k in DTYPES}
    for _ in range(rounds):
        for label in DTYPES:
            ops.merge_grouped(items[label])              # warm
            torch.cuda.synchronize()
            ops.profile_enable(True)
            for _ in range(10):
                ops.merge_grouped(items[label])
            torch.cuda.synchronize()
            ms, work, n = ops.profile_read("merge")
            ops.profile_enable(False)
            res[label].append((ms / 10, work / ms / 1e6))
    for label, v in res.items():
        v = sorted(v)
        row[label] = {"ms_median": round(v[len(v) // 2][0], 4), "GBps": round(v[len(v) // 2][1], 0)}
    del items
    torch.cuda.empty_cache()
    return [row]


def bench_adam(rounds):
    from sow_b200.optim import FusedAdamW
    r = 50
    opts = {}
    for label, dt in DTYPES.items():
        fac = []
        for fin, fout in llama350m_shapes():
            fac += [torch.nn.Parameter(torch.randn(fin, r, device=DEV).to(dt)), torch.nn.Parameter(torch.randn(r, fout, device=DEV).to(dt))]
        dense = [torch.nn.Parameter(torch.randn(32000, 1024, device=DEV).to(dt)) for _ in range(2)]
        dense += [torch.nn.Parameter(torch.randn(1024, device=DEV).to(dt)) for _ in range(49)]
        for p in fac + dense:
            p.grad = torch.randn_like(p)
        opts[label] = FusedAdamW([{"params": fac, "lr": 1e-3}, {"params": dense, "lr": 1e-3}])
    row = {"row": "adam"}
    res = {k: [] for k in DTYPES}
    for _ in range(rounds):
        for label in DTYPES:
            opts[label].step()
            torch.cuda.synchronize()
            ops.profile_enable(True)
            for _ in range(10):
                opts[label].step()
            torch.cuda.synchronize()
            ms, work, n = ops.profile_read("adam")
            ops.profile_enable(False)
            res[label].append((ms / 10, work / ms / 1e6))
    for label, v in res.items():
        v = sorted(v)
        row[label] = {"ms_median": round(v[len(v) // 2][0], 4), "GBps": round(v[len(v) // 2][1], 0)}
    del opts
    torch.cuda.empty_cache()
    return [row]


def bench_trainer(rounds, steps=6):
    from sow_b200.trainer import SoWTrainer, TrainConfig
    batch, seq = 128, 256
    row = {"row": "trainer", "model": "llama_350m", "batch": batch, "seq": seq}
    res = {k: [] for k in DTYPES}
    for _ in range(rounds):
        for label, dt in DTYPES.items():
            cfg = TrainConfig(model="llama_350m", rank=50, seq_len=seq, batch_size=batch, dtype=dt, init_method="normal")
            tr = SoWTrainer(cfg, DEV)
            g = torch.Generator().manual_seed(0)
            ids = [torch.randint(1, 32000, (batch, seq), generator=g).to(DEV) for _ in range(steps + 2)]
            for i in range(2):
                tr.step(ids[i])
            ms = timed(lambda it=iter(ids[2:]): tr.step(next(it)), steps, warmup=0)
            res[label].append(batch * seq / (ms * 1e-3))
            del tr
            torch.cuda.empty_cache()
    for label, v in res.items():
        v = sorted(v)
        row[label] = {"tokens_per_s_median": round(v[len(v) // 2], 0)}
    return [row]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the rows to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fp16 needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    rows = [{"row": "gpu", "nvidia_smi": q[0] if q else "?"}]
    print(json.dumps(rows[0]), flush=True)
    for fn in (bench_layer, bench_merge, bench_adam, bench_trainer):
        for row in fn(a.rounds):
            print(json.dumps(row), flush=True)
            rows.append(row)
    if a.out:
        with open(a.out, "w") as f:
            for row in rows:
                f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
